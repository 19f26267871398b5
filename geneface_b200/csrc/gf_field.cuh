// Device-side building blocks of the RAD-NeRF field shared by the fused kernels:
// per-level grid geometry, C=2 fp32 tiled/hash grid sampling (same rounding sequence as
// k_grid_forward / reference gridencoder.cu:87-196), degree-4 SH, and the packed model layout.
#pragma once
#include "gf_common.cuh"

namespace gf {

// ---- per-level geometry, computed ON DEVICE once per model (exp2f must be the GPU's) ----------
// The reference recomputes `get_grid_index` (3 conditional stride steps + a runtime modulo) for every
// corner (gridencoder.cu:66-84).  Both are level constants: which dimensions enter the index
// (stride <= hashmap_size), and the modulo, which is a no-op on dense levels (index < hsize) and a
// power-of-two mask on clipped/hashed levels (hsize == 2^log2_hashmap_size).  k_level_geometry
// derives sy/sz/mask/hashed once; the integer results are identical to the reference's.
struct GridLevels {
    float scale[16];
    uint32_t res[16];      // resolution = ceil(scale)+1
    uint32_t hsize[16];    // entries in the level
    uint32_t offset[16];   // first entry of the level
    uint32_t sy[16];       // stride of y in the index (0 when dropped)
    uint32_t sz[16];       // stride of z (0 when dropped; unused for 2-D grids)
    uint32_t mask[16];     // index & mask  ==  index % hsize
    uint32_t hashed[16];   // 1: fast_hash index (gridtype 0 on a clipped level)
    // Wrapping levels (not hashed, and the largest corner index reaches hsize, so `& mask` changes it) are read from a padded image:
    // E[k] = T[k % hsize] for k < hsize + pad, pad = 1 + sy + sz (the largest corner offset).  Then E[(b & mask) + d] == T[(b + d) & mask]
    // for every corner offset d, so the corners of a cell are rows of adjacent entries.  pad = 0 on every other level.
    uint32_t pad[16];
    uint32_t img_offset[16];   // first entry of the level in the padded image (levels of hsize + pad entries, level-major)
};

struct GridDesc {
    const float2* lbase[16];   // first entry of level l (padded image: img_offset[l]; table read in place: offset[l]); address = IMAD.WIDE(idx, 8, base)
    GridLevels lv;
    uint32_t gridtype;     // 0 hash, 1 tiled
    uint32_t interp;       // 0 linear, 1 smoothstep
};

__device__ __forceinline__ float smooth_(float v) { return v * v * (3.0f - 2.0f * v); }

constexpr uint32_t HASH_P1 = 2654435761u, HASH_P2 = 805459861u;   // gridencoder.cu:54

// indices of the 8 corners of level `l` around integer cell (gx,gy,gz)
__device__ __forceinline__ void corner_index3(const GridLevels& lv, int l, uint32_t gx, uint32_t gy, uint32_t gz, uint32_t (&idx)[8]) {
    const uint32_t mask = lv.mask[l];
    if (lv.hashed[l]) {
        const uint32_t hx[2] = {gx, gx + 1}, hy[2] = {gy * HASH_P1, (gy + 1) * HASH_P1}, hz[2] = {gz * HASH_P2, (gz + 1) * HASH_P2};
        #pragma unroll
        for (int c = 0; c < 8; c++) idx[c] = (hx[c & 1] ^ hy[(c >> 1) & 1] ^ hz[c >> 2]) & mask;
    } else {
        const uint32_t sy = lv.sy[l], sz = lv.sz[l];
        const uint32_t b = gx + gy * sy + gz * sz;
        #pragma unroll
        for (int c = 0; c < 8; c++) idx[c] = (b + (c & 1) + ((c >> 1) & 1) * sy + (c >> 2) * sz) & mask;
    }
}

__device__ __forceinline__ void corner_index2(const GridLevels& lv, int l, uint32_t gx, uint32_t gy, uint32_t (&idx)[4]) {
    const uint32_t mask = lv.mask[l];
    if (lv.hashed[l]) {
        const uint32_t hx[2] = {gx, gx + 1}, hy[2] = {gy * HASH_P1, (gy + 1) * HASH_P1};
        #pragma unroll
        for (int c = 0; c < 4; c++) idx[c] = (hx[c & 1] ^ hy[c >> 1]) & mask;
    } else {
        const uint32_t sy = lv.sy[l];
        const uint32_t b = gx + gy * sy;
        #pragma unroll
        for (int c = 0; c < 4; c++) idx[c] = (b + (c & 1) + (c >> 1) * sy) & mask;
    }
}

// NL consecutive levels of the 3-D grid with ALL corner loads issued before any is consumed (memory-level
// parallelism: the gathers are latency bound).  x,y,z already mapped to [0,1] (grid.py:149).
// FAST = false: interpolation arithmetic and accumulation order are the reference's (bit-identical to k_grid_forward).
// FAST = true (tensor-core path, features are rounded to fp16 afterwards): levels whose index drops z (sz == 0, the
// "tiled" quirk of gridencoder.cu:72) fetch their 4 distinct corners once instead of 8 (w_z0 + w_z1 = 1).
// Out-of-range inputs return 0 (gridencoder.cu:110-135): handled by sampling a clamped point and zeroing the result, so
// no load is predicated.  out[i] = the 2 channels of level l0+i.
template <int NL, bool FAST = false>
__device__ __forceinline__ void grid3_levels(const GridDesc& g, int l0, float x, float y, float z, float2 (&out)[NL]) {
    const bool oob = x < 0 || x > 1 || y < 0 || y > 1 || z < 0 || z > 1;
    if (oob) { x = 0.5f; y = 0.5f; z = 0.5f; }
    float fx[NL], fy[NL], fz[NL];
    float2 v[NL][8];
    #pragma unroll
    for (int i = 0; i < NL; i++) {
        const int l = l0 + i;
        const float scale = g.lv.scale[l];
        float px = __fmaf_rn(x, scale, 0.5f), py = __fmaf_rn(y, scale, 0.5f), pz = __fmaf_rn(z, scale, 0.5f);
        const uint32_t gx = (uint32_t)floorf(px), gy = (uint32_t)floorf(py), gz = (uint32_t)floorf(pz);
        px = __fsub_rn(px, (float)gx); py = __fsub_rn(py, (float)gy); pz = __fsub_rn(pz, (float)gz);
        if (g.interp == 1) { px = smooth_(px); py = smooth_(py); pz = smooth_(pz); }
        fx[i] = px; fy[i] = py; fz[i] = pz;
        const float2* __restrict__ tab = g.lbase[l];
        if (FAST && g.lv.sz[l] == 0 && !g.lv.hashed[l]) {
            uint32_t idx[4];
            const uint32_t sy = g.lv.sy[l], mask = g.lv.mask[l], b = gx + gy * sy;
            #pragma unroll
            for (int c = 0; c < 4; c++) idx[c] = (b + (c & 1) + (c >> 1) * sy) & mask;
            #pragma unroll
            for (int c = 0; c < 4; c++) v[i][c] = __ldg(tab + idx[c]);
        } else {
            uint32_t idx[8];
            corner_index3(g.lv, l, gx, gy, gz, idx);
            #pragma unroll
            for (int c = 0; c < 8; c++) v[i][c] = __ldg(tab + idx[c]);
        }
    }
    #pragma unroll
    for (int i = 0; i < NL; i++) {
        const int l = l0 + i;
        const float px = fx[i], py = fy[i], pz = fz[i];
        const float qx = __fsub_rn(1.0f, px), qy = __fsub_rn(1.0f, py), qz = __fsub_rn(1.0f, pz);
        float r0 = 0.f, r1 = 0.f;
        if (FAST && g.lv.sz[l] == 0 && !g.lv.hashed[l]) {
            #pragma unroll
            for (int c = 0; c < 4; c++) {
                const float w = __fmul_rn((c & 1) ? px : qx, (c >> 1) ? py : qy);
                r0 = __fmaf_rn(w, v[i][c].x, r0);
                r1 = __fmaf_rn(w, v[i][c].y, r1);
            }
        } else {
            #pragma unroll
            for (int c = 0; c < 8; c++) {
                // w = ((1 * wx) * wy) * wz in the reference's order (d = 0,1,2)
                const float w = __fmul_rn(__fmul_rn((c & 1) ? px : qx, ((c >> 1) & 1) ? py : qy), (c >> 2) ? pz : qz);
                r0 = __fmaf_rn(w, v[i][c].x, r0);
                r1 = __fmaf_rn(w, v[i][c].y, r1);
            }
        }
        out[i] = oob ? make_float2(0.f, 0.f) : make_float2(r0, r1);
    }
}

template <int NL>
__device__ __forceinline__ void grid2_levels(const GridDesc& g, int l0, float x, float y, float2 (&out)[NL]) {
    const bool oob = x < 0 || x > 1 || y < 0 || y > 1;
    if (oob) { x = 0.5f; y = 0.5f; }
    float fx[NL], fy[NL];
    float2 v[NL][4];
    #pragma unroll
    for (int i = 0; i < NL; i++) {
        const int l = l0 + i;
        const float scale = g.lv.scale[l];
        float px = __fmaf_rn(x, scale, 0.5f), py = __fmaf_rn(y, scale, 0.5f);
        const uint32_t gx = (uint32_t)floorf(px), gy = (uint32_t)floorf(py);
        px = __fsub_rn(px, (float)gx); py = __fsub_rn(py, (float)gy);
        if (g.interp == 1) { px = smooth_(px); py = smooth_(py); }
        fx[i] = px; fy[i] = py;
        uint32_t idx[4];
        corner_index2(g.lv, l, gx, gy, idx);
        const float2* __restrict__ tab = g.lbase[l];
        #pragma unroll
        for (int c = 0; c < 4; c++) v[i][c] = __ldg(tab + idx[c]);
    }
    #pragma unroll
    for (int i = 0; i < NL; i++) {
        const float px = fx[i], py = fy[i];
        const float qx = __fsub_rn(1.0f, px), qy = __fsub_rn(1.0f, py);
        float r0 = 0.f, r1 = 0.f;
        #pragma unroll
        for (int c = 0; c < 4; c++) {
            const float w = __fmul_rn((c & 1) ? px : qx, (c >> 1) ? py : qy);
            r0 = __fmaf_rn(w, v[i][c].x, r0);
            r1 = __fmaf_rn(w, v[i][c].y, r1);
        }
        out[i] = oob ? make_float2(0.f, 0.f) : make_float2(r0, r1);
    }
}

// single-level conveniences (fp32 SIMT kernels: one (sample, level) task per thread)
__device__ __forceinline__ float2 grid3_sample(const GridDesc& g, int level, float x, float y, float z) {
    float2 o[1];
    grid3_levels<1>(g, level, x, y, z, o);
    return o[0];
}
__device__ __forceinline__ float2 grid2_sample(const GridDesc& g, int level, float x, float y) {
    float2 o[1];
    grid2_levels<1>(g, level, x, y, o);
    return o[0];
}

// map a world coordinate in [-bound, bound] to [0,1] exactly as grid.py:149 does in fp32
__device__ __forceinline__ float to_unit(float x, float bound) { return __fdiv_rn(__fadd_rn(x, bound), 2.0f * bound); }

// Real SH, degree 4 (16 values), Condon-Shortley phase, unit-norm input assumed
// (values of shencoder.cu:43-68; written from the definition with shared sub-terms).
__device__ __forceinline__ void sh4(float x, float y, float z, float* o) {
    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
    o[0] = 0.28209479177387814f;
    o[1] = -0.48860251190291987f * y;
    o[2] = 0.48860251190291987f * z;
    o[3] = -0.48860251190291987f * x;
    o[4] = 1.0925484305920792f * xy;
    o[5] = -1.0925484305920792f * yz;
    o[6] = 0.94617469575755997f * zz - 0.31539156525251999f;
    o[7] = -1.0925484305920792f * xz;
    o[8] = 0.54627421529603959f * (xx - yy);
    const float a = yy - 3.0f * xx;       // -3x^2 + y^2
    const float b = 3.0f * yy - xx;       // -x^2 + 3y^2
    const float c = 1.0f - 5.0f * zz;
    o[9] = 0.59004358992664352f * y * a;
    o[10] = 2.8906114426405538f * xy * z;
    o[11] = 0.45704579946446572f * y * c;
    o[12] = 0.3731763325901154f * z * (5.0f * zz - 3.0f);
    o[13] = 0.45704579946446572f * x * c;
    o[14] = 1.4453057213202769f * z * (xx - yy);
    o[15] = 0.59004358992664352f * x * b;
}

}  // namespace gf
