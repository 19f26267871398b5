// libgfrender: warp-specialised, two-kernel tcgen05 field pipeline (precision = 1, the default).
//
// One 128-sample tile needs, per layer, 128 accumulator + 64..128 operand columns of the SM's 512 tensor-memory columns, so only two
// tiles can be inside the MLP chain at once, and the 184 KB of fp16 weights of the whole field would leave no shared memory to gather
// ahead (the single-kernel variant of round 1 alternated gathers and MMAs: 16.8 ms/frame, issue slots 37 % busy; removed in round 2).
// Splitting the field at the ambient coordinate halves the weights each kernel keeps resident, which buys a 6-deep ring of feature
// tiles and lets DEDICATED PRODUCER WARPS gather ahead while two consumer streams run the MMA chain back to back:
//
//   k_tc_amb     producers (8 warps): 3-D grid gather -> fp16 hi/lo feature tile in the smem ring (+ hi copy to HBM)
//                consumers (2 x 4 warps, one thread per sample row = TMEM lane):
//                    ambient L0 (split precision, SS) -> ambient L1 (split precision, TS) -> 128->2 in fp32 -> tanh
//                    -> ambient coordinate (8 B/sample) to HBM
//   k_tc_sigcol  producers: 64 B/sample of position features back from HBM + 2-D ambient-grid gather -> smem ring
//                consumers: sigma L0 (SS) -> sigma L1 (TS) -> merged sigma-L2 x colour-L0 (+ SH, SS) -> colour L1 -> sigma, rgb
//
// Producer -> consumer hand-off: one `full` mbarrier per ring slot (256 producer arrivals, generic->async proxy fence before
// the arrive), one `empty` mbarrier per slot (arrived by the stream leader once the tcgen05.commit of the last MMA reading
// the slot has completed).  Extra HBM traffic: 64 + 8 B/sample written and read once (4.8 GB/frame at 512x512x128, <10 %
// of the algorithmic gather bytes).
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>

#include "gf_model.cuh"
#include "gf_tc.cuh"

namespace gf {

constexpr int SP_THREADS = 512;        // kernel B: warps 0-7 producers, 8-11 consumer stream 0, 12-15 consumer stream 1
// kernel A: GF_A_PROD_WG producer warpgroups, default 2 (same warp roles as kernel B).  3 (warps 0-11 producers, 12-15 stream 0, 16-19 stream 1) was
// measured SLOWER twice: with 96 registers for every thread 10.09 vs 8.75 ms per frame (the same 4-level batch takes 3,300 instead of 2,450 cycles, the
// split epilogue 2,700 instead of 2,050), and with setmaxnreg (producers 112, consumers 72 registers, non-pipelined consumer epilogues) 8.72 / 8.98 vs
// 8.57 / 8.66 ms.  More gathering warps do not help: the SM's issue slots bound this kernel (profiles/r02_summary.md section 7).  Note for setmaxnreg:
// the increase is served from the registers the CTA itself released (USETMAXREG.TRY_ALLOC.CTAPOOL) -- the launch-time slack does not count, so
// consumers 80 / producers 112 (256 x 16 < 384 x 16) spins forever.
#ifndef GF_A_PROD_WG
#define GF_A_PROD_WG 2
#endif
constexpr int SPA_PROD_WG = GF_A_PROD_WG, SPA_PROD_THREADS = 128 * SPA_PROD_WG, SPA_THREADS = SPA_PROD_THREADS + 256;
static_assert(SPA_PROD_WG == 2 || SPA_PROD_WG == 3, "2 or 3 producer warpgroups");
constexpr int SP_NSLOT = 6;            // feature-tile ring depth
constexpr uint32_t SP_TILE_BYTES = 128 * 128;

// ---- weight images ---------------------------------------------------------------------------------------------------
// kernel A (80 KB)
constexpr uint32_t WA_A0 = 0;                               // [128]: k 0..31 Wa0_hi, k 32..63 Wa0_lo
constexpr uint32_t WA_A1H = WA_A0 + 128 * 128;              // 2 chunks x [128]
constexpr uint32_t WA_A1L = WA_A1H + 2 * 128 * 128;
constexpr uint32_t WA_TOTAL = WA_A1L + 2 * 128 * 128;       // 81,920
// kernel B (104 KB)
constexpr uint32_t WB2_SIG0 = 0;                            // [128] k 0..63
constexpr uint32_t WB2_SIG1 = WB2_SIG0 + 128 * 128;         // 2 chunks x [128]
constexpr uint32_t WB2_MRG = WB2_SIG1 + 2 * 128 * 128;      // 2 chunks x [144]
constexpr uint32_t WB2_COL1 = WB2_MRG + 2 * 144 * 128;      // 2 chunks x [16]
constexpr uint32_t WB2_SH = WB2_COL1 + 2 * 16 * 128;        // [128]: k 0..15 colour-L0 SH columns
constexpr uint32_t WB2_TOTAL = WB2_SH + 128 * 128;          // 106,496
static_assert(WA_TOTAL == 81920 && WB2_TOTAL == 106496, "image sizes");
static_assert(WB2_MRG % 1024 == 0 && WB2_COL1 % 1024 == 0 && WB2_SH % 1024 == 0, "1024-byte aligned blocks");

// Tried and removed (measured, profiles/r02_summary.md): staging the whole 3-D level 0 (4,913 entries, 39 KB) into kernel A's spare shared
// memory with cp.async.bulk and serving its 8 corner loads per sample from there: 8.530 vs 8.536 ms/frame, l1tex hit rate 62.8 -> 54.5 %
// (the level was L1-resident anyway; only the remaining, colder loads are left in the statistic), +0.7 % instructions.  The dense coarse
// levels are not where the gathers cost: the producers are issue-bound, not L1-bound.

// shared-memory layout (same skeleton for both kernels; W = weight image bytes)
template <uint32_t W>
struct SpSmem {
    static constexpr uint32_t F = W;
    static constexpr uint32_t DIR = F + SP_NSLOT * SP_TILE_BYTES;    // per slot: 128 x float4 view directions (kernel B)
    static constexpr uint32_t BIAS = DIR + SP_NSLOT * 128 * 16;      // 128 floats
    // per-kernel extras (9 KB): kernel A: W2 = ambient output layer, 64 x float4 {w0[c], w0[c+1], w1[c], w1[c+1]}; POS = 2 x 256 x float4 per-thread
    // staged sample positions.  kernel B: AP = 2 x 256 x float2 per-thread staged ambient coordinates (over POS), RAY = 3 x 128 x u32 staged ray ids (over W2..)
    static constexpr uint32_t W2 = BIAS + 512;
    static constexpr uint32_t POS = W2 + 1024;
    static constexpr uint32_t AP = POS, RAY = POS + 2 * 256 * 8;
    static constexpr uint32_t BAR = POS + 2 * 384 * 16;              // wbar, full[NSLOT], empty[NSLOT], mma[2]
    static constexpr uint32_t TMEM = BAR + 8 * (1 + 2 * SP_NSLOT + 4);   // barriers: wbar, full[NSLOT], empty[NSLOT], mma[2], early-layer-0[2]
    static constexpr uint32_t TOTAL = TMEM + 16;
    static constexpr uint32_t BYTES = TOTAL + 1024;
};
static_assert(SpSmem<WB2_TOTAL>::BYTES <= 232448, "exceeds 227 KB");

// TMEM columns per consumer stream (256): D at +0; ambient phase A_hi +128 / A_lo +192; later layers A at +144
constexpr uint32_t SP_TM_STREAM = 256, SP_TM_AHI = 128, SP_TM_ALO = 192, SP_TM_A = 144;

struct TcPackSrc2 {
    const float *a0, *a1, *s0, *s1, *s2, *c0, *c1;
    int cond, ind, G;
};

__device__ __forceinline__ void put_half2(uint8_t* img, uint32_t block, uint32_t rows, uint32_t n, uint32_t k, float v, bool lo) {
    const uint32_t chunk = k >> 6, kk = k & 63;
    const uint32_t off = block + chunk * rows * 128 + sw128(n, kk >> 3) + (kk & 7) * 2;
    const __half hi = __float2half_rn(v);
    *reinterpret_cast<__half*>(img + off) = lo ? __float2half_rn(v - __half2float(hi)) : hi;
}

__global__ void k_tc_pack_split(TcPackSrc2 s, uint8_t* __restrict__ imgA, uint8_t* __restrict__ imgB) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;   // (n, k) of a 144 x 128 index space
    const int n = i / 128, k = i % 128;
    if (n >= 144) return;
    const int a_in = 32 + s.cond, c_in = 16 + s.G + s.ind;
    if (n < 128) {
        if (k < 32) {
            const float w = s.a0[(size_t)n * a_in + k];
            put_half2(imgA, WA_A0, 128, n, k, w, false);
            put_half2(imgA, WA_A0, 128, n, 32 + k, w, true);
        }
        const float w1 = s.a1[(size_t)n * 128 + k];
        put_half2(imgA, WA_A1H, 128, n, k, w1, false);
        put_half2(imgA, WA_A1L, 128, n, k, w1, true);
        if (k < 64) put_half2(imgB, WB2_SIG0, 128, n, k, s.s0[(size_t)n * 64 + k], false);
        put_half2(imgB, WB2_SIG1, 128, n, k, s.s1[(size_t)n * 128 + k], false);
        float acc = 0.f;
        for (int j = 0; j < s.G; j++) acc = fmaf(s.c0[(size_t)n * c_in + 16 + j], s.s2[(size_t)(1 + j) * 128 + k], acc);
        put_half2(imgB, WB2_MRG, 144, n, k, acc, false);
        if (k < 16) put_half2(imgB, WB2_SH, 128, n, k, s.c0[(size_t)n * c_in + k], false);
    } else {
        put_half2(imgB, WB2_MRG, 144, n, k, n == 128 ? s.s2[k] : 0.f, false);
    }
    if (n < 16) put_half2(imgB, WB2_COL1, 16, n, k, n < 3 ? s.c1[(size_t)n * 128 + k] : 0.f, false);
}

// MMA completion for a consumer stream: every consumer thread polls the stream's mbarrier itself (parking three of the four warps on a
// named barrier while one polls was measured neutral, 8.45 vs 8.43 ms/frame, and removed).
__device__ __forceinline__ void stream_wait_mma(uint32_t bar_mma, uint32_t& phase) {
    mbar_wait(bar_mma, phase);
    phase ^= 1;
}


// -DGF_TC_TIMING=1 (experiment builds only): CTA 0 stamps clock64() at every phase boundary of its tiles TT_J0 .. TT_J0+TT_NJ-1 into the
// gf_tc_debug buffer, read back by scripts/tc_timeline.py.  Layout: long long [kernel 2][who 4: stream 0, stream 1, producer half 0, half 1][TT_NJ][8].
#ifndef GF_TC_TIMING
#define GF_TC_TIMING 0
#endif
#if GF_TC_TIMING
constexpr uint32_t TT_J0 = 96, TT_NJ = 64;
#define TT_STAMP(kern, who, j, k)                                                                                            \
    do {                                                                                                                     \
        if (a.dbg && blockIdx.x == 0 && (j) >= TT_J0 && (j) < TT_J0 + TT_NJ)                                                    \
            reinterpret_cast<long long*>(a.dbg)[((((kern) * 4 + (who)) * TT_NJ) + ((j) - TT_J0)) * 8 + (k)] = clock64();     \
    } while (0)
#define TT_LSTAMP(kern, who, j, k) do { if (lead_warp && elect_one_sync()) TT_STAMP(kern, who, j, k); } while (0)
#else
#define TT_STAMP(kern, who, j, k) do { } while (0)
#define TT_LSTAMP(kern, who, j, k) do { } while (0)
#endif

struct SpArgs {
    GridDesc grid;              // A: 3-D position grid; B: 2-D ambient grid
    float bound, inv2b;
    const uint8_t* wimg;
    const float* bias;          // A: per-frame cond bias [128]; B: individual-code bias [128] or null
    float w_amb2[256];          // A only
    FieldTcIO io;
    float* dbg;
};

// common prologue: barriers, TMEM, weights, bias.  Returns the TMEM base.
template <uint32_t W>
__device__ __forceinline__ uint32_t sp_setup(uint8_t* smem, uint32_t sbase, const SpArgs& a, const uint32_t* cuts, int ncuts, uint32_t nprod) {
    using L = SpSmem<W>;
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    float* bias = reinterpret_cast<float*>(smem + L::BIAS);
    if (tid == 0) {
        mbar_init(sbase + L::BAR, 1);
        for (int s = 0; s < SP_NSLOT; s++) {
            mbar_init(sbase + L::BAR + 8 * (1 + s), nprod);             // full: every producer thread arrives
            mbar_init(sbase + L::BAR + 8 * (1 + SP_NSLOT + s), 1);      // empty: the stream leader arrives
        }
        for (int s = 0; s < 4; s++) mbar_init(sbase + L::BAR + 8 * (1 + 2 * SP_NSLOT + s), 1);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc(sbase + L::TMEM, 512);
    if (tid < 128) bias[tid] = a.bias ? a.bias[tid] : 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (tid == 0) {
        mbar_expect_tx(sbase + L::BAR, W);
        for (int i = 0; i < ncuts; i++) bulk_g2s(sbase + cuts[i], a.wimg + cuts[i], cuts[i + 1] - cuts[i], sbase + L::BAR);
    }
    mbar_wait(sbase + L::BAR, 0);
    return *reinterpret_cast<uint32_t*>(smem + L::TMEM);
}

// ======================================================================================================================
// kernel A: 3-D gather -> ambient branch -> ambient coordinate + fp16 position features
// ======================================================================================================================
// ---- gathers with a RUN-TIME level index ------------------------------------------------------------------------------
// The producers' code must stay small: four instruction streams (2 producer + 2 consumer warps) share each scheduler's
// ~6 KB L0 / the SM's 32 KB L1.5 instruction cache, and the fully unrolled per-level code of the removed single-kernel variant (72 KB of SASS)
// left the producer warps starved for instructions (ncu: 45 % of their stall samples were no_instruction).  Here ONE
// copy of a 4-level batch serves both halves and both batches; level constants are indexed loads from the constant bank.
//
// 3-D position grid, 4 consecutive levels from l0.  Levels whose index drops z (gridencoder.cu:72 quirk) or are dense fetch the
// z+1 plane only when it exists.  Interpolation is bilinear per z-plane, then a lerp in z (the fp32 result differs from the
// reference's corner-order sum by rounding only; it is rounded to fp16 right after).
// ALLFLAT: every level of the batch drops z and is not hashed -> only the 4 corners of the z0 plane exist (uniform fast path).
// CONTIG: no level of the batch is hashed.  The tables are the padded images of GridLevels::pad, so a cell's corners are rows of 2 adjacent
// entries from the masked base index, on wrapping levels too: one address per row, the +1 corner an immediate offset of the load (uniform fast
// path).  Only batches with a hashed level compute, mask and address each corner.
// floor() of a grid coordinate without the conversion pipe.  p = x * scale + 0.5 lies in [0.5, 2^23): adding 2^23 with round-toward-minus-infinity
// leaves floor(p) in the mantissa, exactly; the integer is the low 23 bits and the float is recovered by an exact subtraction.  Replaces F2I.FLOOR +
// I2F (two conversion-pipe instructions, ~4x the issue cost and ~3x the latency of an FADD, in front of every level's dependent address chain) by
// FADD.RM + LOP + FADD.  Bit-identical to floorf / (float) for this range.  -DGF_FAST_FLOOR=0 restores the conversions (A/B).
// experiment switch: compile the smoothstep interpolation out (linear-interpolation models only; measurement aid)
#ifndef GF_ASSUME_LINEAR
#define GF_ASSUME_LINEAR 0
#endif
#ifndef GF_FAST_FLOOR
#define GF_FAST_FLOOR 1
#endif
__device__ __forceinline__ void floor_split2(float2& p, uint32_t (&g)[2]) {
#if GF_FAST_FLOOR
    const float2 t = fadd2_rm(p, bcast2(8388608.0f));
    p = fsub2(p, fsub2(t, bcast2(8388608.0f)));
    g[0] = __float_as_uint(t.x) & 0x7fffffu;
    g[1] = __float_as_uint(t.y) & 0x7fffffu;
#else
    g[0] = (uint32_t)floorf(p.x); g[1] = (uint32_t)floorf(p.y);
    p = fsub2(p, make_float2((float)g[0], (float)g[1]));
#endif
}
// v * v * (3 - 2 v) on both lanes, in the scalar smooth_'s order
__device__ __forceinline__ float2 smooth2(float2 v) { return fmul2(fmul2(v, v), fsub2(bcast2(3.0f), fadd2(v, v))); }

// The per-level coordinate arithmetic runs on LEVEL PAIRS (lane 0 = level l, lane 1 = level l + 1) in packed fp32, and the interpolation on
// CHANNEL PAIRS (both channels of a corner share its weight, which is broadcast to the two lanes): every lane performs the same IEEE
// operations in the same order as the scalar form, so the features are bit-identical to it.
template <bool ALLFLAT, bool CONTIG>
__device__ __forceinline__ void gather3_dyn4(const GridDesc& g, int l0, float x, float y, float z, float2 (&out)[4]) {
    static_assert(CONTIG || !ALLFLAT, "an ALLFLAT batch has no hashed level");
    float2 fx[2], fy[2], fz[2];           // fractional coordinates of levels (l0 + 2k, l0 + 2k + 1)
    float2 v[4][8];
    #pragma unroll
    for (int k = 0; k < 2; k++) {
        const int l = l0 + 2 * k;
        const float2 scale = make_float2(g.lv.scale[l], g.lv.scale[l + 1]);
        float2 px = ffma2(bcast2(x), scale, bcast2(0.5f)), py = ffma2(bcast2(y), scale, bcast2(0.5f)), pz = ffma2(bcast2(z), scale, bcast2(0.5f));
        uint32_t gx[2], gy[2], gz[2];
        floor_split2(px, gx); floor_split2(py, gy); floor_split2(pz, gz);
        if (!GF_ASSUME_LINEAR && g.interp == 1) { px = smooth2(px); py = smooth2(py); pz = smooth2(pz); }
        #pragma unroll
        for (int h = 0; h < 2; h++) {
            const int i = 2 * k + h;
            const float2* __restrict__ tab = g.lbase[l + h];
            const uint32_t mask = g.lv.mask[l + h], sy = g.lv.sy[l + h], sz = g.lv.sz[l + h];
            const bool hashed = !CONTIG && g.lv.hashed[l + h] != 0;
            const bool has_z = !ALLFLAT && (hashed || sz != 0);
            if (CONTIG) {
                const float2* __restrict__ r0 = tab + ((ALLFLAT ? gx[h] + gy[h] * sy : gx[h] + gy[h] * sy + gz[h] * sz) & mask);
                const float2* __restrict__ r1 = r0 + sy;
                v[i][0] = __ldg(r0); v[i][1] = __ldg(r0 + 1); v[i][2] = __ldg(r1); v[i][3] = __ldg(r1 + 1);
                if (!ALLFLAT) {
                    v[i][4] = has_z ? __ldg(r0 + sz) : make_float2(0.f, 0.f); v[i][5] = has_z ? __ldg(r0 + sz + 1) : make_float2(0.f, 0.f);
                    v[i][6] = has_z ? __ldg(r1 + sz) : make_float2(0.f, 0.f); v[i][7] = has_z ? __ldg(r1 + sz + 1) : make_float2(0.f, 0.f);
                    if (!has_z) { if (h == 0) pz.x = 0.f; else pz.y = 0.f; }
                }
                continue;
            }
            uint32_t idx[8];
            if (hashed) {
                const uint32_t y0 = gy[h] * HASH_P1, y1 = y0 + HASH_P1, z0 = gz[h] * HASH_P2, z1 = z0 + HASH_P2;
                const uint32_t x0 = gx[h], x1 = gx[h] + 1;
                idx[0] = x0 ^ y0 ^ z0; idx[1] = x1 ^ y0 ^ z0; idx[2] = x0 ^ y1 ^ z0; idx[3] = x1 ^ y1 ^ z0;
                idx[4] = x0 ^ y0 ^ z1; idx[5] = x1 ^ y0 ^ z1; idx[6] = x0 ^ y1 ^ z1; idx[7] = x1 ^ y1 ^ z1;
            } else {
                const uint32_t b = gx[h] + gy[h] * sy + gz[h] * sz;
                idx[0] = b; idx[1] = b + 1; idx[2] = b + sy; idx[3] = b + sy + 1;
                idx[4] = b + sz; idx[5] = b + sz + 1; idx[6] = b + sz + sy; idx[7] = b + sz + sy + 1;
            }
            #pragma unroll
            for (int c = 0; c < 4; c++) v[i][c] = __ldg(tab + (idx[c] & mask));
            if (!ALLFLAT) {
                #pragma unroll
                for (int c = 4; c < 8; c++) v[i][c] = has_z ? __ldg(tab + (idx[c] & mask)) : make_float2(0.f, 0.f);
                if (!has_z) { if (h == 0) pz.x = 0.f; else pz.y = 0.f; }
            }
        }
        fx[k] = px; fy[k] = py; fz[k] = pz;
    }
    #pragma unroll
    for (int k = 0; k < 2; k++) {
        const float2 qx = fsub2(bcast2(1.0f), fx[k]), qy = fsub2(bcast2(1.0f), fy[k]);
        const float2 w00 = fmul2(qx, qy), w10 = fmul2(fx[k], qy), w01 = fmul2(qx, fy[k]), w11 = fmul2(fx[k], fy[k]);
        #pragma unroll
        for (int h = 0; h < 2; h++) {
            const int i = 2 * k + h;
            const float a00 = h ? w00.y : w00.x, a10 = h ? w10.y : w10.x, a01 = h ? w01.y : w01.x, a11 = h ? w11.y : w11.x;
            const float2 a = ffma2(bcast2(a11), v[i][3], ffma2(bcast2(a01), v[i][2], ffma2(bcast2(a10), v[i][1], fmul2(bcast2(a00), v[i][0]))));
            if (ALLFLAT) { out[i] = a; continue; }
            const float2 b = ffma2(bcast2(a11), v[i][7], ffma2(bcast2(a01), v[i][6], ffma2(bcast2(a10), v[i][5], fmul2(bcast2(a00), v[i][4]))));
            out[i] = ffma2(bcast2(h ? fz[k].y : fz[k].x), fsub2(b, a), a);
        }
    }
}

// 1 when none of the n levels from l0 is hashed (uniform: level constants)
__device__ __forceinline__ bool levels_unhashed(const GridLevels& lv, int l0, int n) {
    bool c = true;
    #pragma unroll
    for (int q = 0; q < n; q++) c = c && lv.hashed[l0 + q] == 0;
    return c;
}
// unit u (levels 4u..4u+3) of the 3-D grid, with the batch's uniform ALLFLAT / CONTIG properties (ALLFLAT implies CONTIG)
__device__ __forceinline__ void gather3_unit(const GridDesc& g, uint32_t u, bool flat, bool contig, float x, float y, float z, float2 (&out)[4]) {
    if (flat) gather3_dyn4<true, true>(g, 4 * u, x, y, z, out);
    else if (contig) gather3_dyn4<false, true>(g, 4 * u, x, y, z, out);
    else gather3_dyn4<false, false>(g, 4 * u, x, y, z, out);
}

// 2-D ambient grid, 8 consecutive levels from l0 (32 gathers in flight); level pairs, channel pairs and CONTIG as in gather3_dyn4
template <bool CONTIG>
__device__ __forceinline__ void gather2_dyn8(const GridDesc& g, int l0, float x, float y, float2 (&out)[8]) {
    const bool oob = x < 0 || x > 1 || y < 0 || y > 1;            // tanh output mapped to [0,1]: cannot happen, kept for safety
    if (oob) { x = 0.5f; y = 0.5f; }
    float2 fx[4], fy[4];
    float2 v[8][4];
    #pragma unroll
    for (int k = 0; k < 4; k++) {
        const int l = l0 + 2 * k;
        const float2 scale = make_float2(g.lv.scale[l], g.lv.scale[l + 1]);
        float2 px = ffma2(bcast2(x), scale, bcast2(0.5f)), py = ffma2(bcast2(y), scale, bcast2(0.5f));
        uint32_t gx[2], gy[2];
        floor_split2(px, gx); floor_split2(py, gy);
        if (!GF_ASSUME_LINEAR && g.interp == 1) { px = smooth2(px); py = smooth2(py); }
        fx[k] = px; fy[k] = py;
        #pragma unroll
        for (int h = 0; h < 2; h++) {
            const float2* __restrict__ tab = g.lbase[l + h];
            const uint32_t mask = g.lv.mask[l + h], sy = g.lv.sy[l + h];
            if (CONTIG) {
                const float2* __restrict__ r0 = tab + ((gx[h] + gy[h] * sy) & mask), * __restrict__ r1 = r0 + sy;
                v[2 * k + h][0] = __ldg(r0); v[2 * k + h][1] = __ldg(r0 + 1); v[2 * k + h][2] = __ldg(r1); v[2 * k + h][3] = __ldg(r1 + 1);
                continue;
            }
            uint32_t idx[4];
            if (g.lv.hashed[l + h]) {
                const uint32_t y0 = gy[h] * HASH_P1, y1 = y0 + HASH_P1;
                idx[0] = gx[h] ^ y0; idx[1] = (gx[h] + 1) ^ y0; idx[2] = gx[h] ^ y1; idx[3] = (gx[h] + 1) ^ y1;
            } else {
                const uint32_t b = gx[h] + gy[h] * sy;
                idx[0] = b; idx[1] = b + 1; idx[2] = b + sy; idx[3] = b + sy + 1;
            }
            #pragma unroll
            for (int c = 0; c < 4; c++) v[2 * k + h][c] = __ldg(tab + (idx[c] & mask));
        }
    }
    #pragma unroll
    for (int k = 0; k < 4; k++) {
        const float2 qx = fsub2(bcast2(1.0f), fx[k]), qy = fsub2(bcast2(1.0f), fy[k]);
        const float2 w00 = fmul2(qx, qy), w10 = fmul2(fx[k], qy), w01 = fmul2(qx, fy[k]), w11 = fmul2(fx[k], fy[k]);
        #pragma unroll
        for (int h = 0; h < 2; h++) {
            const int i = 2 * k + h;
            const float a00 = h ? w00.y : w00.x, a10 = h ? w10.y : w10.x, a01 = h ? w01.y : w01.x, a11 = h ? w11.y : w11.x;
            const float2 a = ffma2(bcast2(a11), v[i][3], ffma2(bcast2(a01), v[i][2], ffma2(bcast2(a10), v[i][1], fmul2(bcast2(a00), v[i][0]))));
            out[i] = oob ? make_float2(0.f, 0.f) : a;
        }
    }
}

template <bool DBG>
__global__ void __launch_bounds__(SPA_THREADS, 1) k_tc_amb(const SpArgs a) {
    using L = SpSmem<WA_TOTAL>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const uint32_t sbase = smem_u32(smem);
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    const uint32_t M = a.io.M_dev ? *a.io.M_dev : a.io.M_host;
    if (M == 0) return;                      // e.g. the extra round of a frame whose budget is 0: skip weight staging / TMEM allocation
    const uint32_t cuts[4] = {0, WA_A1H, WA_A1L, WA_TOTAL};
    if (tid < 64)          // ambient output layer -> shared memory (read as broadcast LDS.128 by the consumers); visible after sp_setup's __syncthreads
        sts128f(sbase + L::W2 + 16 * tid, make_float4(a.w_amb2[2 * tid], a.w_amb2[2 * tid + 1], a.w_amb2[128 + 2 * tid], a.w_amb2[128 + 2 * tid + 1]));
    const uint32_t tmem_base = sp_setup<WA_TOTAL>(smem, sbase, a, cuts, 3, SPA_PROD_THREADS);
    const uint32_t bias_cond = sbase + L::BIAS;
    const uint32_t bar_full = sbase + L::BAR + 8, bar_empty = sbase + L::BAR + 8 * (1 + SP_NSLOT);
    const uint32_t num_tiles = (M + 127) / 128;
    const uint32_t my_tiles = num_tiles > blockIdx.x ? (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp < 4 * SPA_PROD_WG) {
        // ------------------------------------------------ producers ------------------------------------------------
#if GF_A_PROD_WG == 3
        // 640 threads start with 96 registers each; the gathering warpgroups take 112 (32 loads in flight need them), the consumer warpgroups give
        // theirs back (72: non-pipelined epilogues).  The increase is served from the registers the CTA itself released (CTAPOOL): 256 x 24 = 384 x 16
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
#endif
        const uint32_t half = tid >> 7, row = tid & 127;     // half = producer warpgroup 0 .. SPA_PROD_WG-1
        uint32_t flat_units = 0, contig_units = 0;     // bit u: levels 4u..4u+3 all drop z and are not hashed / are not hashed
        #pragma unroll
        for (int u = 0; u < 4; u++) {
            bool flat = true;
            #pragma unroll
            for (int q = 0; q < 4; q++) flat = flat && a.grid.lv.sz[4 * u + q] == 0 && a.grid.lv.hashed[4 * u + q] == 0;
            flat_units |= (flat ? 1u : 0u) << u;
            contig_units |= (levels_unhashed(a.grid.lv, 4 * u, 4) ? 1u : 0u) << u;
        }
        // This warpgroup's units (4 levels each) of a row.  Two warpgroups: u = wg and wg + 2 (one 8-corner coarse unit + one z-dropped fine unit
        // each).  Three: the cheapest pair of units (cost 2 per 8-corner unit, 1 per z-dropped one) shares a warpgroup, the other two units get one each.
        uint32_t my_u0, my_u1, my_nu;
        if (SPA_PROD_WG == 2) { my_u0 = half; my_u1 = half + 2; my_nu = 2; }
        else {
            uint32_t best = 99, bp = 2, bq = 3;
            #pragma unroll
            for (uint32_t p = 0; p < 4; p++)
                #pragma unroll
                for (uint32_t q = p + 1; q < 4; q++) {
                    const uint32_t c = 4 - ((flat_units >> p) & 1) - ((flat_units >> q) & 1);
                    if (c <= best) { best = c; bp = p; bq = q; }      // <=: prefer the finest pair on ties
                }
            uint32_t singles[2], ns = 0;
            #pragma unroll
            for (uint32_t u = 0; u < 4; u++) if (u != bp && u != bq) { if (ns == 0) singles[0] = u; else singles[1] = u; ns++; }
            if (half == 2) { my_u0 = bp; my_u1 = bq; my_nu = 2; }
            else { my_u0 = half == 0 ? singles[0] : singles[1]; my_u1 = my_u0; my_nu = 1; }
        }
        // The row's position is staged ONE TILE AHEAD into this thread's own 16 bytes of shared memory with cp.async (double-buffered).  A plain
        // register prefetch did not help (8.46 vs 8.48 ms): ptxas put the prefetch LDG on the same scoreboard as the uniform constant loads at the
        // top of the loop, so the first use of the CURRENT position waited for the NEXT tile's DRAM access (7 % of the kernel's stall samples on
        // that one FADD, ~750 of the producers' 5,280 cycles per tile; profiles/r02_summary.md section 7).  cp.async completion is tracked by the
        // async-group counter instead.
        const uint32_t pos_s = sbase + L::POS + 16 * tid;
        auto stage_pos = [&](uint32_t j) {
            const uint32_t i = (blockIdx.x + j * gridDim.x) * 128 + row;
            if (j < my_tiles && i < M) {
                const uint32_t dst = pos_s + (j & 1) * (SPA_PROD_THREADS * 16);
                if (a.io.pos4) cp_async16(dst, a.io.pos4 + i);
                else { cp_async4(dst, a.io.xyzs + 3 * (size_t)i); cp_async4(dst + 4, a.io.xyzs + 3 * (size_t)i + 1); cp_async4(dst + 8, a.io.xyzs + 3 * (size_t)i + 2); }
            }
            cp_async_commit();
        };
        stage_pos(0);
        #pragma unroll 1
        for (uint32_t j = 0; j < my_tiles; j++) {
            const uint32_t tile = blockIdx.x + j * gridDim.x, slot = j % SP_NSLOT, n = j / SP_NSLOT;
            const uint32_t i = tile * 128 + row;
            const bool valid = i < M;
            cp_async_wait_all();
            float4 cur = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) cur = lds128(pos_s + (j & 1) * (SPA_PROD_THREADS * 16));
            const float x = cur.x, y = cur.y, z = cur.z;
            stage_pos(j + 1);
            float ux = (x + a.bound) * a.inv2b, uy = (y + a.bound) * a.inv2b, uz = (z + a.bound) * a.inv2b;
            // out-of-range inputs encode to 0 (gridencoder.cu:110-135): sample the centre, zero the result
            const bool oob = ux < 0 || ux > 1 || uy < 0 || uy > 1 || uz < 0 || uz > 1;
            if (oob) { ux = 0.5f; uy = 0.5f; uz = 0.5f; }
            if (row == 0 && half < 2) TT_STAMP(0, 2 + half, j, 0);
            mbar_wait(bar_empty + 8 * slot, (n & 1) ^ 1);                 // slot released by the consumer of its previous use
            if (row == 0 && half < 2) TT_STAMP(0, 2 + half, j, 1);
            const uint32_t F = sbase + L::F + slot * SP_TILE_BYTES;
            uint4 keep0 = make_uint4(0, 0, 0, 0), keep1 = keep0;
            #pragma unroll 1
            for (uint32_t b = 0; b < my_nu; b++) {
                const uint32_t u = b == 0 ? my_u0 : my_u1;
                float2 f[4];
                gather3_unit(a.grid, u, (flat_units >> u) & 1, (contig_units >> u) & 1, ux, uy, uz, f);
                if (oob) { f[0] = f[1] = f[2] = f[3] = make_float2(0.f, 0.f); }
                uint4 hi, lo;
                pack_hilo_h2(f[0], hi.x, lo.x); pack_hilo_h2(f[1], hi.y, lo.y); pack_hilo_h2(f[2], hi.z, lo.z); pack_hilo_h2(f[3], hi.w, lo.w);
                sts128(F + sw128(row, u), hi);
                sts128(F + sw128(row, 4 + u), lo);
                if (b == 0) keep0 = hi; else keep1 = hi;
                if (row == 0 && half < 2) TT_STAMP(0, 2 + half, j, 2 + b);
                if (row == 0 && half < 2 && my_nu == 1) TT_STAMP(0, 2 + half, j, 3);
            }
            fence_async_smem();
            mbar_arrive(bar_full + 8 * slot);
            // the fp16 features for kernel B go to HBM AFTER the hand-off: fence.proxy.async is a MEMBAR.ALL.CTA in SASS and would otherwise wait
            // for these global stores to be acknowledged before the tile can be handed to the consumers
            if (valid) {
                a.io.feat_hi[(size_t)i * 4 + my_u0] = keep0;
                if (my_nu == 2) a.io.feat_hi[(size_t)i * 4 + my_u1] = keep1;
            }
            if (row == 0 && half < 2) TT_STAMP(0, 2 + half, j, 4);
        }
    } else {
        // ------------------------------------------------ consumers ------------------------------------------------
        // warp-uniform copies of the warp index and the TMEM base: the tcgen05.mma operands derived from them then live in uniform registers.
        // Derived from threadIdx / a shared-memory load they were per-thread values, and every MMA was issued through an ELECT / R2UR
        // broadcast loop of 13 instructions (~75 cycles per MMA on the stream's critical path, longer than the MMA itself).
#if GF_A_PROD_WG == 3
        asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
#endif
        const uint32_t warp_u = __shfl_sync(0xffffffffu, warp, 0), tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const uint32_t stream = (warp_u - 4 * SPA_PROD_WG) >> 2, row = tid & 127;
        const uint32_t t_d = tmem_u + (((warp_u & 3) * 32) << 16) + stream * SP_TM_STREAM;
        const uint32_t m_d = tmem_u + stream * SP_TM_STREAM;
        const uint32_t bar_mma = sbase + L::BAR + 8 * (1 + 2 * SP_NSLOT + stream);
        const uint32_t w_addr = sbase;
        // One elected lane of the stream's first warp waits on / arrives at the ring barriers and issues the MMAs.  The region must be guarded by
        // a warp-uniform test followed DIRECTLY by elect.sync (the CUTLASS idiom): only then does ptxas know that a single thread runs it and emit
        // the tcgen05.mma instructions back to back.  Guarded by `threadIdx == x` every MMA was wrapped in an ELECT / R2UR / branch loop of 11-13
        // instructions (~75 cycles per MMA on the stream's critical path -- longer than the 64 tensor-pipe cycles of the MMA itself).
        const bool lead_warp = (warp_u & 3) == 0;
        uint32_t phase = 0;
        for (uint32_t j = stream; j < my_tiles; j += 2) {
            const uint32_t tile = blockIdx.x + j * gridDim.x, slot = j % SP_NSLOT, n = j / SP_NSLOT;
            const uint32_t i = tile * 128 + row;
            float* dbg = (DBG && a.dbg && tile == 0) ? a.dbg + (size_t)row * 144 : nullptr;   // DBG = false: folds every dump away
            const uint32_t f_addr = sbase + L::F + slot * SP_TILE_BYTES;
            tc_fence_before();
            bar_named(1 + stream, 128);                                   // previous tile's accumulator reads are done
            if (lead_warp && elect_one_sync()) {
                TT_STAMP(0, stream, j, 0);
                mbar_wait(bar_full + 8 * slot, n & 1);
                TT_STAMP(0, stream, j, 1);
                tc_fence_after();
                // split precision: F_hi W_hi + F_lo W_hi + F_hi W_lo  (K = 32 each)
                #pragma unroll
                for (int k = 0; k < 2; k++) mma_ss(m_d, smem_desc(f_addr + 32 * k), smem_desc(w_addr + WA_A0 + 32 * k), idesc_f16(128), k);
                #pragma unroll
                for (int k = 0; k < 2; k++) mma_ss(m_d, smem_desc(f_addr + 64 + 32 * k), smem_desc(w_addr + WA_A0 + 32 * k), idesc_f16(128), 1);
                #pragma unroll
                for (int k = 0; k < 2; k++) mma_ss(m_d, smem_desc(f_addr + 32 * k), smem_desc(w_addr + WA_A0 + 64 + 32 * k), idesc_f16(128), 1);
                mma_commit(bar_mma);
            }
            stream_wait_mma(bar_mma, phase);
            tc_fence_after();
            TT_LSTAMP(0, stream, j, 2);
            if (lead_warp && elect_one_sync()) mbar_arrive(bar_empty + 8 * slot);                // the feature tile has been consumed
#if GF_A_PROD_WG == 3
            epilogue_relu_to_A_n<true, 4>(t_d, t_d + SP_TM_AHI, t_d + SP_TM_ALO, 0, bias_cond, dbg ? dbg + 0 * 128 * 144 : nullptr);      // 80-register budget
#else
            epilogue_split_to_A_pipe(t_d, t_d + SP_TM_AHI, t_d + SP_TM_ALO, bias_cond, dbg ? dbg + 0 * 128 * 144 : nullptr);
#endif
            TT_LSTAMP(0, stream, j, 3);
            tc_fence_before();
            bar_named(1 + stream, 128);
            if (lead_warp && elect_one_sync()) {
                TT_STAMP(0, stream, j, 4);
                tc_fence_after();
                #pragma unroll
                for (int k = 0; k < 8; k++)
                    mma_ts(m_d, m_d + SP_TM_AHI + 8 * k, smem_desc(w_addr + WA_A1H + (k >> 2) * (128 * 128) + 32 * (k & 3)), idesc_f16(128), k);
                #pragma unroll
                for (int k = 0; k < 8; k++)
                    mma_ts(m_d, m_d + SP_TM_ALO + 8 * k, smem_desc(w_addr + WA_A1H + (k >> 2) * (128 * 128) + 32 * (k & 3)), idesc_f16(128), 1);
                #pragma unroll
                for (int k = 0; k < 8; k++)
                    mma_ts(m_d, m_d + SP_TM_AHI + 8 * k, smem_desc(w_addr + WA_A1L + (k >> 2) * (128 * 128) + 32 * (k & 3)), idesc_f16(128), 1);
                mma_commit(bar_mma);
            }
            stream_wait_mma(bar_mma, phase);
            tc_fence_after();
            TT_LSTAMP(0, stream, j, 5);
            // ambient output layer (128 -> 2) in fp32 from the accumulator; tanh.  Weights come from shared memory as broadcast LDS.128 (one per
            // column pair and both outputs): indexing the kernel-parameter copy with the loop variable compiled to 128 LDC.64 per row, and the
            // constant path's throughput made this phase 2,400 cycles per tile (the longest of the stream's chain; tc_timeline).  The accumulator
            // load of the next 32 columns is in flight while the current ones are reduced.
            float2 acc0 = make_float2(0.f, 0.f), acc1 = acc0;          // (even, odd) column partial sums of the two outputs
#if GF_A_PROD_WG == 3
            #pragma unroll 1
            for (int c = 0; c < 4; c++) {                                // 80-register budget: one 32-column load at a time
                float v[32];
                tmem_ld32(t_d + 32 * c, v);
                #pragma unroll
                for (int q = 0; q < 32; q += 2) {
                    const float4 w = lds128(sbase + L::W2 + 16 * (16 * c + (q >> 1)));
                    const float2 h = make_float2(fmaxf(v[q], 0.f), fmaxf(v[q + 1], 0.f));
                    acc0 = ffma2(h, make_float2(w.x, w.y), acc0);
                    acc1 = ffma2(h, make_float2(w.z, w.w), acc1);
                }
            }
#else
            {
                uint32_t r[2][32];
                tmem_ld32_issue(t_d, r[0]);
                tmem_wait_ld32(r[0]);
                #pragma unroll
                for (int c = 0; c < 4; c++) {
                    uint32_t (&v)[32] = r[c & 1];
                    if (c < 3) tmem_ld32_issue(t_d + 32 * (c + 1), r[(c + 1) & 1]);
                    if (dbg) {
                        #pragma unroll
                        for (int q = 0; q < 32; q++) dbg[1 * 128 * 144 + 32 * c + q] = __uint_as_float(v[q]);
                    }
                    #pragma unroll
                    for (int q = 0; q < 32; q += 2) {
                        const float4 w = lds128(sbase + L::W2 + 16 * (16 * c + (q >> 1)));
                        const float2 h = make_float2(fmaxf(__uint_as_float(v[q]), 0.f), fmaxf(__uint_as_float(v[q + 1]), 0.f));
                        acc0 = ffma2(h, make_float2(w.x, w.y), acc0);
                        acc1 = ffma2(h, make_float2(w.z, w.w), acc1);
                    }
                    if (c < 3) tmem_wait_ld32(r[(c + 1) & 1]);
                }
            }
#endif
            const float s0 = acc0.x + acc0.y, s1 = acc1.x + acc1.y;
            if (dbg) { dbg[2 * 128 * 144 + 0] = s0; dbg[2 * 128 * 144 + 1] = s1; }
            if (i < M) a.io.amb_pos[i] = make_float2(tanhf(s0), tanhf(s1));
            TT_LSTAMP(0, stream, j, 6);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// ======================================================================================================================
// kernel B: features + 2-D gather -> sigma / colour
// ======================================================================================================================
template <bool DBG>
__global__ void __launch_bounds__(SP_THREADS, 1) k_tc_sigcol(const SpArgs a) {
    using L = SpSmem<WB2_TOTAL>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const uint32_t sbase = smem_u32(smem);
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    const uint32_t M = a.io.M_dev ? *a.io.M_dev : a.io.M_host;
    if (M == 0) return;
    const uint32_t cuts[5] = {0, WB2_SIG1, WB2_MRG, WB2_COL1, WB2_TOTAL};
    const uint32_t tmem_base = sp_setup<WB2_TOTAL>(smem, sbase, a, cuts, 4, 256);
    const uint32_t bias_ind = sbase + L::BIAS;
    const uint32_t bar_full = sbase + L::BAR + 8, bar_empty = sbase + L::BAR + 8 * (1 + SP_NSLOT);
    const uint32_t num_tiles = (M + 127) / 128;
    const uint32_t my_tiles = num_tiles > blockIdx.x ? (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp < 8) {
        // ------------------------------------------------ producers ------------------------------------------------
        const uint32_t half = tid >> 7, row = tid & 127;
        const bool contig_half = levels_unhashed(a.grid.lv, 8 * half, 8);
        // Per-row inputs of a tile (32 B of position features, the ambient coordinate, the ray's view direction) are staged ONE TILE AHEAD with
        // cp.async -- the features and the direction straight into the NEXT ring slot, which is therefore acquired one tile early -- and the ray
        // id TWO tiles ahead, so that the dependent pos4.w -> rays_d chain never sits on a producer's critical path.  (As register prefetches the
        // loads shared a scoreboard with unrelated instructions and the first use of the current tile's values waited for the next tile's DRAM
        // access; half 1, which also fetched the direction, had become the kernel's bottleneck: tc_timeline, profiles/r02_summary.md section 7.)
        const uint32_t ap_s = sbase + L::AP + 8 * tid, ray_s = sbase + L::RAY + 4 * row;
        auto tile_row = [&](uint32_t j) { return (blockIdx.x + j * gridDim.x) * 128 + row; };
        auto stage_ray = [&](uint32_t j) {          // half 1, sample-list form only
            const uint32_t i = tile_row(j);
            if (half == 1 && a.io.pos4 && j < my_tiles && i < M) cp_async4(ray_s + (j % 3) * 512, reinterpret_cast<const float*>(a.io.pos4 + i) + 3);
        };
        auto stage_inputs = [&](uint32_t j) {       // needs: slot of tile j acquired; ray id of tile j staged and complete
            const uint32_t i = tile_row(j), slot = j % SP_NSLOT;
            if (j < my_tiles && i < M) {
                const uint32_t F = sbase + L::F + slot * SP_TILE_BYTES;
                cp_async16(F + sw128(row, 2 * half), a.io.feat_hi + (size_t)i * 4 + 2 * half);
                cp_async16(F + sw128(row, 2 * half + 1), a.io.feat_hi + (size_t)i * 4 + 2 * half + 1);
                cp_async8(ap_s + (j & 1) * 2048, a.io.amb_pos + i);
                if (half == 1) {
                    const uint32_t d = sbase + L::DIR + 16 * (slot * 128 + row);
                    const float* src = nullptr;
                    if (a.io.pos4) src = a.io.rays_d + 3 * (size_t)lds32(ray_s + (j % 3) * 512);
                    else if (a.io.dirs) src = a.io.dirs + 3 * (size_t)i;
                    if (src) { cp_async4(d, src); cp_async4(d + 4, src + 1); cp_async4(d + 8, src + 2); }
                    else sts128f(d, make_float4(0.f, 0.f, 1.f, 0.f));
                }
            }
        };
        stage_ray(0);
        cp_async_commit();
        cp_async_wait_all();
        mbar_wait(bar_empty, 1);                      // slot 0 (free at start)
        stage_inputs(0);
        stage_ray(1);
        cp_async_commit();
        #pragma unroll 1
        for (uint32_t j = 0; j < my_tiles; j++) {
            const uint32_t slot = j % SP_NSLOT;
            const bool valid = tile_row(j) < M;
            cp_async_wait_all();                      // this tile's staged inputs (issued one tile ago) and the next tile's ray id have landed
            if (row == 0) TT_STAMP(1, 2 + half, j, 0);
            if (j + 1 < my_tiles) mbar_wait(bar_empty + 8 * ((j + 1) % SP_NSLOT), (((j + 1) / SP_NSLOT) & 1) ^ 1);   // acquire the NEXT slot
            if (row == 0) TT_STAMP(1, 2 + half, j, 1);
            stage_inputs(j + 1);
            stage_ray(j + 2);
            cp_async_commit();
            const uint32_t F = sbase + L::F + slot * SP_TILE_BYTES;
            float2 ap = make_float2(0.f, 0.f);
            if (valid) ap = lds64(ap_s + (j & 1) * 2048);
            else {                                    // rows past the end of the list: defined (zero) operands
                sts128(F + sw128(row, 2 * half), make_uint4(0, 0, 0, 0));
                sts128(F + sw128(row, 2 * half + 1), make_uint4(0, 0, 0, 0));
                if (half == 1) sts128f(sbase + L::DIR + 16 * (slot * 128 + row), make_float4(0.f, 0.f, 1.f, 0.f));
            }
            const float vx = (ap.x + 1.0f) * 0.5f, vy = (ap.y + 1.0f) * 0.5f;
            float2 f[8];
            if (contig_half) gather2_dyn8<true>(a.grid, 8 * half, vx, vy, f);
            else gather2_dyn8<false>(a.grid, 8 * half, vx, vy, f);
            #pragma unroll
            for (int u = 0; u < 2; u++)
                sts128(F + sw128(row, 4 + 2 * half + u), make_uint4(pack_h2(f[4 * u].x, f[4 * u].y), pack_h2(f[4 * u + 1].x, f[4 * u + 1].y),
                                                                    pack_h2(f[4 * u + 2].x, f[4 * u + 2].y), pack_h2(f[4 * u + 3].x, f[4 * u + 3].y)));
            fence_async_smem();
            mbar_arrive(bar_full + 8 * slot);
            if (row == 0) TT_STAMP(1, 2 + half, j, 2);
        }
    } else {
        // ------------------------------------------------ consumers ------------------------------------------------
        // warp-uniform copies of the warp index and the TMEM base: the tcgen05.mma operands derived from them then live in uniform registers.
        // Derived from threadIdx / a shared-memory load they were per-thread values, and every MMA was issued through an ELECT / R2UR
        // broadcast loop of 13 instructions (~75 cycles per MMA on the stream's critical path, longer than the MMA itself).
        const uint32_t warp_u = __shfl_sync(0xffffffffu, warp, 0), tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const uint32_t stream = (warp_u - 8) >> 2, row = tid & 127;
        const uint32_t t_d = tmem_u + (((warp_u & 3) * 32) << 16) + stream * SP_TM_STREAM;
        const uint32_t m_d = tmem_u + stream * SP_TM_STREAM;
        const uint32_t t_a = t_d + SP_TM_A, m_a = m_d + SP_TM_A;
        const uint32_t bar_mma = sbase + L::BAR + 8 * (1 + 2 * SP_NSLOT + stream);
        const uint32_t w_addr = sbase;
        // One elected lane of the stream's first warp waits on / arrives at the ring barriers and issues the MMAs.  The region must be guarded by
        // a warp-uniform test followed DIRECTLY by elect.sync (the CUTLASS idiom): only then does ptxas know that a single thread runs it and emit
        // the tcgen05.mma instructions back to back.  Guarded by `threadIdx == x` every MMA was wrapped in an ELECT / R2UR / branch loop of 11-13
        // instructions (~75 cycles per MMA on the stream's critical path -- longer than the 64 tensor-pipe cycles of the MMA itself).
        const bool lead_warp = (warp_u & 3) == 0;
        const bool sigma_only = !a.io.out4 && !a.io.rgbs;          // density query (uniform)
        // Software pipelining across a stream's tiles: sigma layer 0 of the NEXT tile (an SS MMA: needs only that tile's feature slot and accumulator
        // columns 0..127, which nobody reads once the last activation epilogue of the current tile has passed its barrier) is issued right behind the
        // current tile's last MMAs, which therefore write columns 128..143.  It runs while the threads finish the current tile (exp / sigmoid / store),
        // so the layer's issue -> commit -> wake-up latency (~800 of the stream's ~7,500 cycles per tile, tc_timeline) leaves the chain.
        const uint32_t bar_s0 = sbase + L::BAR + 8 * (3 + 2 * SP_NSLOT + stream);
        auto issue_sig0 = [&](uint32_t jj) {                          // called by the elected lane only
            const uint32_t sl = jj % SP_NSLOT, fa = sbase + L::F + sl * SP_TILE_BYTES;
            mbar_wait(bar_full + 8 * sl, (jj / SP_NSLOT) & 1);
            tc_fence_after();
            #pragma unroll
            for (int k = 0; k < 4; k++) mma_ss(m_d, smem_desc(fa + 32 * k), smem_desc(w_addr + WB2_SIG0 + 32 * k), idesc_f16(128), k);
            mma_commit(bar_s0);
        };
        uint32_t phase = 0, phase0 = 0;
        if (stream < my_tiles && lead_warp && elect_one_sync()) issue_sig0(stream);
        for (uint32_t j = stream; j < my_tiles; j += 2) {
            const uint32_t tile = blockIdx.x + j * gridDim.x, slot = j % SP_NSLOT;
            const uint32_t i = tile * 128 + row;
            const bool valid = i < M;
            float* dbg = (DBG && a.dbg && tile == 0) ? a.dbg + (size_t)row * 144 : nullptr;   // DBG = false: folds every dump away
            const uint32_t f_addr = sbase + L::F + slot * SP_TILE_BYTES;
            // ---- sigma layer 0: D = F[:, 0:64] @ Ws0^T (issued one tile ahead) -------------------------------------------
            TT_LSTAMP(1, stream, j, 0);
            TT_LSTAMP(1, stream, j, 1);
            stream_wait_mma(bar_s0, phase0);
            tc_fence_after();
            TT_LSTAMP(1, stream, j, 2);
            epilogue_relu_to_A_pipe<false>(t_d, t_a, 0u, dbg ? dbg + 3 * 128 * 144 : nullptr);
            TT_LSTAMP(1, stream, j, 3);
            tc_fence_before();
            bar_named(1 + stream, 128);
            // ---- sigma layer 1 -----------------------------------------------------------------------------------------
            if (lead_warp && elect_one_sync()) {
                tc_fence_after();
                #pragma unroll
                for (int k = 0; k < 8; k++)
                    mma_ts(m_d, m_a + 8 * k, smem_desc(w_addr + WB2_SIG1 + (k >> 2) * (128 * 128) + 32 * (k & 3)), idesc_f16(128), k);
                mma_commit(bar_mma);
            }
            // SH(dir) -> F[row][k 32..47]: the sigma-layer-0 MMA that read this slot has completed (waited above)
            {
                const float4 dir = lds128(sbase + L::DIR + 16 * (slot * 128 + row));   // visible: the leader's full-barrier wait + bar.sync
                float sh[16];
                sh4(dir.x, dir.y, dir.z, sh);
                uint32_t p[8];
                #pragma unroll
                for (int q = 0; q < 8; q++) p[q] = pack_h2(sh[2 * q], sh[2 * q + 1]);
                sts128(f_addr + sw128(row, 4), make_uint4(p[0], p[1], p[2], p[3]));
                sts128(f_addr + sw128(row, 5), make_uint4(p[4], p[5], p[6], p[7]));
                fence_async_smem();
            }
            stream_wait_mma(bar_mma, phase);
            tc_fence_after();
            TT_LSTAMP(1, stream, j, 4);
            epilogue_relu_to_A_pipe<false>(t_d, t_a, 0u, dbg ? dbg + 4 * 128 * 144 : nullptr);
            TT_LSTAMP(1, stream, j, 5);
            tc_fence_before();
            bar_named(1 + stream, 128);
            if (sigma_only) {
                // density query: only the sigma-logit row block of the merged layer (rows 128..143 of the image, N = 16); no colour net
                if (lead_warp && elect_one_sync()) {
                    tc_fence_after();
                    #pragma unroll
                    for (int k = 0; k < 8; k++)
                        mma_ts(m_d + 128, m_a + 8 * k, smem_desc(w_addr + WB2_MRG + (k >> 2) * (144 * 128) + 128 * 128 + 32 * (k & 3)), idesc_f16(16), k);
                    mma_commit(bar_mma);
                    mbar_arrive(bar_empty + 8 * slot);          // sigma layer 0 (waited above) was the slot's only reader in this mode
                    if (j + 2 < my_tiles) issue_sig0(j + 2);
                }
                stream_wait_mma(bar_mma, phase);
                tc_fence_after();
                float s4[4];
                tmem_ld4(t_d + 128, s4);
                if (valid) {
                    a.io.sigmas[i] = __expf(s4[0]);
                    if (a.io.ambient) { const float2 ap = a.io.amb_pos[i]; a.io.ambient[2 * (size_t)i] = ap.x; a.io.ambient[2 * (size_t)i + 1] = ap.y; }
                }
                continue;
            }
            // ---- merged sigma layer 2 x colour layer 0 (N = 144) + SH part (SS, K = 16, N = 128) --------------------------
            if (lead_warp && elect_one_sync()) {
                tc_fence_after();
                #pragma unroll
                for (int k = 0; k < 8; k++)
                    mma_ts(m_d, m_a + 8 * k, smem_desc(w_addr + WB2_MRG + (k >> 2) * (144 * 128) + 32 * (k & 3)), idesc_f16(144), k);
                mma_ss(m_d, smem_desc(f_addr + 64), smem_desc(w_addr + WB2_SH), idesc_f16(128), 1);
                mma_commit(bar_mma);
            }
            stream_wait_mma(bar_mma, phase);
            tc_fence_after();
            TT_LSTAMP(1, stream, j, 6);
            if (lead_warp && elect_one_sync()) mbar_arrive(bar_empty + 8 * slot);                // last reader of the feature tile is done
            float sg[4];
            tmem_ld4(t_d + 128, sg);
            if (dbg) dbg[5 * 128 * 144 + 128] = sg[0];
            if (a.bias) epilogue_relu_to_A_pipe<true>(t_d, t_a, bias_ind, dbg ? dbg + 5 * 128 * 144 : nullptr);
            else epilogue_relu_to_A_pipe<false>(t_d, t_a, 0u, dbg ? dbg + 5 * 128 * 144 : nullptr);
            tc_fence_before();
            bar_named(1 + stream, 128);
            // ---- colour layer 1 (N = 16; 3 real outputs) -> sigmoid ---------------------------------------------------------
            if (lead_warp && elect_one_sync()) {
                tc_fence_after();
                #pragma unroll
                for (int k = 0; k < 8; k++)
                    mma_ts(m_d + 128, m_a + 8 * k, smem_desc(w_addr + WB2_COL1 + (k >> 2) * (16 * 128) + 32 * (k & 3)), idesc_f16(16), k);
                mma_commit(bar_mma);
                if (j + 2 < my_tiles) issue_sig0(j + 2);
            }
            TT_LSTAMP(1, stream, j, 7);
            stream_wait_mma(bar_mma, phase);
            tc_fence_after();
            float c[4];
            tmem_ld4(t_d + 128, c);
            if (dbg) { dbg[6 * 128 * 144 + 0] = c[0]; dbg[6 * 128 * 144 + 1] = c[1]; dbg[6 * 128 * 144 + 2] = c[2]; }
            if (valid) {
                const float sigma = __expf(sg[0]);
                const float cr = __fdividef(1.0f, 1.0f + __expf(-c[0]));
                const float cg = __fdividef(1.0f, 1.0f + __expf(-c[1]));
                const float cb = __fdividef(1.0f, 1.0f + __expf(-c[2]));
                if (a.io.out4) a.io.out4[i] = make_float4(sigma, cr, cg, cb);
                if (a.io.sigmas) a.io.sigmas[i] = sigma;
                if (a.io.rgbs) { a.io.rgbs[3 * (size_t)i] = cr; a.io.rgbs[3 * (size_t)i + 1] = cg; a.io.rgbs[3 * (size_t)i + 2] = cb; }
                if (a.io.ambient) { const float2 ap = a.io.amb_pos[i]; a.io.ambient[2 * (size_t)i] = ap.x; a.io.ambient[2 * (size_t)i + 1] = ap.y; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
    if (a.io.stat_samples && blockIdx.x == 0 && tid == 0) atomicAdd(a.io.stat_samples, (unsigned long long)M);
}

// ======================================================================================================================
// gather-only probe: the field's grid gathers WITHOUT the MLPs (measurement aid for roofline.frac_of_gather_ceiling)
// ======================================================================================================================
// One thread per sample runs exactly the producers' gather code (gather3_dyn4 x 4 batches on the 3-D position grid, gather2_dyn8 x 2 on
// the 2-D ambient grid at the given ambient coordinate), folds the 64 features into one float2 and writes it: 1,536 algorithmic bytes
// gathered per sample, 8 B written.  With no tensor-core chain, no ring and full occupancy this is what the L1/L2 path delivers for THIS
// access pattern -- the ceiling the field kernels' gather rate is compared with.
__global__ void __launch_bounds__(256) k_gather_probe(GridDesc pos, GridDesc amb, float bound, float inv2b, const float* __restrict__ xyzs,
                                                      const float2* __restrict__ amb_pos, uint32_t M, float2* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    float ux = (xyzs[3 * (size_t)i] + bound) * inv2b, uy = (xyzs[3 * (size_t)i + 1] + bound) * inv2b, uz = (xyzs[3 * (size_t)i + 2] + bound) * inv2b;
    if (ux < 0 || ux > 1 || uy < 0 || uy > 1 || uz < 0 || uz > 1) { ux = 0.5f; uy = 0.5f; uz = 0.5f; }     // as the producers: corner indices stay in range
    float2 acc = make_float2(0.f, 0.f);
    #pragma unroll 1
    for (int u = 0; u < 4; u++) {
        bool flat = true;
        #pragma unroll
        for (int q = 0; q < 4; q++) flat = flat && pos.lv.sz[4 * u + q] == 0 && pos.lv.hashed[4 * u + q] == 0;
        float2 f[4];
        gather3_unit(pos, u, flat, levels_unhashed(pos.lv, 4 * u, 4), ux, uy, uz, f);
        #pragma unroll
        for (int q = 0; q < 4; q++) { acc.x += f[q].x; acc.y += f[q].y; }
    }
    const float2 ap = amb_pos[i];
    const float vx = (ap.x + 1.0f) * 0.5f, vy = (ap.y + 1.0f) * 0.5f;
    #pragma unroll 1
    for (int h = 0; h < 2; h++) {
        float2 f[8];
        if (levels_unhashed(amb.lv, 8 * h, 8)) gather2_dyn8<true>(amb, 8 * h, vx, vy, f);
        else gather2_dyn8<false>(amb, 8 * h, vx, vy, f);
        #pragma unroll
        for (int q = 0; q < 8; q++) { acc.x += f[q].x; acc.y += f[q].y; }
    }
    out[i] = acc;
}

int gather_probe_launch(const GfModel* model, const float* xyzs, const float* amb_pos, uint32_t M, float* out, cudaStream_t st) {
    k_gather_probe<<<(M + 255) / 256, 256, 0, st>>>(model->dev.pos, model->dev.amb, model->dev.bound, 0.5f / model->dev.bound, xyzs,
                                                  reinterpret_cast<const float2*>(amb_pos), M, reinterpret_cast<float2*>(out));
    return check_launch("gather_probe");
}

// ======================================================================================================================
// host
// ======================================================================================================================
// Builds the fp16 weight images of both kernels; called ONCE from gf_model_create (nothing is packed lazily on the frame path, so
// gf_render_frame never allocates or synchronises and can be captured into a CUDA graph).  Models outside the tcgen05 envelope
// (hidden_dim / geo_feat_dim != 128) simply have no image: precision = 1 then returns GF_ERR_UNSUPPORTED.
int field_tc_pack(GfModel* m, cudaStream_t st) {
    const GfModelDesc& d = m->desc;
    if (d.hidden_dim != 128 || d.geo_feat_dim != 128) return GF_OK;
    uint8_t* img = nullptr;
    if (cudaMalloc(&img, WA_TOTAL + WB2_TOTAL) != cudaSuccess) { cudaGetLastError(); set_error("tc pack: cudaMalloc failed"); return GF_ERR_CUDA; }
    cudaMemsetAsync(img, 0, WA_TOTAL + WB2_TOTAL, st);
    TcPackSrc2 s;
    s.a0 = d.ambient_w0; s.a1 = d.ambient_w1; s.s0 = d.sigma_w0; s.s1 = d.sigma_w1; s.s2 = d.sigma_w2; s.c0 = d.color_w0; s.c1 = d.color_w1;
    s.cond = (int)d.cond_dim; s.ind = (int)d.ind_dim; s.G = (int)d.geo_feat_dim;
    k_tc_pack_split<<<(144 * 128 + 255) / 256, 256, 0, st>>>(s, img, img + WA_TOTAL);
    int rc = check_launch("tc split pack");
    if (rc) { cudaFree(img); return rc; }
    if (cudaFuncSetAttribute(k_tc_amb<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SpSmem<WA_TOTAL>::BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(k_tc_amb<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SpSmem<WA_TOTAL>::BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(k_tc_sigcol<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SpSmem<WB2_TOTAL>::BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(k_tc_sigcol<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SpSmem<WB2_TOTAL>::BYTES) != cudaSuccess ||
        cudaMemcpyAsync(m->w_amb2_host, m->w + m->dev.a_w2, sizeof(float) * 256, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(img);
        set_error("tc split pack: setup failed");
        return GF_ERR_CUDA;
    }
    m->tc2_blob = img;
    return GF_OK;
}

// bytes of caller-owned scratch one stand-alone field evaluation of M samples needs (fp16 position features + ambient coordinates)
size_t field_tc_scratch_bytes(uint32_t M) { return (((size_t)M * 64 + 255) & ~size_t(255)) + (size_t)M * 8 + 256; }

int field_tc_kernel_count() { return 2; }

int field_tc_launch(const GfModel* model, const FieldTcIO& io_in, cudaStream_t st) {
    if (!model->tc2_blob) {
        set_error("precision=1 (tcgen05) supports hidden_dim == 128 and geo_feat_dim == 128 only; use precision=0");
        return GF_ERR_UNSUPPORTED;
    }
    const FieldTcIO& io = io_in;
    if (!io.feat_hi || !io.amb_pos) { set_error("field_tc: the feature / ambient-coordinate scratch is missing"); return GF_ERR_INVALID; }
    uint32_t grid = (uint32_t)model->num_sms;
    if (!io.M_dev) {
        const uint32_t tiles = (io.M_host + 127) / 128;
        if (tiles < grid) grid = tiles ? tiles : 1;
    }
    SpArgs a;
    memset(&a, 0, sizeof(a));
    a.bound = model->dev.bound; a.inv2b = 0.5f / model->dev.bound;
    a.io = io;
    a.dbg = model->tc_dbg;
    a.grid = model->dev.pos;
    a.wimg = (const uint8_t*)model->tc2_blob;
    a.bias = io.bias_amb;
    memcpy(a.w_amb2, model->w_amb2_host, sizeof(a.w_amb2));
    if (a.dbg && !GF_TC_TIMING) k_tc_amb<true><<<grid, SPA_THREADS, SpSmem<WA_TOTAL>::BYTES, st>>>(a);
    else k_tc_amb<false><<<grid, SPA_THREADS, SpSmem<WA_TOTAL>::BYTES, st>>>(a);
    const int rc = check_launch("field_tc_split(amb)");
    if (rc) return rc;
    a.grid = model->dev.amb;
    a.wimg = (const uint8_t*)model->tc2_blob + WA_TOTAL;
    a.bias = model->dev.ind ? model->dev.w + model->dev.c_bind : nullptr;
    if (a.dbg && !GF_TC_TIMING) k_tc_sigcol<true><<<grid, SP_THREADS, SpSmem<WB2_TOTAL>::BYTES, st>>>(a);
    else k_tc_sigcol<false><<<grid, SP_THREADS, SpSmem<WB2_TOTAL>::BYTES, st>>>(a);
    return check_launch("field_tc_split(sigcol)");
}

}  // namespace gf

extern "C" {
// Diagnostics: make the next precision-1 launches dump the fp32 accumulators of tile 0 after each MMA stage into dbg
// (device float[9*128*144]); pass NULL to switch it off.  Used by tests/test_parity_gpu.py.
GF_API int gf_tc_debug(GfModel* model, float* dbg) {
    if (!model) return GF_ERR_INVALID;
    model->tc_dbg = dbg;
    return GF_OK;
}
}
