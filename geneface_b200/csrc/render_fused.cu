// libgfrender: fused frame renderer (coarse drop-in boundary).
//
// Replaces the eval branch of NeRFRenderer.render() (modules/radnerfs/renderer.py:263-367) and
// RADNeRFTorso.render() (modules/radnerfs/radnerf_torso.py:86-198).  The reference drives up
// to max_steps iterations of {march_rays, ~25 torch kernels + 8 cuBLAS GEMMs, composite_rays,
// boolean-mask compaction} from the host with two device syncs per iteration.  Here a frame is
// a FIXED sequence of launches with no host sync:
//
//   k_frame_setup      per-frame bias folds (cond -> ambient layer-0 bias, pose -> torso biases)
//   k_rays_init        ray generation (utils.py:282-363) or load, slab test (K1), state init
//   R rounds of        k_march_chunk     each live ray emits its next <=chunk occupied samples
//                                        into a DENSE sample list (warp-aggregated allocation)
//                      k_field_*         field evaluation over the dense list (fp32 SIMT here,
//                                        fp16 tcgen05 in field_tc_split.cu)
//                      k_composite_chunk per-ray front-to-back compositing, termination, histogram
//   k_schedule         replays the reference's host loop n_step = clamp(N // n_alive, 1, 8) from the
//                      termination histogram -> S_total in [max_steps, max_steps+7]
//   1 extra round      budget = S_total - max_steps (device-side; no-op when 0)
//   k_torso_*          torso occupancy mask + deformation/canonical field (radnerf_torso.py:51-84,155-188)
//   k_finish           background/torso mix, clamp, depth normalisation, RGB8 (renderer.py:354-362)
//
// Why this reproduces the reference bit-for-bit in its integer outputs: a ray's sample sequence does
// not depend on how the host loop batches it (march resumes at rays_t); the only global coupling is
// the cap `step < max_steps` with step += n_step, i.e. every live ray is offered S_total slots, and
// n_alive at iteration i is the number of rays whose termination slot exceeds the slots offered so
// far -- which the histogram gives exactly (SURVEY.md section 7 "Termination semantics").
#include <cstdlib>
#include <cstring>
#include <vector>

#include "gf_dense.cuh"
#include "gf_field.cuh"
#include "gf_model.cuh"

namespace gf {

// ======================================================================================
// model setup kernels
// ======================================================================================
// one warp: lane l < 16 computes level l, all 32 lanes take part in the scan of the padded image's level sizes
__global__ void k_level_geometry(const int* __restrict__ offsets, float S, uint32_t H, uint32_t D, uint32_t gridtype, GridLevels* out,
                                 int* __restrict__ bad) {
    const int l = threadIdx.x;
    uint32_t entries = 0;          // entries of level l in the padded image
    if (l < 16) {
        // gridencoder.cu:137-139 (device exp2f on purpose: bit-identical scale to the reference kernel)
        const float scale = __fmaf_rn(exp2f(__fmul_rn((float)l, S)), (float)H, -1.0f);
        const uint32_t res = (uint32_t)ceilf(scale) + 1;
        const uint32_t hs = (uint32_t)(offsets[l + 1] - offsets[l]);
        out->scale[l] = scale;
        out->res[l] = res;
        out->hsize[l] = hs;
        out->offset[l] = (uint32_t)offsets[l];
        // replay of the stride loop of get_grid_index (gridencoder.cu:68-75, align_corners = false), uint32 wrap-around included
        const uint32_t R = res + 1;
        uint32_t stride = 1, sy = 0, sz = 0;
        stride *= R;                                              // d = 0 is always taken (1 <= hashmap_size)
        if (stride <= hs) { sy = stride; stride *= R; }
        if (D == 3 && stride <= hs) { sz = stride; stride *= R; }
        out->sy[l] = sy;
        out->sz[l] = sz;
        const bool hashed = gridtype == 0 && stride > hs;
        out->hashed[l] = hashed ? 1u : 0u;
        const bool pow2 = hs && (hs & (hs - 1)) == 0;
        out->mask[l] = pow2 ? hs - 1 : 0xFFFFFFFFu;
        // `index % hsize` is only replaced by the mask when it is provably the same: power-of-two level, or a dense level
        // whose largest reachable index (pos_grid <= res per axis) stays below hsize.
        const unsigned long long maxidx = (unsigned long long)res * (1ull + sy + sz);
        const bool nowrap = !hashed && maxidx < hs;
        if (!pow2 && !nowrap) *bad = 1;
        const uint32_t pad = (hashed || nowrap) ? 0u : 1u + sy + sz;
        out->pad[l] = pad;
        entries = hs + pad;
    }
    uint32_t incl = entries;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (l >= o) incl += v;
    }
    if (l < 16) out->img_offset[l] = incl - entries;
}

// padded image of a grid table (GridLevels::pad): dst[img_offset[l] + k] = src[offset[l] + k % hsize[l]], k < hsize[l] + pad[l]
__global__ void k_grid_image(const float2* __restrict__ src, const GridLevels lv, float2* __restrict__ dst) {
    const uint32_t l = blockIdx.y, hs = lv.hsize[l], n = hs + lv.pad[l];
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x)
        dst[lv.img_offset[l] + k] = src[lv.offset[l] + k % hs];
}

// dst[k][n] = src[n][k0 + k]   (src row-major [N][ldsrc]); dst row stride ldd
__global__ void k_transpose_pack(const float* __restrict__ src, int ldsrc, int k0, int K, int N, float* __restrict__ dst, int ldd) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * N) return;
    const int k = i / N, n = i - k * N;
    dst[(size_t)k * ldd + n] = src[(size_t)n * ldsrc + k0 + k];
}

// out[n] = sum_k W[n][k0+k] * v[k]   (tiny GEMV: bias folds)
__global__ void k_gemv_fold(const float* __restrict__ W, int ldw, int k0, int K, int N, const float* __restrict__ v, float* __restrict__ out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float acc = 0.f;
    for (int k = 0; k < K; k++) acc = fmaf(W[(size_t)n * ldw + k0 + k], v[k], acc);
    out[n] = acc;
}

// ======================================================================================
// per-frame setup: cond bias fold + torso pose bias folds
// ======================================================================================
struct FrameSetup {
    const float* cond_feat;   // [cond]
    float torso_pose[6];
    int has_torso;
    const float* dyn;         // GfFrame.dyn (device float[22]) or null
};

// block 0: ambient bias[h] = sum_c W_a0[h][32 + c] * cond[c]     (radnerf.py:80,84 folded)
// block 1: torso: enc_pose = freq(pose6, 4) (54) ++ code (8) -> deform bias [64], canon bias [32]
__global__ void k_frame_setup(ModelDev m, FrameSetup fs, float* __restrict__ bias_amb, float* __restrict__ bias_deform,
                              float* __restrict__ bias_canon) {
    const int t = threadIdx.x;
    if (blockIdx.x == 0) {
        if (t < m.H) {
            const float* W = m.w + m.a_wc;   // [cond][H] transposed
            float acc = 0.f;
            for (int c = 0; c < m.cond; c++) acc = fmaf(__ldg(W + (size_t)c * m.H + t), __ldg(fs.cond_feat + c), acc);
            bias_amb[t] = acc;
        }
        return;
    }
    if (!fs.has_torso) return;
    __shared__ float cst[64];   // [enc_pose(54) | code(<=8)]
    if (t < 54) {
        // freqencoder.cu:30-58 with D=6, deg=4
        const int c = t;
        float v;
        const int d = c % 6;
        const float pd = fs.dyn ? __ldg(fs.dyn + 16 + d) : fs.torso_pose[d];
        if (c < 6) v = pd;
        else {
            const int col = c / 6 - 1, freq = col / 2;
            const float phase = (float)(col % 2) * (3.141592653589793f / 2);
            v = __sinf(__fadd_rn(scalbnf(pd, freq), phase));
        }
        cst[c] = v;
    } else if (t < 54 + m.t_ind) cst[t] = m.t_code ? __ldg(m.t_code + (t - 54)) : 0.f;
    __syncthreads();
    const int KC = 54 + m.t_ind;
    if (t < 64) {   // deform layer 0: columns [42, 42+KC) of W [64][104]
        const float* W = m.w + m.td_wc;   // [KC][64]
        float acc = 0.f;
        for (int k = 0; k < KC; k++) acc = fmaf(__ldg(W + k * 64 + t), cst[k], acc);
        bias_deform[t] = acc;
    } else if (t < 96) {   // canonical layer 0: columns [32+42, 32+42+KC) of W [32][136]
        const int n = t - 64;
        const float* W = m.w + m.tc_wc;   // [KC][32]
        float acc = 0.f;
        for (int k = 0; k < KC; k++) acc = fmaf(__ldg(W + k * 32 + n), cst[k], acc);
        bias_canon[n] = acc;
    }
}

// ======================================================================================
// ray generation + slab test + state init
// ======================================================================================
// Tile-friendly ray order is NOT applied here: ray n is pixel (y = n / W, x = n % W), the
// reference's order (utils.py:301-303).
// utils.py:300-352: i = x + 0.5, j = y + 0.5; dir = normalize([(i-cx)/fx, (j-cy)/fy, 1]) @ R^T; origin = translation.  P = c2w rows 0..2.
__device__ __forceinline__ void pixel_ray(const float (&P)[12], float fx, float fy, float cx, float cy, uint32_t px, uint32_t py,
                                          float& ox, float& oy, float& oz, float& dx, float& dy, float& dz, float& i, float& j) {
    i = __fadd_rn((float)px, 0.5f); j = __fadd_rn((float)py, 0.5f);
    const float xs = __fdiv_rn(__fsub_rn(i, cx), fx);
    const float ys = __fdiv_rn(__fsub_rn(j, cy), fy);
    const float nrm = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(xs, xs), __fmul_rn(ys, ys)), 1.0f));
    const float ux = __fdiv_rn(xs, nrm), uy = __fdiv_rn(ys, nrm), uz = __fdiv_rn(1.0f, nrm);
    dx = P[0] * ux + P[1] * uy + P[2] * uz;
    dy = P[4] * ux + P[5] * uy + P[6] * uz;
    dz = P[8] * ux + P[9] * uy + P[10] * uz;
    ox = P[3]; oy = P[7]; oz = P[11];
}

// get_rays as a fine-grained op (utils.py:282-363): rays for a list of flat pixel indices (inds == null: all H*W pixels in order) of B poses
__global__ void k_get_rays(const float* __restrict__ poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t W,
                           const int64_t* __restrict__ inds, uint32_t N, float* __restrict__ rays_o, float* __restrict__ rays_d,
                           float* __restrict__ out_i, float* __restrict__ out_j) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * N) return;
    const uint32_t b = t / N, n = t - b * N;
    const uint32_t idx = inds ? (uint32_t)inds[n] : n;
    float P[12];
    #pragma unroll
    for (int k = 0; k < 12; k++) P[k] = __ldg(poses + 16 * (size_t)b + k);
    float ox, oy, oz, dx, dy, dz, i, j;
    pixel_ray(P, fx, fy, cx, cy, idx % W, idx / W, ox, oy, oz, dx, dy, dz, i, j);
    rays_o[3 * (size_t)t] = ox; rays_o[3 * (size_t)t + 1] = oy; rays_o[3 * (size_t)t + 2] = oz;
    rays_d[3 * (size_t)t] = dx; rays_d[3 * (size_t)t + 1] = dy; rays_d[3 * (size_t)t + 2] = dz;
    if (b == 0) {
        if (out_i) out_i[n] = i;
        if (out_j) out_j[n] = j;
    }
}

__global__ void k_rays_init(RayInit ri, RayState st) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= ri.N) return;
    float ox, oy, oz, dx, dy, dz;
    if (ri.rays_o) {
        ox = ri.rays_o[3 * (size_t)n]; oy = ri.rays_o[3 * (size_t)n + 1]; oz = ri.rays_o[3 * (size_t)n + 2];
        dx = ri.rays_d[3 * (size_t)n]; dy = ri.rays_d[3 * (size_t)n + 1]; dz = ri.rays_d[3 * (size_t)n + 2];
    } else {
        float P[12], fx = ri.fx, fy = ri.fy, cx = ri.cx, cy = ri.cy;
        if (ri.dyn) {           // per-frame scalars from device memory (CUDA-graph replay): 16 broadcast loads
            #pragma unroll
            for (int k = 0; k < 12; k++) P[k] = __ldg(ri.dyn + k);
            fx = __ldg(ri.dyn + 12); fy = __ldg(ri.dyn + 13); cx = __ldg(ri.dyn + 14); cy = __ldg(ri.dyn + 15);
        } else {
            #pragma unroll
            for (int k = 0; k < 12; k++) P[k] = ri.pose[k];
        }
        const uint32_t py = n / ri.W, px = n - py * ri.W;
        float i, j;
        pixel_ray(P, fx, fy, cx, cy, px, py, ox, oy, oz, dx, dy, dz, i, j);
    }
    st.rays_o[3 * (size_t)n] = ox; st.rays_o[3 * (size_t)n + 1] = oy; st.rays_o[3 * (size_t)n + 2] = oz;
    st.rays_d[3 * (size_t)n] = dx; st.rays_d[3 * (size_t)n + 1] = dy; st.rays_d[3 * (size_t)n + 2] = dz;
    const Ray r = make_ray(ox, oy, oz, dx, dy, dz);
    float near, far;
    near_far_aabb(r, ri.aabb, ri.min_near, near, far);
    st.nears[n] = near;
    st.fars[n] = far;
    st.t[n] = near;          // rays_t = nears.clone()  (renderer.py:324)
    st.alive[n] = 1;         // rays_alive = arange(N)  (renderer.py:323)
    st.wsum[n] = 0.f; st.depth[n] = 0.f;
    st.img[3 * (size_t)n] = 0.f; st.img[3 * (size_t)n + 1] = 0.f; st.img[3 * (size_t)n + 2] = 0.f;
    st.nsamp[n] = 0;
    st.term[n] = 0;
    st.seg_cnt[n] = 0;
}

__global__ void k_zero_u32(uint32_t* p, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0;
}

// ======================================================================================
// march one chunk: count, warp-aggregated allocate, write
// ======================================================================================
// ctl[CTL_TOTAL]   running sample total of the current round (allocation cursor)
// budget: pass A = min(chunk, max_steps - slots_before); pass B = ctl[CTL_EXTRA] (device value)
__global__ void __launch_bounds__(128) k_march_chunk(MarchArgs a, RayState st, SampleBuf sb, uint32_t* __restrict__ ctl) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t budget = a.budget_from_ctl ? ctl[CTL_EXTRA] : a.budget;
    if (budget == 0) return;
    const bool active = n < a.N && st.alive[n];
    uint32_t count = 0;
    MarchConst m = make_march_const(a.bound, a.dt_gamma, a.max_steps, a.C, a.H, a.grid);
    Ray r;
    float far = 0.f, t0 = 0.f;
    if (active) {
        r = make_ray(st.rays_o[3 * (size_t)n], st.rays_o[3 * (size_t)n + 1], st.rays_o[3 * (size_t)n + 2],
                     st.rays_d[3 * (size_t)n], st.rays_d[3 * (size_t)n + 1], st.rays_d[3 * (size_t)n + 2]);
        far = st.fars[n];
        t0 = st.t[n];
        // (raymarching.cu:873: perturbation noise is zero in eval -> t unchanged)
        float t = t0;
        Probe p;
        while (count < budget && march_next(m, r, far, t, p)) { count++; t = __fadd_rn(t, p.dt); }
    }
    // warp-aggregated allocation of `count` slots.  Layout inside the warp's block: SLOT-MAJOR across the warp's 32 rays
    // (slot k of every ray that has one, then slot k+1, ...), dense.  The 32 rays of a warp are 32 neighbouring pixels of an
    // image row, so 32 consecutive samples of the list lie side by side in space: the field kernels' grid gathers of one
    // warp then share cache lines instead of touching 32 different ones (consecutive samples of ONE ray are a whole step apart).
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1u;
    uint32_t warp_total = count, warp_max = count;
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        warp_total += __shfl_xor_sync(0xffffffffu, warp_total, o);
        warp_max = max(warp_max, __shfl_xor_sync(0xffffffffu, warp_max, o));
    }
    uint32_t base = 0;
    if (lane == 0 && warp_total) base = atomicAdd(ctl + CTL_TOTAL, warp_total);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (active) { st.seg_off[n] = base; st.seg_cnt[n] = count; }
    float t = t0;
    uint32_t off = base;
    for (uint32_t k = 0; k < warp_max; k++) {
        const uint32_t have = __ballot_sync(0xffffffffu, k < count);
        if (k < count) {
            Probe p;
            march_next(m, r, far, t, p);               // succeeds: the counting pass took the same steps
            t = __fadd_rn(t, p.dt);
            const uint32_t idx = off + __popc(have & lt);
            sb.pos4[idx] = make_float4(p.x, p.y, p.z, __int_as_float((int)n));
            sb.dl[idx] = make_float2(p.dt, t);
            if (sb.occ_index) sb.occ_index[idx] = p.index;
        }
        off += __popc(have);
    }
}

// ======================================================================================
// composite one chunk (K12 semantics, raymarching.cu:942-1029) + termination bookkeeping
// ======================================================================================
__global__ void __launch_bounds__(128) k_composite_chunk(CompArgs a, RayState st, SampleBuf sb, uint32_t* __restrict__ ctl) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t budget = a.budget_from_ctl ? ctl[CTL_EXTRA] : a.budget;
    if (budget == 0) return;
    const bool active = n < a.N && st.alive[n];
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1u;
    const uint32_t cnt = active ? st.seg_cnt[n] : 0;
    uint32_t off = active ? st.seg_off[n] : 0;                    // the warp's block (same value in every active lane)
    uint32_t warp_max = cnt;
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) warp_max = max(warp_max, __shfl_xor_sync(0xffffffffu, warp_max, o));
    float weight_sum = 0.f, d = 0.f, r = 0.f, g = 0.f, b = 0.f, t = 0.f;
    if (active) {
        weight_sum = st.wsum[n]; d = st.depth[n];
        r = st.img[3 * (size_t)n]; g = st.img[3 * (size_t)n + 1]; b = st.img[3 * (size_t)n + 2];
        t = st.t[n];
    }
    uint32_t step = 0;
    bool terminated = false;
    // slot-major walk of the warp's block (layout of k_march_chunk)
    for (uint32_t k = 0; k < warp_max; k++) {
        const uint32_t have = __ballot_sync(0xffffffffu, k < cnt);
        if (k < cnt && !terminated) {
            const uint32_t idx = off + __popc(have & lt);
            const float4 o = sb.out4[idx];          // sigma, r, g, b
            const float2 dl = sb.dl[idx];
            const float alpha = 1.0f - __expf(-o.x * dl.x);
            const float T = 1 - weight_sum;
            const float weight = alpha * T;
            weight_sum += weight;
            t = dl.y;
            d = fmaf(weight, t, d);
            r = fmaf(weight, o.y, r);
            g = fmaf(weight, o.z, g);
            b = fmaf(weight, o.w, b);
            if (T < a.T_thresh) terminated = true; else step++;
        }
        off += __popc(have);
    }
    // slots consumed this round: terminated at sample (step+1); ran dry at slot cnt+1 (delta == 0 terminator)
    const bool dead = active && (terminated || cnt < budget);
    const uint32_t k = a.slots_before + (terminated ? step + 1 : cnt + 1);       // termination slot (1-based)
    // termination histogram, warp-aggregated: lanes with the same slot elect one lane that adds their count.  (In the May configuration
    // the 59 % of rays that miss the occupied region all die at slot 1: 155 K same-address atomics made this kernel 4x slower than the
    // 5x larger benchmark round.)
    const bool counts = dead && !a.budget_from_ctl && k <= a.max_steps;
    const uint32_t peers = __match_any_sync(0xffffffffu, counts ? k : 0xffffffffu);
    if (counts && lane == (uint32_t)(__ffs(peers) - 1)) atomicAdd(ctl + CTL_HIST + k, (uint32_t)__popc(peers));
    if (!active) return;
    const uint32_t composited = terminated ? step + 1 : cnt;
    st.nsamp[n] += (int)composited;
    st.wsum[n] = weight_sum; st.depth[n] = d;
    st.img[3 * (size_t)n] = r; st.img[3 * (size_t)n + 1] = g; st.img[3 * (size_t)n + 2] = b;
    if (dead) {
        st.alive[n] = 0;
        st.term[n] = (int)k;
    } else {
        st.t[n] = t;
    }
}

// ======================================================================================
// replay of the host loop (renderer.py:326-351)
// ======================================================================================
__global__ void k_schedule(uint32_t N, uint32_t max_steps, uint32_t* __restrict__ ctl) {
    // the histogram is staged into shared memory by the whole block first: the replay itself is a serial dependence chain and used to pay
    // one global-memory round trip per slot (36 us at max_steps = 128)
    __shared__ uint32_t hist[RENDER_MAX_STEPS + 1];
    for (uint32_t k = threadIdx.x; k <= max_steps; k += blockDim.x) hist[k] = k ? ctl[CTL_HIST + k] : 0;
    __syncthreads();
    if (threadIdx.x) return;
    uint32_t alive = N, step = 0;
    while (step < max_steps) {
        if (alive == 0) break;
        uint32_t n_step = N / alive;
        n_step = n_step > 8 ? 8 : n_step;
        n_step = n_step < 1 ? 1 : n_step;
        uint32_t died = 0;
        for (uint32_t k = step + 1; k <= step + n_step && k <= max_steps; k++) died += hist[k];
        alive -= died;
        step += n_step;
    }
    // alive == 0 before reaching max_steps: nobody is left to receive extra slots
    ctl[CTL_STOTAL] = step;
    ctl[CTL_EXTRA] = step > max_steps ? step - max_steps : 0;
    ctl[CTL_TOTAL] = 0;   // allocation cursor for the extra round
}

// ======================================================================================
// fp32 reference-arithmetic field over a dense sample list
// ======================================================================================
struct FieldIO {
    // input A: packed samples + ray table
    const float4* pos4;
    const float* rays_d;
    // input B: reference layout (march_rays outputs)
    const float* xyzs;
    const float* dirs;
    const uint32_t* M_dev;   // sample count on device (or null -> M_host)
    uint32_t M_host;
    // outputs (any may be null)
    float4* out4;
    float* sigmas;
    float* rgbs;
    float* ambient;          // [M,2]
    const float* bias_amb;   // [H]
    unsigned long long* stat_samples;
};

// smem: F [64][128] | P [144][128] | Q [144][128] | wstage [2][16][128] | misc
constexpr int FP32_SMEM_FLOATS = 64 * 128 + 144 * 128 + 144 * 128 + 2 * 16 * 128 + 16 * 128;

__global__ void __launch_bounds__(DENSE_THREADS, 1) k_field_fp32(ModelDev m, FieldIO io) {
    extern __shared__ __align__(16) float smem[];
    float* F = smem;                        // features: rows 0..31 pos grid, 32..63 ambient grid
    float* P = F + 64 * 128;
    float* Q = P + 144 * 128;
    float* wstage = Q + 144 * 128;
    float* misc = wstage + 2 * 16 * 128;    // [0..2] xyz unit coords, [3..5] dir, [6..7] ambient pos, [8] sigma, [9..11] rgb, [12..15] scratch
    const uint32_t M = io.M_dev ? *io.M_dev : io.M_host;
    const int tid = threadIdx.x;
    const int H = m.H, G = m.G;
    const bool sigma_only = !io.out4 && !io.rgbs;      // density query (grid maintenance): skip the geometry features and the colour net

    for (uint32_t tile = blockIdx.x; (uint64_t)tile * TILE_S < M; tile += gridDim.x) {
        const uint32_t base = tile * TILE_S;
        // ---- load samples ----------------------------------------------------------------
        if (tid < TILE_S) {
            const uint32_t i = base + tid;
            float x = 0.f, y = 0.f, z = 0.f, dx = 0.f, dy = 0.f, dz = 0.f;
            if (i < M) {
                if (io.pos4) {
                    const float4 p = io.pos4[i];
                    x = p.x; y = p.y; z = p.z;
                    const int ray = __float_as_int(p.w);
                    dx = __ldg(io.rays_d + 3 * (size_t)ray); dy = __ldg(io.rays_d + 3 * (size_t)ray + 1); dz = __ldg(io.rays_d + 3 * (size_t)ray + 2);
                } else {
                    x = io.xyzs[3 * (size_t)i]; y = io.xyzs[3 * (size_t)i + 1]; z = io.xyzs[3 * (size_t)i + 2];
                    if (io.dirs) { dx = io.dirs[3 * (size_t)i]; dy = io.dirs[3 * (size_t)i + 1]; dz = io.dirs[3 * (size_t)i + 2]; }
                }
            }
            misc[0 * 128 + tid] = to_unit(x, m.bound);
            misc[1 * 128 + tid] = to_unit(y, m.bound);
            misc[2 * 128 + tid] = to_unit(z, m.bound);
            misc[3 * 128 + tid] = dx; misc[4 * 128 + tid] = dy; misc[5 * 128 + tid] = dz;
        }
        __syncthreads();
        // ---- 3D position grid: 128 samples x 16 levels over 256 threads ---------------------
        {
            const int s = tid & 127;
            const float ux = misc[s], uy = misc[128 + s], uz = misc[256 + s];
            #pragma unroll 2
            for (int j = 0; j < 8; j++) {
                const int level = (tid >> 7) + 2 * j;
                const float2 f = grid3_sample(m.pos, level, ux, uy, uz);
                F[(2 * level) * 128 + s] = f.x;
                F[(2 * level + 1) * 128 + s] = f.y;
            }
        }
        __syncthreads();
        // ---- ambient MLP: 32(+cond via bias) -> H -> H -> 2, tanh ----------------------------
        dense_tile(F, 32, m.w + m.a_wt0, H, H, P, io.bias_amb, true, wstage);
        dense_tile(P, H, m.w + m.a_wt1, H, H, Q, nullptr, true, wstage);
        dense_small(Q, H, m.w + m.a_w2, 2, misc + 6 * 128, misc + 12 * 128);
        if (tid < 2 * TILE_S) {
            const int s = tid & 127, c = tid >> 7;
            const float a = tanhf(misc[(6 + c) * 128 + s]);
            misc[(6 + c) * 128 + s] = a;
        }
        __syncthreads();
        // ---- 2D ambient grid ------------------------------------------------------------------
        {
            const int s = tid & 127;
            const float ax = to_unit(misc[6 * 128 + s], 1.0f), ay = to_unit(misc[7 * 128 + s], 1.0f);
            #pragma unroll 2
            for (int j = 0; j < 8; j++) {
                const int level = (tid >> 7) + 2 * j;
                const float2 f = grid2_sample(m.amb, level, ax, ay);
                F[(32 + 2 * level) * 128 + s] = f.x;
                F[(32 + 2 * level + 1) * 128 + s] = f.y;
            }
        }
        __syncthreads();
        // ---- sigma MLP: 64 -> H -> H -> 1 + G ---------------------------------------------------
        dense_tile(F, 64, m.w + m.s_wt0, H, H, P, nullptr, true, wstage);
        dense_tile(P, H, m.w + m.s_wt1, H, H, Q, nullptr, true, wstage);
        dense_small(Q, H, m.w + m.s_w2s, 1, misc + 8 * 128, misc + 12 * 128);
        if (sigma_only) {
            if (tid < TILE_S && base + tid < M) {
                io.sigmas[base + tid] = expf(misc[8 * 128 + tid]);
                if (io.ambient) { io.ambient[2 * (size_t)(base + tid)] = misc[6 * 128 + tid]; io.ambient[2 * (size_t)(base + tid) + 1] = misc[7 * 128 + tid]; }
            }
            __syncthreads();
            continue;
        }
        dense_tile(Q, H, m.w + m.s_wt2g, G, G, P + 16 * 128, nullptr, false, wstage);   // geo -> P rows 16..16+G
        // ---- SH(dir) -> P rows 0..15 --------------------------------------------------------------
        if (tid < TILE_S) {
            float sh[16];
            sh4(misc[3 * 128 + tid], misc[4 * 128 + tid], misc[5 * 128 + tid], sh);
            #pragma unroll
            for (int k = 0; k < 16; k++) P[k * 128 + tid] = sh[k];
        }
        __syncthreads();
        // ---- colour MLP: (16 + G [+ ind via bias]) -> H -> 3, sigmoid ------------------------------
        dense_tile(P, 16 + G, m.w + m.c_wt0, H, H, Q, m.ind ? m.w + m.c_bind : nullptr, true, wstage);
        dense_small(Q, H, m.w + m.c_w1, 3, misc + 9 * 128, misc + 12 * 128);
        // ---- outputs ---------------------------------------------------------------------------------
        if (tid < TILE_S) {
            const uint32_t i = base + tid;
            if (i < M) {
                const float sigma = expf(misc[8 * 128 + tid]);      // trunc_exp forward (utils.py:36-42)
                const float cr = 1.0f / (1.0f + expf(-misc[9 * 128 + tid]));
                const float cg = 1.0f / (1.0f + expf(-misc[10 * 128 + tid]));
                const float cb = 1.0f / (1.0f + expf(-misc[11 * 128 + tid]));
                if (io.out4) io.out4[i] = make_float4(sigma, cr, cg, cb);
                if (io.sigmas) io.sigmas[i] = sigma;
                if (io.rgbs) { io.rgbs[3 * (size_t)i] = cr; io.rgbs[3 * (size_t)i + 1] = cg; io.rgbs[3 * (size_t)i + 2] = cb; }
                if (io.ambient) { io.ambient[2 * (size_t)i] = misc[6 * 128 + tid]; io.ambient[2 * (size_t)i + 1] = misc[7 * 128 + tid]; }
            }
        }
        __syncthreads();
    }
    if (io.stat_samples && blockIdx.x == 0 && tid == 0) atomicAdd(io.stat_samples, (unsigned long long)M);
}

// ======================================================================================
// torso: mask + compaction, field, (mix happens in k_finish)
// ======================================================================================
// F.grid_sample(grid.view(1,1,H,H), coords, align_corners=True), bilinear, zeros padding
__device__ __forceinline__ float bilinear_occ(const float* __restrict__ g, int Hh, float cx, float cy) {
    const float x = (cx + 1.0f) * 0.5f * (float)(Hh - 1), y = (cy + 1.0f) * 0.5f * (float)(Hh - 1);
    const float fx = floorf(x), fy = floorf(y);
    const int x0 = (int)fx, y0 = (int)fy, x1 = x0 + 1, y1 = y0 + 1;
    const float wx1 = x - fx, wx0 = 1.0f - wx1, wy1 = y - fy, wy0 = 1.0f - wy1;
    auto at = [&](int yy, int xx) -> float { return (xx >= 0 && xx < Hh && yy >= 0 && yy < Hh) ? __ldg(g + yy * Hh + xx) : 0.f; };
    return at(y0, x0) * wx0 * wy0 + at(y0, x1) * wx1 * wy0 + at(y1, x0) * wx0 * wy1 + at(y1, x1) * wx1 * wy1;
}

__device__ __forceinline__ float2 bg_coord_of(const TorsoArgs& a, uint32_t n) {
    if (a.bg_coords) return make_float2(a.bg_coords[2 * (size_t)n], a.bg_coords[2 * (size_t)n + 1]);
    // utils.py:273-278: coordinate 0 runs over the FIRST meshgrid axis (size H), 'ij' order:
    // entry n = i * W + j -> (X[i], Y[j]) with X = arange(H)/(H-1)*2-1, Y = arange(W)/(W-1)*2-1
    const uint32_t i = n / a.W, j = n - i * a.W;
    const float X = __fsub_rn(__fmul_rn(__fdiv_rn((float)i, (float)(a.Himg - 1)), 2.0f), 1.0f);
    const float Y = __fsub_rn(__fmul_rn(__fdiv_rn((float)j, (float)(a.W - 1)), 2.0f), 1.0f);
    return make_float2(X, Y);
}

__global__ void k_torso_mask(TorsoArgs a, uint32_t* __restrict__ list, uint32_t* __restrict__ ctl) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    bool on = false;
    if (n < a.N) {
        const float2 c = bg_coord_of(a, n);
        on = bilinear_occ(a.density_grid_torso, a.grid_size, c.x, c.y) > a.thresh;   // radnerf_torso.py:166-168
    }
    const uint32_t ballot = __ballot_sync(0xffffffffu, on);
    const uint32_t lane = threadIdx.x & 31;
    uint32_t base = 0;
    if (lane == 0 && ballot) base = atomicAdd(ctl + CTL_TORSO, __popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (on) list[base + __popc(ballot & ((1u << lane) - 1))] = n;
}

// smem: X [42][128] enc_x | Fq [74][128] (feat 32 + enc_x 42) | P [64][128] | Q [64][128] | wstage | misc
constexpr int TORSO_SMEM_FLOATS = 42 * 128 + 74 * 128 + 64 * 128 + 64 * 128 + 2 * 16 * 128 + 12 * 128;

__global__ void __launch_bounds__(DENSE_THREADS, 1) k_torso_field(ModelDev m, TorsoArgs a, const uint32_t* __restrict__ list,
                                                                   const uint32_t* __restrict__ ctl, const float* __restrict__ bias_deform,
                                                                   const float* __restrict__ bias_canon, float* __restrict__ torso_alpha,
                                                                   float* __restrict__ torso_color) {
    extern __shared__ __align__(16) float smem[];
    float* X = smem;
    float* Fq = X + 42 * 128;
    float* P = Fq + 74 * 128;
    float* Q = P + 64 * 128;
    float* wstage = Q + 64 * 128;
    float* misc = wstage + 2 * 16 * 128;   // [0..1] x (shrunk), [2..3] dx / deformed x, [4..7] out, [8..11] scratch
    const uint32_t M = ctl[CTL_TORSO];
    const int tid = threadIdx.x;
    for (uint32_t tile = blockIdx.x; (uint64_t)tile * TILE_S < M; tile += gridDim.x) {
        const uint32_t base = tile * TILE_S;
        if (tid < TILE_S) {
            const uint32_t i = base + tid;
            float2 c = make_float2(0.f, 0.f);
            if (i < M) c = bg_coord_of(a, list[i]);
            misc[tid] = __fmul_rn(c.x, a.shrink);             // radnerf_torso.py:57
            misc[128 + tid] = __fmul_rn(c.y, a.shrink);
        }
        __syncthreads();
        // enc_x = freq(x, 10): 42 outputs (freqencoder.cu:30-58 with D=2)
        for (int idx = tid; idx < 42 * TILE_S; idx += DENSE_THREADS) {
            const int c = idx >> 7, s = idx & 127;
            float v;
            if (c < 2) v = misc[c * 128 + s];
            else {
                const int col = c / 2 - 1, d = c % 2, freq = col / 2;
                const float phase = (float)(col % 2) * (3.141592653589793f / 2);
                v = __sinf(__fadd_rn(scalbnf(misc[d * 128 + s], freq), phase));
            }
            X[c * 128 + s] = v;
            Fq[(32 + c) * 128 + s] = v;
        }
        __syncthreads();
        // deformation MLP 42(+pose,code via bias) -> 64 -> 64 -> 2
        dense_tile_narrow<4>(X, 42, m.w + m.td_wt0, 64, P, bias_deform, true, wstage);
        dense_tile_narrow<4>(P, 64, m.w + m.td_wt1, 64, Q, nullptr, true, wstage);
        dense_small(Q, 64, m.w + m.td_w2, 2, misc + 2 * 128, misc + 8 * 128);
        if (tid < TILE_S) {
            // x = (x + dx).clamp(-1, 1); grid input (x+1)/2
            misc[2 * 128 + tid] = clampf(__fadd_rn(misc[tid], misc[2 * 128 + tid]), -1.0f, 1.0f);
            misc[3 * 128 + tid] = clampf(__fadd_rn(misc[128 + tid], misc[3 * 128 + tid]), -1.0f, 1.0f);
        }
        __syncthreads();
        {
            const int s = tid & 127;
            const float ax = to_unit(misc[2 * 128 + s], 1.0f), ay = to_unit(misc[3 * 128 + s], 1.0f);
            #pragma unroll 2
            for (int j = 0; j < 8; j++) {
                const int level = (tid >> 7) + 2 * j;
                const float2 f = grid2_sample(m.torso, level, ax, ay);
                Fq[(2 * level) * 128 + s] = f.x;
                Fq[(2 * level + 1) * 128 + s] = f.y;
            }
        }
        __syncthreads();
        // canonical MLP (32 + 42 (+pose,code via bias)) -> 32 -> 32 -> 4, sigmoid
        dense_tile_narrow<2>(Fq, 74, m.w + m.tc_wt0, 32, P, bias_canon, true, wstage);
        dense_tile_narrow<2>(P, 32, m.w + m.tc_wt1, 32, Q, nullptr, true, wstage);
        dense_small(Q, 32, m.w + m.tc_w2, 4, misc + 4 * 128, misc + 8 * 128);
        if (tid < TILE_S) {
            const uint32_t i = base + tid;
            if (i < M) {
                const uint32_t n = list[i];
                torso_alpha[n] = 1.0f / (1.0f + expf(-misc[4 * 128 + tid]));
                torso_color[3 * (size_t)n] = 1.0f / (1.0f + expf(-misc[5 * 128 + tid]));
                torso_color[3 * (size_t)n + 1] = 1.0f / (1.0f + expf(-misc[6 * 128 + tid]));
                torso_color[3 * (size_t)n + 2] = 1.0f / (1.0f + expf(-misc[7 * 128 + tid]));
            }
        }
        __syncthreads();
    }
}

// ======================================================================================
// finish: torso/bg mix, clamp, depth normalise, RGB8   (renderer.py:354-362, radnerf_torso.py:186-196)
// ======================================================================================
__global__ void k_finish(FinishArgs a, RayState st) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= a.N) return;
    float bg[3];
    #pragma unroll
    for (int c = 0; c < 3; c++) bg[c] = a.bg_color ? a.bg_color[3 * (size_t)n + c] : 1.0f;
    if (a.has_torso) {
        const float ta = a.torso_alpha[n];
        #pragma unroll
        for (int c = 0; c < 3; c++) bg[c] = a.torso_color[3 * (size_t)n + c] * ta + bg[c] * (1 - ta);   // radnerf_torso.py:186
        if (a.out_torso_alpha) a.out_torso_alpha[n] = ta;
        if (a.out_torso_rgb) {
            #pragma unroll
            for (int c = 0; c < 3; c++) a.out_torso_rgb[3 * (size_t)n + c] = bg[c];
        }
    }
    const float ws = st.wsum[n];
    #pragma unroll
    for (int c = 0; c < 3; c++) {
        const float v = clampf(st.img[3 * (size_t)n + c] + (1 - ws) * bg[c], 0.f, 1.f);
        a.rgb_map[3 * (size_t)n + c] = v;
        if (a.rgb8) a.rgb8[3 * (size_t)n + c] = (uint8_t)(v * 255.0f);   // (pred_rgb * 255).astype(uint8): truncation
    }
    const float near = st.nears[n], far = st.fars[n];
    a.depth_map[n] = fmaxf(st.depth[n] - near, 0.f) / (far - near);
    if (a.weights_sum) a.weights_sum[n] = ws;
    if (a.n_samples) a.n_samples[n] = st.nsamp[n];
    if (a.term_slot) a.term_slot[n] = st.term[n];
}

__global__ void k_hist_out(const uint32_t* __restrict__ ctl, uint32_t max_steps, uint32_t* __restrict__ out) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > max_steps) return;
    out[k] = k == 0 ? ctl[CTL_STOTAL] : ctl[CTL_HIST + k];
}

__global__ void k_counters_out(const uint32_t* __restrict__ ctl, const unsigned long long* __restrict__ stat, uint64_t* __restrict__ out, uint32_t launches) {
    if (threadIdx.x || blockIdx.x) return;
    out[0] = stat[0];
    out[1] = ctl[CTL_TORSO];
    out[2] = ctl[CTL_STOTAL];
    out[3] = launches;
}

// ======================================================================================
// workspace carving
// ======================================================================================
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Workspace {
    RayState st;
    SampleBuf sb;
    uint32_t* ctl;
    unsigned long long* stat;
    float *bias_amb, *bias_deform, *bias_canon;
    uint32_t* torso_list;
    float *torso_alpha, *torso_color;
    uint4* feat_hi;      // split tensor-core pipeline: fp16 position features, 64 B per sample
    float2* amb_pos;     // split tensor-core pipeline: ambient coordinate per sample
    size_t bytes;
};

static Workspace carve(void* base, uint32_t N) {
    Workspace w;
    size_t off = 0;
    auto take = [&](size_t bytes) -> void* {
        void* p = base ? (void*)((char*)base + off) : nullptr;
        off = align_up(off + bytes, 256);
        return p;
    };
    const size_t cap = (size_t)N * RENDER_CHUNK_MAX;
    w.st.rays_o = (float*)take(sizeof(float) * 3 * N);
    w.st.rays_d = (float*)take(sizeof(float) * 3 * N);
    w.st.nears = (float*)take(sizeof(float) * N);
    w.st.fars = (float*)take(sizeof(float) * N);
    w.st.t = (float*)take(sizeof(float) * N);
    w.st.wsum = (float*)take(sizeof(float) * N);
    w.st.depth = (float*)take(sizeof(float) * N);
    w.st.img = (float*)take(sizeof(float) * 3 * N);
    w.st.alive = (uint8_t*)take(N);
    w.st.nsamp = (int*)take(sizeof(int) * N);
    w.st.term = (int*)take(sizeof(int) * N);
    w.st.seg_off = (uint32_t*)take(sizeof(uint32_t) * N);
    w.st.seg_cnt = (uint32_t*)take(sizeof(uint32_t) * N);
    w.sb.pos4 = (float4*)take(sizeof(float4) * cap);
    w.sb.dl = (float2*)take(sizeof(float2) * cap);
    w.sb.out4 = (float4*)take(sizeof(float4) * cap);
    w.sb.occ_index = nullptr;
    w.ctl = (uint32_t*)take(sizeof(uint32_t) * CTL_WORDS);
    w.stat = (unsigned long long*)take(sizeof(unsigned long long) * 4);
    w.bias_amb = (float*)take(sizeof(float) * 128);
    w.bias_deform = (float*)take(sizeof(float) * 64);
    w.bias_canon = (float*)take(sizeof(float) * 32);
    w.torso_list = (uint32_t*)take(sizeof(uint32_t) * N);
    w.torso_alpha = (float*)take(sizeof(float) * N);
    w.torso_color = (float*)take(sizeof(float) * 3 * N);
    w.feat_hi = (uint4*)take(64 * cap);
    w.amb_pos = (float2*)take(sizeof(float2) * cap);
    w.bytes = off;
    return w;
}

}  // namespace gf

// ======================================================================================
// C ABI
// ======================================================================================
using namespace gf;
#define ST(s) ((cudaStream_t)(s))

namespace gf {
int field_tc_launch(const GfModel* model, const FieldTcIO& io, cudaStream_t st);   // field_tc_split.cu
int field_tc_kernel_count();
int field_tc_pack(GfModel* m, cudaStream_t st);
size_t field_tc_scratch_bytes(uint32_t M);
int gather_probe_launch(const GfModel* model, const float* xyzs, const float* amb_pos, uint32_t M, float* out, cudaStream_t st);
}

extern "C" {

GF_API int gf_model_create(const GfModelDesc* d, GfModel** out, gf_stream_t stream) {
    GF_REQUIRE(d && out, "model_create: null pointer");
    GF_REQUIRE(d->hidden_dim == 128 || d->hidden_dim == 64, "model_create: hidden_dim must be 64 or 128");
    GF_REQUIRE(d->geo_feat_dim >= 8 && d->geo_feat_dim <= 128 && d->geo_feat_dim % 8 == 0, "model_create: geo_feat_dim must be a multiple of 8 in [8,128]");
    GF_REQUIRE(d->cond_dim >= 1 && d->cond_dim <= 256, "model_create: cond_dim out of range");
    GF_REQUIRE(d->ind_dim <= 16 && d->torso_ind_dim <= 10, "model_create: individual code too long");
    GF_REQUIRE(d->cascade >= 1 && d->cascade <= 8 && d->grid_size >= 1 && d->grid_size <= 1024, "model_create: bad cascade/grid_size");
    GF_REQUIRE(d->density_bitfield && d->pos_embeddings && d->pos_offsets && d->amb_embeddings && d->amb_offsets, "model_create: null grid pointer");
    GF_REQUIRE(d->ambient_w0 && d->ambient_w1 && d->ambient_w2 && d->sigma_w0 && d->sigma_w1 && d->sigma_w2 && d->color_w0 && d->color_w1,
               "model_create: null MLP weight pointer");
    GF_REQUIRE(d->ind_dim == 0 || d->ind_code, "model_create: ind_dim > 0 but ind_code is null");
    if (d->has_torso) {
        GF_REQUIRE(d->density_grid_torso && d->torso_embeddings && d->torso_offsets && d->torso_deform_w0 && d->torso_deform_w1 &&
                       d->torso_deform_w2 && d->torso_canon_w0 && d->torso_canon_w1 && d->torso_canon_w2,
                   "model_create: has_torso but a torso pointer is null");
        GF_REQUIRE(d->torso_ind_dim == 0 || d->torso_ind_code, "model_create: torso_ind_dim > 0 but torso_ind_code is null");
    }
    cudaStream_t st = ST(stream);
    GfModel* m = new GfModel();
    memset(m, 0, sizeof(GfModel));
    m->desc = *d;
    const int H = (int)d->hidden_dim, G = (int)d->geo_feat_dim, CD = (int)d->cond_dim, ID = (int)d->ind_dim;
    ModelDev& md = m->dev;
    md.H = H; md.G = G; md.cond = CD; md.ind = ID; md.bound = d->bound;

    // ---- packed fp32 blob layout (floats) ----
    size_t off = 0;
    auto take = [&](size_t n) { size_t o = off; off += (n + 3) / 4 * 4; return (uint32_t)o; };
    md.a_wt0 = take((size_t)32 * H);  md.a_wc = take((size_t)CD * H);  md.a_wt1 = take((size_t)H * H);  md.a_w2 = take((size_t)2 * H);
    md.s_wt0 = take((size_t)64 * H);  md.s_wt1 = take((size_t)H * H);  md.s_wt2g = take((size_t)H * G);  md.s_w2s = take((size_t)H);
    md.c_wt0 = take((size_t)(16 + G) * H);  md.c_bind = take((size_t)H);  md.c_w1 = take((size_t)3 * H);
    const int TI = (int)d->torso_ind_dim;
    const int KC = 54 + TI;
    md.t_ind = TI;
    if (d->has_torso) {
        md.td_wt0 = take((size_t)42 * 64); md.td_wc = take((size_t)KC * 64); md.td_wt1 = take((size_t)64 * 64); md.td_w2 = take((size_t)2 * 64);
        md.tc_wt0 = take((size_t)74 * 32); md.tc_wc = take((size_t)KC * 32); md.tc_wt1 = take((size_t)32 * 32); md.tc_w2 = take((size_t)4 * 32);
        md.t_codeoff = take(16);
    }
    m->w_floats = off;
    float* w = nullptr;
    if (cudaMalloc(&w, off * sizeof(float)) != cudaSuccess) { delete m; set_error("model_create: cudaMalloc failed"); cudaGetLastError(); return GF_ERR_CUDA; }
    cudaMemsetAsync(w, 0, off * sizeof(float), st);
    m->w = w;
    md.w = w;
    auto tp = [&](const float* src, int ldsrc, int k0, int K, int N, uint32_t dst, int ldd) {
        k_transpose_pack<<<div_up((uint32_t)(K * N), 256), 256, 0, st>>>(src, ldsrc, k0, K, N, w + dst, ldd);
    };
    const int a_in = 32 + CD, c_in = 16 + G + ID;
    tp(d->ambient_w0, a_in, 0, 32, H, md.a_wt0, H);
    tp(d->ambient_w0, a_in, 32, CD, H, md.a_wc, H);
    tp(d->ambient_w1, H, 0, H, H, md.a_wt1, H);
    cudaMemcpyAsync(w + md.a_w2, d->ambient_w2, sizeof(float) * 2 * H, cudaMemcpyDeviceToDevice, st);
    tp(d->sigma_w0, 64, 0, 64, H, md.s_wt0, H);
    tp(d->sigma_w1, H, 0, H, H, md.s_wt1, H);
    tp(d->sigma_w2 + H, H, 0, H, G, md.s_wt2g, G);                 // rows 1..G of [1+G][H]
    cudaMemcpyAsync(w + md.s_w2s, d->sigma_w2, sizeof(float) * H, cudaMemcpyDeviceToDevice, st);   // row 0
    tp(d->color_w0, c_in, 0, 16 + G, H, md.c_wt0, H);
    if (ID > 0) {
        k_gemv_fold<<<div_up((uint32_t)H, 128), 128, 0, st>>>(d->color_w0, c_in, 16 + G, ID, H, d->ind_code, w + md.c_bind);
    }
    cudaMemcpyAsync(w + md.c_w1, d->color_w1, sizeof(float) * 3 * H, cudaMemcpyDeviceToDevice, st);
    if (d->has_torso) {
        const int d_in = 42 + KC, q_in = 32 + 42 + KC;
        tp(d->torso_deform_w0, d_in, 0, 42, 64, md.td_wt0, 64);
        tp(d->torso_deform_w0, d_in, 42, KC, 64, md.td_wc, 64);
        tp(d->torso_deform_w1, 64, 0, 64, 64, md.td_wt1, 64);
        cudaMemcpyAsync(w + md.td_w2, d->torso_deform_w2, sizeof(float) * 2 * 64, cudaMemcpyDeviceToDevice, st);
        tp(d->torso_canon_w0, q_in, 0, 74, 32, md.tc_wt0, 32);
        tp(d->torso_canon_w0, q_in, 74, KC, 32, md.tc_wc, 32);
        tp(d->torso_canon_w1, 32, 0, 32, 32, md.tc_wt1, 32);
        cudaMemcpyAsync(w + md.tc_w2, d->torso_canon_w2, sizeof(float) * 4 * 32, cudaMemcpyDeviceToDevice, st);
        if (TI > 0) {
            cudaMemcpyAsync(w + md.t_codeoff, d->torso_ind_code, sizeof(float) * TI, cudaMemcpyDeviceToDevice, st);
            md.t_code = w + md.t_codeoff;
        }
    }
    // ---- level geometry on device ----
    GridLevels* lv_dev = nullptr;
    cudaMalloc(&lv_dev, 3 * sizeof(GridLevels) + 16);
    int* bad_dev = reinterpret_cast<int*>(lv_dev + 3);
    cudaMemsetAsync(lv_dev, 0, 3 * sizeof(GridLevels) + 16, st);
    k_level_geometry<<<1, 32, 0, st>>>(d->pos_offsets, d->pos_S, d->pos_H, 3, d->gridtype, lv_dev + 0, bad_dev);
    k_level_geometry<<<1, 32, 0, st>>>(d->amb_offsets, d->amb_S, d->amb_H, 2, d->gridtype, lv_dev + 1, bad_dev);
    if (d->has_torso) k_level_geometry<<<1, 32, 0, st>>>(d->torso_offsets, d->torso_S, d->torso_H, 2, 1, lv_dev + 2, bad_dev);
    GridLevels lv_host[3];
    int bad_host = 0;
    memset(lv_host, 0, sizeof(lv_host));
    cudaMemcpyAsync(lv_host, lv_dev, 3 * sizeof(GridLevels), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(&bad_host, bad_dev, sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(lv_dev);
    if (e == cudaSuccess && bad_host) {
        set_error("model_create: a grid level is neither dense nor a power of two in size (offsets not produced by GridEncoder?)");
        cudaFree(w);
        delete m;
        return GF_ERR_UNSUPPORTED;
    }
    if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
        set_error("model_create: %s", cudaGetErrorString(e));
        cudaFree(w);
        delete m;
        return GF_ERR_CUDA;
    }
    md.pos.lv = lv_host[0]; md.pos.gridtype = d->gridtype; md.pos.interp = d->interp;
    md.amb.lv = lv_host[1]; md.amb.gridtype = d->gridtype; md.amb.interp = d->interp;
    md.torso.lv = lv_host[2]; md.torso.gridtype = 1; md.torso.interp = 0;   // radnerf_torso.py:36 ('tiledgrid', linear)
    // Padded images of the position and ambient tables (GridLevels::pad): the field kernels' producers address every non-hashed level's
    // corners as rows of adjacent entries.  Copied here, like the weights; the torso table is read in place.
    auto img_entries = [](const GridLevels& lv) { return (size_t)lv.img_offset[15] + lv.hsize[15] + lv.pad[15]; };
    const size_t pos_n = img_entries(lv_host[0]), amb_n = img_entries(lv_host[1]);
    if (cudaMalloc(&m->grid_img, (pos_n + amb_n) * sizeof(float2)) != cudaSuccess) {
        cudaGetLastError();
        set_error("model_create: cudaMalloc of the grid images failed");
        gf_model_destroy(m);
        return GF_ERR_CUDA;
    }
    const dim3 img_grid(256, 16);        // grid-stride over each level
    k_grid_image<<<img_grid, 256, 0, st>>>(reinterpret_cast<const float2*>(d->pos_embeddings), lv_host[0], m->grid_img);
    k_grid_image<<<img_grid, 256, 0, st>>>(reinterpret_cast<const float2*>(d->amb_embeddings), lv_host[1], m->grid_img + pos_n);
    if (int rc = check_launch("model_create: grid images")) { gf_model_destroy(m); return rc; }
    const float2* torso_tab = reinterpret_cast<const float2*>(d->torso_embeddings);
    for (int l = 0; l < 16; l++) {
        md.pos.lbase[l] = m->grid_img + lv_host[0].img_offset[l];
        md.amb.lbase[l] = m->grid_img + pos_n + lv_host[1].img_offset[l];
        md.torso.lbase[l] = torso_tab ? torso_tab + lv_host[2].offset[l] : nullptr;
    }
    // fp16 weight images of the tcgen05 pipeline (field_tc_split.cu): packed here, once -- the frame path never allocates or synchronises
    if (int prc = field_tc_pack(m, st)) { gf_model_destroy(m); return prc; }
    cudaFuncSetAttribute(k_field_fp32, cudaFuncAttributeMaxDynamicSharedMemorySize, FP32_SMEM_FLOATS * (int)sizeof(float));
    cudaFuncSetAttribute(k_torso_field, cudaFuncAttributeMaxDynamicSharedMemorySize, TORSO_SMEM_FLOATS * (int)sizeof(float));
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&m->num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (m->num_sms <= 0) m->num_sms = 148;
    *out = m;
    return check_launch("model_create");
}

GF_API void gf_model_destroy(GfModel* m) {
    if (!m) return;
    if (m->w) cudaFree(m->w);
    if (m->grid_img) cudaFree(m->grid_img);
    if (m->tc2_blob) cudaFree(m->tc2_blob);
    for (int i = 0; i < GF_MAX_PROFILE_EVENTS; i++)
        if (m->ev[i]) cudaEventDestroy(m->ev[i]);
    delete m;
}

GF_API int gf_profile_enable(GfModel* m, int enable) {
    if (!m) return GF_ERR_INVALID;
    m->profiling = enable != 0;
    m->ev_used = 0;
    return GF_OK;
}

// Sum of the CUDA-event durations (ms) of the field launches of the LAST gf_render_frame call; the caller must have
// synchronised the stream.  *n_launches receives the number of bracketed launches.
GF_API int gf_profile_field_ms(GfModel* m, float* total_ms, int* n_launches) {
    if (!m || !total_ms) return GF_ERR_INVALID;
    float tot = 0.f;
    int n = 0;
    for (int i = 0; i + 1 < m->ev_used; i += 2) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, m->ev[i], m->ev[i + 1]) != cudaSuccess) { cudaGetLastError(); set_error("profile: events not complete"); return GF_ERR_CUDA; }
        tot += ms;
        n++;
    }
    *total_ms = tot;
    if (n_launches) *n_launches = n;
    return GF_OK;
}

GF_API uint64_t gf_model_packed_bytes(const GfModel* m) { return m ? (uint64_t)m->w_floats * sizeof(float) : 0; }

GF_API uint64_t gf_render_workspace_bytes(uint32_t N) { return (uint64_t)carve(nullptr, N).bytes; }

// get_rays (modules/radnerfs/utils.py:282-363) for B poses and a list of N flat pixel indices (NULL: N must be H*W, all pixels in
// row-major order).  poses: device [B,4,4] c2w; outputs caller-allocated: rays_o / rays_d [B,N,3]; i / j [N] pixel-centre coordinates or NULL.
GF_API int gf_get_rays(const float* poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t H, uint32_t W, const int64_t* inds,
                       uint32_t N, float* rays_o, float* rays_d, float* i, float* j, gf_stream_t stream) {
    GF_REQUIRE(poses && rays_o && rays_d, "get_rays: null pointer");
    GF_REQUIRE(H >= 1 && W >= 1 && (uint64_t)H * W < (1ull << 31), "get_rays: bad H/W");
    GF_REQUIRE(inds || N == H * W, "get_rays: without an index list N must be H*W");
    GF_REQUIRE((uint64_t)B * N < (1ull << 32), "get_rays: B*N too large");
    if (B == 0 || N == 0) return GF_OK;
    k_get_rays<<<div_up(B * N, 256), 256, 0, ST(stream)>>>(poses, B, fx, fy, cx, cy, W, inds, N, rays_o, rays_d, i, j);
    return check_launch("get_rays");
}

// Measurement aid: the field's grid gathers alone (3-D position grid at xyzs [M,3] + 2-D ambient grid at amb_pos [M,2]; out [M,2] =
// the sum of the 32 gathered feature pairs), by the very gather code of the tcgen05 field kernels' producer warps.  bench.py times it for
// roofline.frac_of_gather_ceiling; it is not part of the render path.
GF_API int gf_gather_probe(const GfModel* model, const float* xyzs, const float* amb_pos, uint32_t M, float* out, gf_stream_t stream) {
    GF_REQUIRE(model && xyzs && amb_pos && out, "gather_probe: null pointer");
    if (M == 0) return GF_OK;
    return gather_probe_launch(model, xyzs, amb_pos, M, out, ST(stream));
}

GF_API uint64_t gf_field_workspace_bytes(uint32_t M, uint32_t precision) {
    return 1024 + (precision ? (uint64_t)field_tc_scratch_bytes(M) : 0);
}

// Standalone field evaluation: the `self(xyzs, dirs, cond_feat, ind_code)` call of the reference loop
// (renderer.py:342 -> radnerf.py:73-105).  xyzs/dirs [M,3]; sigmas [M]; rgbs [M,3]; ambient [M,2] or NULL.
// workspace: caller-owned device scratch of gf_field_workspace_bytes(M, precision) bytes, 256-byte aligned (per-call cond bias +,
// for precision 1, the hand-off buffers between the two tcgen05 kernels).  The model is not modified: re-entrant across streams.
GF_API int gf_field_forward(const GfModel* model, const float* xyzs, const float* dirs, const float* cond_feat, uint32_t M, float* sigmas,
                            float* rgbs, float* ambient, uint32_t precision, void* workspace, uint64_t workspace_bytes, gf_stream_t stream) {
    GF_REQUIRE(model && xyzs && cond_feat && sigmas, "field_forward: null pointer");
    GF_REQUIRE(dirs || !rgbs, "field_forward: dirs may be NULL only for a density query (rgbs == NULL)");
    GF_REQUIRE(precision <= 1, "field_forward: precision must be 0 (fp32) or 1 (fp16 tensor cores)");
    if (M == 0) return GF_OK;
    GF_REQUIRE(workspace && ((uintptr_t)workspace & 255) == 0, "field_forward: workspace must be a 256-byte aligned device pointer");
    GF_REQUIRE(workspace_bytes >= gf_field_workspace_bytes(M, precision), "field_forward: workspace too small (%llu < %llu)",
               (unsigned long long)workspace_bytes, (unsigned long long)gf_field_workspace_bytes(M, precision));
    cudaStream_t st = ST(stream);
    float* bias = reinterpret_cast<float*>(workspace);
    FrameSetup fs;
    memset(&fs, 0, sizeof(fs));
    fs.cond_feat = cond_feat;
    fs.has_torso = 0;
    k_frame_setup<<<1, 128, 0, st>>>(model->dev, fs, bias, nullptr, nullptr);
    if (precision == 0) {
        FieldIO io;
        memset(&io, 0, sizeof(io));
        io.xyzs = xyzs; io.dirs = dirs; io.M_host = M; io.sigmas = sigmas; io.rgbs = rgbs; io.ambient = ambient; io.bias_amb = bias;
        const uint32_t tiles = div_up(M, TILE_S);
        const uint32_t grid = tiles < (uint32_t)model->num_sms ? tiles : (uint32_t)model->num_sms;
        k_field_fp32<<<grid, DENSE_THREADS, FP32_SMEM_FLOATS * sizeof(float), st>>>(model->dev, io);
        return check_launch("field_forward(fp32)");
    }
    FieldTcIO io;
    memset(&io, 0, sizeof(io));
    io.xyzs = xyzs; io.dirs = dirs; io.M_host = M; io.sigmas = sigmas; io.rgbs = rgbs; io.ambient = ambient; io.bias_amb = bias;
    char* scr = reinterpret_cast<char*>(workspace) + 1024;
    io.feat_hi = reinterpret_cast<uint4*>(scr);
    io.amb_pos = reinterpret_cast<float2*>(scr + (((size_t)M * 64 + 255) & ~size_t(255)));
    return field_tc_launch(model, io, st);
}

GF_API int gf_render_frame(const GfModel* model, const GfFrame* f, const GfOut* o, void* workspace, uint64_t workspace_bytes,
                           gf_stream_t stream) {
    GF_REQUIRE(model && f && o && workspace, "render_frame: null pointer");
    GF_REQUIRE(o->rgb_map && o->depth_map, "render_frame: rgb_map and depth_map are required outputs");
    GF_REQUIRE(f->cond_feat, "render_frame: cond_feat is required");
    GF_REQUIRE((f->rays_o == nullptr) == (f->rays_d == nullptr), "render_frame: give both rays_o and rays_d or neither");
    GF_REQUIRE(f->H >= 1 && f->W >= 1 && (uint64_t)f->H * f->W < (1ull << 26), "render_frame: bad H/W");
    GF_REQUIRE(f->max_steps >= 1 && f->max_steps <= RENDER_MAX_STEPS, "render_frame: max_steps must be in [1, %d]", RENDER_MAX_STEPS);
    GF_REQUIRE(f->precision <= 1, "render_frame: precision must be 0 (fp32) or 1 (fp16 tensor cores)");
    const uint32_t N = f->H * f->W;
    const Workspace w = carve(workspace, N);
    GF_REQUIRE(workspace_bytes >= w.bytes, "render_frame: workspace too small (%llu < %llu)", (unsigned long long)workspace_bytes,
               (unsigned long long)w.bytes);
    GF_REQUIRE(((uintptr_t)workspace & 255) == 0, "render_frame: workspace must be 256-byte aligned");
    const GfModelDesc& d = model->desc;
    cudaStream_t st = ST(stream);
    const bool torso = d.has_torso != 0;
    uint32_t launches = 0;
    int rc;

    // control words + counters
    k_zero_u32<<<div_up(CTL_WORDS + 8, 256), 256, 0, st>>>(w.ctl, CTL_WORDS);
    cudaMemsetAsync(w.stat, 0, sizeof(unsigned long long) * 4, st);
    launches++;

    FrameSetup fs;
    memset(&fs, 0, sizeof(fs));
    fs.cond_feat = f->cond_feat;
    memcpy(fs.torso_pose, f->torso_pose, sizeof(float) * 6);
    fs.has_torso = torso;
    fs.dyn = f->dyn;
    k_frame_setup<<<torso ? 2 : 1, 128, 0, st>>>(model->dev, fs, w.bias_amb, w.bias_deform, w.bias_canon);
    launches++;

    RayInit ri;
    memset(&ri, 0, sizeof(ri));
    ri.N = N; ri.W = f->W; ri.rays_o = f->rays_o; ri.rays_d = f->rays_d;
    memcpy(ri.pose, f->pose, sizeof(float) * 12);
    ri.dyn = f->dyn;
    ri.fx = f->intrinsics[0]; ri.fy = f->intrinsics[1]; ri.cx = f->intrinsics[2]; ri.cy = f->intrinsics[3];
    memcpy(ri.aabb, d.aabb, sizeof(float) * 6);
    ri.min_near = d.min_near;
    k_rays_init<<<div_up(N, 128), 128, 0, st>>>(ri, w.st);
    launches++;
    if ((rc = check_launch("render_frame(init)"))) return rc;

    MarchArgs ma;
    memset(&ma, 0, sizeof(ma));
    ma.N = N; ma.bound = d.bound; ma.dt_gamma = f->dt_gamma; ma.max_steps = f->max_steps; ma.C = d.cascade; ma.H = d.grid_size;
    ma.grid = d.density_bitfield;
    CompArgs ca;
    memset(&ca, 0, sizeof(ca));
    ca.N = N; ca.T_thresh = f->T_thresh; ca.max_steps = f->max_steps;

    const uint32_t chunk = RENDER_CHUNK_MAX;
    GfModel* prof = model->profiling ? const_cast<GfModel*>(model) : nullptr;
    if (prof) prof->ev_used = 0;
    auto field_inner = [&](void) -> int {
        if (f->precision == 0) {
            FieldIO io;
            memset(&io, 0, sizeof(io));
            io.pos4 = w.sb.pos4; io.rays_d = w.st.rays_d; io.M_dev = w.ctl + CTL_TOTAL; io.out4 = w.sb.out4; io.bias_amb = w.bias_amb;
            io.stat_samples = w.stat;
            k_field_fp32<<<model->num_sms, DENSE_THREADS, FP32_SMEM_FLOATS * sizeof(float), st>>>(model->dev, io);
            return check_launch("render_frame(field fp32)");
        }
        FieldTcIO io;
        memset(&io, 0, sizeof(io));
        io.pos4 = w.sb.pos4; io.rays_d = w.st.rays_d; io.M_dev = w.ctl + CTL_TOTAL; io.out4 = w.sb.out4; io.bias_amb = w.bias_amb;
        io.stat_samples = w.stat;
        io.feat_hi = w.feat_hi; io.amb_pos = w.amb_pos;
        return field_tc_launch(model, io, st);
    };
    // optional CUDA-event bracket around every field launch (gf_profile_*): the dominant-kernel timing bench.py reports
    auto field = [&](void) -> int {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (prof && prof->ev_used + 2 <= GF_MAX_PROFILE_EVENTS) {
            for (int k = 0; k < 2; k++)
                if (!prof->ev[prof->ev_used + k]) cudaEventCreate(&prof->ev[prof->ev_used + k]);
            e0 = prof->ev[prof->ev_used]; e1 = prof->ev[prof->ev_used + 1];
            prof->ev_used += 2;
            cudaEventRecord(e0, st);
        }
        const int r = field_inner();
        if (e1) cudaEventRecord(e1, st);
        return r;
    };

    const uint32_t field_kernels = f->precision == 0 ? 1u : (uint32_t)field_tc_kernel_count();
    // pass A: rounds covering exactly max_steps slots
    for (uint32_t before = 0; before < f->max_steps; before += chunk) {
        const uint32_t budget = (f->max_steps - before) < chunk ? (f->max_steps - before) : chunk;
        if (before) { k_zero_u32<<<1, 32, 0, st>>>(w.ctl + CTL_TOTAL, 1); launches++; }
        ma.budget = budget; ma.budget_from_ctl = 0;
        k_march_chunk<<<div_up(N, 128), 128, 0, st>>>(ma, w.st, w.sb, w.ctl);
        if ((rc = field())) return rc;
        ca.budget = budget; ca.budget_from_ctl = 0; ca.slots_before = before;
        k_composite_chunk<<<div_up(N, 128), 128, 0, st>>>(ca, w.st, w.sb, w.ctl);
        launches += 2 + field_kernels;
    }
    // schedule replay -> S_total; extra round with device-side budget
    k_schedule<<<1, 128, 0, st>>>(N, f->max_steps, w.ctl);
    ma.budget = 0; ma.budget_from_ctl = 1;
    k_march_chunk<<<div_up(N, 128), 128, 0, st>>>(ma, w.st, w.sb, w.ctl);
    if ((rc = field())) return rc;
    ca.budget = 0; ca.budget_from_ctl = 1; ca.slots_before = f->max_steps;
    k_composite_chunk<<<div_up(N, 128), 128, 0, st>>>(ca, w.st, w.sb, w.ctl);
    launches += 3 + field_kernels;
    if ((rc = check_launch("render_frame(rounds)"))) return rc;

    FinishArgs fa;
    memset(&fa, 0, sizeof(fa));
    if (torso) {
        TorsoArgs ta;
        memset(&ta, 0, sizeof(ta));
        ta.N = N; ta.W = f->W; ta.Himg = f->H; ta.bg_coords = f->bg_coords; ta.density_grid_torso = d.density_grid_torso;
        ta.grid_size = (int)d.grid_size; ta.thresh = d.density_thresh_torso; ta.shrink = d.torso_shrink;
        cudaMemsetAsync(w.torso_alpha, 0, sizeof(float) * N, st);          // torso_alpha = zeros (radnerf_torso.py:171-172)
        cudaMemsetAsync(w.torso_color, 0, sizeof(float) * 3 * N, st);
        k_torso_mask<<<div_up(N, 256), 256, 0, st>>>(ta, w.torso_list, w.ctl);
        k_torso_field<<<model->num_sms, DENSE_THREADS, TORSO_SMEM_FLOATS * sizeof(float), st>>>(model->dev, ta, w.torso_list, w.ctl, w.bias_deform,
                                                                                                 w.bias_canon, w.torso_alpha, w.torso_color);
        launches += 2;
        fa.has_torso = 1; fa.torso_alpha = w.torso_alpha; fa.torso_color = w.torso_color;
        fa.out_torso_alpha = o->torso_alpha_map; fa.out_torso_rgb = o->torso_rgb_map;
    }
    fa.N = N; fa.bg_color = f->bg_color; fa.rgb_map = o->rgb_map; fa.depth_map = o->depth_map; fa.weights_sum = o->weights_sum;
    fa.n_samples = o->n_samples; fa.term_slot = o->term_slot; fa.rgb8 = o->rgb8;
    k_finish<<<div_up(N, 256), 256, 0, st>>>(fa, w.st);
    launches++;
    if (o->term_hist) k_hist_out<<<div_up(f->max_steps + 1, 256), 256, 0, st>>>(w.ctl, f->max_steps, o->term_hist);
    if (o->counters) { k_counters_out<<<1, 32, 0, st>>>(w.ctl, w.stat, o->counters, launches + 1); }
    return check_launch("render_frame(finish)");
}

}  // extern "C"
