// tcgen05 / TMEM / mbarrier / TMA-bulk PTX wrappers and operand-layout helpers shared by the tensor-core field kernels.
#pragma once
#include <cuda_fp16.h>

#include "gf_common.cuh"

namespace gf {

// swizzled byte offset of 16-byte unit `u` (0..7) of row `r` inside a [rows x 128 B] block
__host__ __device__ __forceinline__ uint32_t sw128(uint32_t r, uint32_t u) { return r * 128 + ((u ^ (r & 7)) << 4); }

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void bar_stream(uint32_t id) { asm volatile("bar.sync %0, 256;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void bar_named(uint32_t id, uint32_t nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO=1 | SBO=1024>>4 | version=1 | layout=2
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D=f32, A=B=f16, both K-major, M=128
__host__ __device__ constexpr uint32_t idesc_f16(uint32_t N) { return (1u << 4) | ((N >> 3) << 17) | ((128u >> 4) << 24); }

__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// elect.sync on the full warp (call it convergently, right after a warp-uniform test): true in exactly one lane
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred = 0, lane = 0;
    asm volatile(
        "{\n\t.reg .b32 %%rx;\n\t.reg .pred %%px;\n\t"
        "elect.sync %%rx|%%px, %2;\n\t"
        "@%%px mov.s32 %1, 1;\n\t"
        "mov.s32 %0, %%rx;\n\t}"
        : "+r"(lane), "+r"(pred)
        : "r"(0xFFFFFFFFu));
    return pred != 0;
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    #pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
    uint32_t r0, r1, r2, r3;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// explicit shared-space accesses by 32-bit shared address.  The kernels' smem pointer is derived from an aligned-up extern array through integer
// arithmetic, so plain C++ dereferences compile to GENERIC LD.E / ST.E (address-space check on every access; seen in SASS and as long-scoreboard
// stalls of the bias loads in the ncu source view, profiles/r02_summary.md section 7); these compile to LDS / STS.
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts128f(uint32_t saddr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// per-thread asynchronous global -> shared copies (LDGSTS): completion is tracked by the async-group counter, not by the register scoreboards
// the compiler shares between unrelated loads
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory"); }
__device__ __forceinline__ void cp_async4(uint32_t saddr, const void* g) { asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr), "l"(g) : "memory"); }
__device__ __forceinline__ void cp_async8(uint32_t saddr, const void* g) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(saddr), "l"(g) : "memory"); }
__device__ __forceinline__ float2 lds64(uint32_t saddr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Packed two-lane fp32 arithmetic (Blackwell FFMA2 / FADD2 / FMUL2): each lane is the same IEEE operation, with the same rounding, as the
// scalar __fmaf_rn / __fadd_rn / __fsub_rn / __fmul_rn (/ __fadd_rd) on that lane, so replacing a pair of scalar operations by one of these keeps
// results bit-identical.  The register-pair moves disappear in SASS when ptxas keeps the float2 in an aligned pair; a lane-broadcast first
// operand (make_float2(w, w)) compiles to the .F32 operand form, without a move.
__device__ __forceinline__ uint64_t f2_pack(float2 a) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
    return r;
}
__device__ __forceinline__ float2 f2_unpack(uint64_t r) {
    float2 d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(r));
    return d;
}
// d = a * b + c
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)), "l"(f2_pack(c)));
    return f2_unpack(d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
    return f2_unpack(d);
}
// rounding toward minus infinity (floor_split2)
__device__ __forceinline__ float2 fadd2_rm(float2 a, float2 b) {
    uint64_t d;
    asm("add.rm.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
    return f2_unpack(d);
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) {
    uint64_t d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
    return f2_unpack(d);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
    return f2_unpack(d);
}
__device__ __forceinline__ float2 bcast2(float w) { return make_float2(w, w); }

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}

// ReLU + fp16x2 pack in ONE instruction (cvt.relu): low half = max(lo, 0), high half = max(hi, 0)
__device__ __forceinline__ uint32_t pack_relu_h2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// same, rounding toward zero: for v >= 0 the packed value never exceeds v, so the residual v - hi is >= 0
__device__ __forceinline__ uint32_t pack_relu_rz_h2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float2 unpack_h2(uint32_t p) { return __half22float2(*reinterpret_cast<const __half2*>(&p)); }
// fp16 hi/lo split of two values: hi = rn(f), lo = rn(f - hi) (the part fp16 drops), each packed as fp16x2
__device__ __forceinline__ void pack_hilo_h2(float2 f, uint32_t& hi, uint32_t& lo) {
    hi = pack_h2(f.x, f.y);
    const float2 r = fsub2(f, unpack_h2(hi));
    lo = pack_h2(r.x, r.y);
}

// NCHUNK x 32 accumulator columns starting at col0 (this thread's TMEM lane) -> (+bias) -> ReLU -> fp16 -> A operand region.
// SPLIT: also emit the fp16 residual into a second A region (hi + lo ~ 21-bit operand): hi = rz(relu(v)) so that the
// residual relu(v) - hi is non-negative and a second cvt.relu packs it (a negative v gives hi = 0 and residual v -> 0).
template <bool SPLIT, int NCHUNK>
__device__ __forceinline__ void epilogue_relu_to_A_n(uint32_t t_d, uint32_t t_a, uint32_t t_alo, int col0, uint32_t bias_saddr, float* dbg) {
    #pragma unroll 1
    for (int c = 0; c < NCHUNK; c++) {
        const int col = col0 + 32 * c;
        float v[32];
        tmem_ld32(t_d + col, v);
        if (dbg) {
            #pragma unroll
            for (int i = 0; i < 32; i++) dbg[col + i] = v[i];
        }
        if (bias_saddr) {
            #pragma unroll
            for (int i = 0; i < 32; i += 4) {
                const float4 b = lds128(bias_saddr + 4 * (col + i));
                v[i] += b.x; v[i + 1] += b.y; v[i + 2] += b.z; v[i + 3] += b.w;
            }
        }
        uint32_t p[16];
        if (SPLIT) {
            #pragma unroll
            for (int i = 0; i < 16; i++) p[i] = pack_relu_rz_h2(v[2 * i], v[2 * i + 1]);
            tmem_st16(t_a + (col >> 1), p);
            #pragma unroll
            for (int i = 0; i < 16; i++) {
                const float2 h = unpack_h2(p[i]);
                p[i] = pack_relu_h2(v[2 * i] - h.x, v[2 * i + 1] - h.y);
            }
            tmem_st16(t_alo + (col >> 1), p);
        } else {
            #pragma unroll
            for (int i = 0; i < 16; i++) p[i] = pack_relu_h2(v[2 * i], v[2 * i + 1]);
            tmem_st16(t_a + (col >> 1), p);
        }
    }
    tmem_wait_st();
}

// asynchronous 32-column accumulator load + the matching wait.  The wait names the destination registers as in/out operands so
// that no use of them can be scheduled above it.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld32(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
                   "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]),
                   "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]),
                   "+r"(r[31])
                 :
                 : "memory");
}

// 128 accumulator columns -> (+bias) -> ReLU -> fp16 A operand, software-pipelined: the load of chunk c+1 is in flight while
// chunk c is converted and stored (this epilogue sits on the consumer streams' critical path).
template <bool BIAS>
__device__ __forceinline__ void epilogue_relu_to_A_pipe(uint32_t t_d, uint32_t t_a, uint32_t bias_saddr, float* dbg) {
    uint32_t r[2][32];
    tmem_ld32_issue(t_d, r[0]);
    tmem_wait_ld32(r[0]);
    #pragma unroll
    for (int c = 0; c < 4; c++) {
        uint32_t (&cur)[32] = r[c & 1];
        if (c < 3) tmem_ld32_issue(t_d + 32 * (c + 1), r[(c + 1) & 1]);
        if (dbg) {
            #pragma unroll
            for (int i = 0; i < 32; i++) dbg[32 * c + i] = __uint_as_float(cur[i]);
        }
        uint32_t p[16];
        #pragma unroll
        for (int i = 0; i < 16; i += 2) {
            float2 v01 = make_float2(__uint_as_float(cur[2 * i]), __uint_as_float(cur[2 * i + 1]));
            float2 v23 = make_float2(__uint_as_float(cur[2 * i + 2]), __uint_as_float(cur[2 * i + 3]));
            if (BIAS) {
                const float4 b = lds128(bias_saddr + 4 * (32 * c + 2 * i));
                v01 = fadd2(v01, make_float2(b.x, b.y));
                v23 = fadd2(v23, make_float2(b.z, b.w));
            }
            p[i] = pack_relu_h2(v01.x, v01.y);
            p[i + 1] = pack_relu_h2(v23.x, v23.y);
        }
        tmem_st16(t_a + 16 * c, p);
        if (c < 3) tmem_wait_ld32(r[(c + 1) & 1]);
    }
    tmem_wait_st();
}

// split-precision form of the above (ambient layer 0 -> layer 1): + bias, hi = rz(relu(v)), lo = relu(v - hi), both stored as A operands; the
// accumulator load of chunk c+1 is in flight while chunk c is converted
__device__ __forceinline__ void epilogue_split_to_A_pipe(uint32_t t_d, uint32_t t_a, uint32_t t_alo, uint32_t bias_saddr, float* dbg) {
    uint32_t r[2][32];
    tmem_ld32_issue(t_d, r[0]);
    tmem_wait_ld32(r[0]);
    #pragma unroll
    for (int c = 0; c < 4; c++) {
        uint32_t (&cur)[32] = r[c & 1];
        if (c < 3) tmem_ld32_issue(t_d + 32 * (c + 1), r[(c + 1) & 1]);
        if (dbg) {
            #pragma unroll
            for (int i = 0; i < 32; i++) dbg[32 * c + i] = __uint_as_float(cur[i]);
        }
        uint32_t p[16], q[16];
        #pragma unroll
        for (int i = 0; i < 16; i += 2) {
            const float4 b = lds128(bias_saddr + 4 * (32 * c + 2 * i));
            const float2 v01 = fadd2(make_float2(__uint_as_float(cur[2 * i]), __uint_as_float(cur[2 * i + 1])), make_float2(b.x, b.y));
            const float2 v23 = fadd2(make_float2(__uint_as_float(cur[2 * i + 2]), __uint_as_float(cur[2 * i + 3])), make_float2(b.z, b.w));
            p[i] = pack_relu_rz_h2(v01.x, v01.y);
            p[i + 1] = pack_relu_rz_h2(v23.x, v23.y);
            const float2 l01 = fsub2(v01, unpack_h2(p[i])), l23 = fsub2(v23, unpack_h2(p[i + 1]));
            q[i] = pack_relu_h2(l01.x, l01.y);
            q[i + 1] = pack_relu_h2(l23.x, l23.y);
        }
        tmem_st16(t_a + 16 * c, p);
        tmem_st16(t_alo + 16 * c, q);
        if (c < 3) tmem_wait_ld32(r[(c + 1) & 1]);
    }
    tmem_wait_st();
}


}  // namespace gf
