// Host/device structs shared by render_fused.cu and field_tc_split.cu.
#pragma once
#include "gf_field.cuh"

namespace gf {

constexpr uint32_t RENDER_CHUNK_MAX = 32;    // slots offered to a live ray per round
constexpr uint32_t RENDER_MAX_STEPS = 1024;  // render(max_steps=...) upper bound (reference default, renderer.py:263)

// control words (uint32) in the workspace
constexpr uint32_t CTL_TOTAL = 0;    // sample-list length of the current round (allocation cursor)
constexpr uint32_t CTL_STOTAL = 1;   // S_total = slots offered to a surviving ray by the reference's host loop
constexpr uint32_t CTL_EXTRA = 2;    // S_total - max_steps (budget of the extra round)
constexpr uint32_t CTL_TORSO = 3;    // masked torso pixel count
constexpr uint32_t CTL_HIST = 8;     // hist[k], k = 1..max_steps: rays whose termination slot is k
constexpr uint32_t CTL_WORDS = CTL_HIST + RENDER_MAX_STEPS + 8;

// Packed fp32 model, passed BY VALUE to kernels (lives in the constant bank).
struct ModelDev {
    GridDesc pos, amb, torso;
    float bound;
    int H, G, cond, ind, t_ind;
    const float* w;          // packed fp32 blob; all offsets below are in floats
    const float* t_code;     // torso individual code (in the blob) or null
    // head field (transposed = [K][N] k-major)
    uint32_t a_wt0, a_wc, a_wt1, a_w2;
    uint32_t s_wt0, s_wt1, s_wt2g, s_w2s;
    uint32_t c_wt0, c_bind, c_w1;
    // torso
    uint32_t td_wt0, td_wc, td_wt1, td_w2, tc_wt0, tc_wc, tc_wt1, tc_w2, t_codeoff;
};

struct RayState {
    float *rays_o, *rays_d;   // [N,3]
    float *nears, *fars, *t;  // [N]
    float *wsum, *depth, *img;
    uint8_t* alive;
    int* nsamp;
    int* term;                // termination slot (1-based) of a dead ray, 0 while alive
    uint32_t *seg_off, *seg_cnt;
};

struct SampleBuf {
    float4* pos4;         // x, y, z, ray id (bit-cast)
    float2* dl;           // dt, t_end
    float4* out4;         // sigma, r, g, b
    uint32_t* occ_index;  // occupancy bit index per sample (diagnostics) or null
};

struct RayInit {
    uint32_t N, W;
    const float *rays_o, *rays_d;
    float pose[12];
    float fx, fy, cx, cy;
    float aabb[6];
    float min_near;
    const float* dyn;          // GfFrame.dyn or null
};

struct MarchArgs {
    uint32_t N;
    float bound, dt_gamma;
    uint32_t max_steps, C, H;
    const uint8_t* grid;
    uint32_t budget;
    int budget_from_ctl;
};

struct CompArgs {
    uint32_t N;
    float T_thresh;
    uint32_t max_steps, budget, slots_before;
    int budget_from_ctl;
};

struct TorsoArgs {
    uint32_t N, W, Himg;
    const float* bg_coords;
    const float* density_grid_torso;
    int grid_size;
    float thresh, shrink;
};

struct FinishArgs {
    uint32_t N;
    const float* bg_color;
    int has_torso;
    const float *torso_alpha, *torso_color;
    float *out_torso_alpha, *out_torso_rgb;
    float *rgb_map, *depth_map, *weights_sum;
    int32_t* n_samples;
    int32_t* term_slot;
    uint8_t* rgb8;
};

// IO of the tensor-core field kernels (field_tc_split.cu); mirrors FieldIO of the fp32 kernel.
struct FieldTcIO {
    const float4* pos4;
    const float* rays_d;
    const float* xyzs;
    const float* dirs;
    const uint32_t* M_dev;
    uint32_t M_host;
    float4* out4;
    float* sigmas;
    float* rgbs;
    float* ambient;
    const float* bias_amb;
    unsigned long long* stat_samples;
    // scratch of the split (two-kernel) pipeline; null -> model-owned scratch
    uint4* feat_hi;        // [M][4] uint4 = 32 fp16 position features per sample
    float2* amb_pos;       // [M] ambient coordinates
};

}  // namespace gf

#define GF_MAX_PROFILE_EVENTS 96

// Opaque handle of the C ABI.
struct GfModel {
    GfModelDesc desc;
    gf::ModelDev dev;
    float* w;               // packed fp32 blob (device)
    size_t w_floats;
    float w_amb2_host[256]; // fp32 ambient output layer [2][128] (host copy, passed by value to k_tc_amb)
    float2* grid_img;       // padded images of the position and ambient grid tables (device, one allocation; GridLevels::pad)
    void* tc2_blob;         // fp16 weight images of the two tcgen05 kernels (device), built in gf_model_create; null outside the envelope
    float* tc_dbg;          // diagnostics buffer for the tcgen05 kernel (gf_tc_debug) or null
    int num_sms;
    int profiling, ev_used;
    cudaEvent_t ev[GF_MAX_PROFILE_EVENTS];
};
