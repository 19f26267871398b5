/*
 * gfrender.h -- C ABI of libgfrender.so, the B200-native (sm_100a) replacement for the
 * RAD-NeRF hot path of yerfor/GeneFace.
 *
 * Every entry point takes raw DEVICE pointers, sizes and scalars plus an explicit CUDA
 * stream; there are no torch types anywhere in this header.  Return value: 0 on success,
 * negative on error (gf_last_error() returns a thread-local description).  The caller
 * allocates every output (SURVEY.md section 8b "Ownership"); kernels never allocate, free or
 * retain pointers, except the opaque GfModel which owns a packed copy of the weights.
 *
 * Each declaration cites the reference interface it replaces (paths under the reference
 * tree, yerfor/GeneFace @ 15ff4e5c).  Argument order follows the reference's pybind
 * functions so that a binding is a 1:1 forward (INTEGRATION.md shows the ctypes stub).
 */
#ifndef GFRENDER_H_
#define GFRENDER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GF_API __attribute__((visibility("default")))
#else
#define GF_API
#endif

typedef void* gf_stream_t; /* cudaStream_t (CUstream); NULL = legacy default stream */

#define GF_OK 0
#define GF_ERR_INVALID -22   /* bad argument (EINVAL) */
#define GF_ERR_CUDA -5       /* CUDA runtime error (EIO) */
#define GF_ERR_UNSUPPORTED -95

GF_API const char* gf_last_error(void);
GF_API int gf_version(void);
/* 1 when a CUDA device with compute capability 10.x is current, else 0 (no exception). */
GF_API int gf_device_ok(void);

/* ------------------------------------------------------------------------------------
 * _raymarching_face   modules/radnerfs/raymarching/src/raymarching.h:7-20
 * ---------------------------------------------------------------------------------- */
/* raymarching.h:7   near_far_from_aabb(rays_o, rays_d, aabb, N, min_near, nears, fars) */
GF_API int gf_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N,
                                 float min_near, float* nears, float* fars, gf_stream_t stream);
/* raymarching.h:8   sph_from_ray(rays_o, rays_d, radius, N, coords) */
GF_API int gf_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords,
                           gf_stream_t stream);
/* raymarching.h:9   morton3D(coords, N, indices) */
GF_API int gf_morton3D(const int32_t* coords, uint32_t N, int32_t* indices, gf_stream_t stream);
/* raymarching.h:10  morton3D_invert(indices, N, coords) */
GF_API int gf_morton3D_invert(const int32_t* indices, uint32_t N, int32_t* coords, gf_stream_t stream);
/* raymarching.h:11  packbits(grid, N, density_thresh, bitfield)   N = C*H^3/8 bytes */
GF_API int gf_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield, gf_stream_t stream);
/* raymarching.h:12  morton3D_dilation(grid, C, H, grid_dilation) */
GF_API int gf_morton3D_dilation(const float* grid, uint32_t C, uint32_t H, float* grid_dilation, gf_stream_t stream);
/* raymarching.h:14  march_rays_train(...)  xyzs/dirs/deltas must be zero-filled by the caller;
 * counter is int32[2] (points, rays) and is advanced atomically. */
GF_API int gf_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                               float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                               const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                               int32_t* rays, int32_t* counter, const float* noises, gf_stream_t stream);
/* raymarching.h:15  march_rays_train_backward(...)  accumulates into grad_rays_o/d */
GF_API int gf_march_rays_train_backward(const float* grad_xyzs, const float* grad_dirs, const int32_t* rays,
                                        const float* deltas, uint32_t N, uint32_t M, float* grad_rays_o,
                                        float* grad_rays_d, gf_stream_t stream);
/* raymarching.h:16  composite_rays_train_forward(...) */
GF_API int gf_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* ambient,
                                           const float* deltas, const int32_t* rays, uint32_t M, uint32_t N,
                                           float T_thresh, float* weights_sum, float* ambient_sum, float* depth,
                                           float* image, gf_stream_t stream);
/* raymarching.h:17  composite_rays_train_backward(...) */
GF_API int gf_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_ambient_sum,
                                            const float* grad_image, const float* sigmas, const float* rgbs,
                                            const float* ambient, const float* deltas, const int32_t* rays,
                                            const float* weights_sum, const float* ambient_sum, const float* image,
                                            uint32_t M, uint32_t N, float T_thresh, float* grad_sigmas,
                                            float* grad_rgbs, float* grad_ambient, gf_stream_t stream);
/* raymarching.h:19  march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound, dt_gamma,
 *                              max_steps, C, H, grid, nears, fars, xyzs, dirs, deltas, noises) */
GF_API int gf_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t* rays_alive, const float* rays_t,
                         const float* rays_o, const float* rays_d, float bound, float dt_gamma, uint32_t max_steps,
                         uint32_t C, uint32_t H, const uint8_t* grid, const float* nears, const float* fars,
                         float* xyzs, float* dirs, float* deltas, const float* noises, gf_stream_t stream);
/* raymarching.h:20  composite_rays(n_alive, n_step, T_thresh, rays_alive, rays_t, sigmas, rgbs, deltas,
 *                                  weights_sum, depth, image)   in place on the last five + rays_alive/rays_t */
GF_API int gf_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* rays_alive, float* rays_t,
                             const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                             float* depth, float* image, gf_stream_t stream);

/* ------------------------------------------------------------------------------------
 * _gridencoder   modules/radnerfs/encoders/gridencoder/src/gridencoder.h:11-14
 * dtype: 0 = float32 table/outputs, 1 = float16 table/outputs (autocast path, grid.py:43-44)
 * ---------------------------------------------------------------------------------- */
/* gridencoder.h:11  grid_encode_forward(inputs, embeddings, offsets, outputs, B, D, C, L, S, H, dy_dx,
 *                                       gridtype, align_corners, interp)   outputs [L,B,C]; dy_dx [B,L*D*C] or NULL */
GF_API int gf_grid_encode_forward(const float* inputs, const void* embeddings, const int32_t* offsets, void* outputs,
                                  uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, void* dy_dx,
                                  uint32_t gridtype, int align_corners, uint32_t interp, int dtype,
                                  gf_stream_t stream);
/* gridencoder.h:12  grid_encode_backward(grad, inputs, embeddings, offsets, grad_embeddings, B, D, C, L, S, H,
 *                                        dy_dx, grad_inputs, gridtype, align_corners, interp) */
GF_API int gf_grid_encode_backward(const void* grad, const float* inputs, const void* embeddings,
                                   const int32_t* offsets, void* grad_embeddings, uint32_t B, uint32_t D, uint32_t C,
                                   uint32_t L, float S, uint32_t H, const void* dy_dx, void* grad_inputs,
                                   uint32_t gridtype, int align_corners, uint32_t interp, int dtype,
                                   gf_stream_t stream);
/* gridencoder.h:14  grad_total_variation(inputs, embeddings, grad, offsets, weight, B, D, C, L, S, H,
 *                                        gridtype, align_corners)   float32 only */
GF_API int gf_grad_total_variation(const float* inputs, const float* embeddings, float* grad, const int32_t* offsets,
                                   float weight, uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H,
                                   uint32_t gridtype, int align_corners, gf_stream_t stream);

/* ------------------------------------------------------------------------------------
 * _shencoder   modules/radnerfs/encoders/shencoder/src/shencoder.h:8-9   (float32)
 * ---------------------------------------------------------------------------------- */
GF_API int gf_sh_encode_forward(const float* inputs, float* outputs, uint32_t B, uint32_t D, uint32_t degree,
                                float* dy_dx, gf_stream_t stream);
GF_API int gf_sh_encode_backward(const float* grad, const float* inputs, uint32_t B, uint32_t D, uint32_t degree,
                                 const float* dy_dx, float* grad_inputs, gf_stream_t stream);

/* ------------------------------------------------------------------------------------
 * _freqencoder   modules/radnerfs/encoders/freqencoder/src/freqencoder.h:8-9
 * ---------------------------------------------------------------------------------- */
GF_API int gf_freq_encode_forward(const float* inputs, uint32_t B, uint32_t D, uint32_t degree, uint32_t C,
                                  float* outputs, gf_stream_t stream);
GF_API int gf_freq_encode_backward(const float* grad, const float* outputs, uint32_t B, uint32_t D, uint32_t degree,
                                   uint32_t C, float* grad_inputs, gf_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Vanilla AD-NeRF path (modules/nerfs; SURVEY.md section 8 row a19): the non-GEMM operators.
 * Inference only.  All tensors fp32, contiguous; the caller allocates every output.
 *   gf_adnerf_get_rays       modules/nerfs/commons/ray_samplers.py:11-44 (get_rays) + the viewdirs normalisation of
 *                            volume_rendering.py:251-259; c2w is 3x4 row-major; viewdirs may be NULL
 *   gf_adnerf_embed          modules/nerfs/commons/embedders.py:5-45 (FreqEmbedder.forward), x [n, D] -> out rows of
 *                            D*(1+2*multi_res) floats at stride ld (floats)
 *   gf_adnerf_embed_points   volume_rendering.py:153,183 (pts = o + d z) fused with the position embedding
 *   gf_adnerf_raw2outputs    volume_rendering.py:9-59 (raw [R,S,4] = rgb logits + sigma, raw_noise_std = 0); any output but
 *                            rgb_map may be NULL
 *   gf_adnerf_sample_pdf     volume_rendering.py:62-96 on (z_mid, weights[1:-1]) as called from :177-182, followed by the
 *                            concatenate + sort; u NULL = det (perturb == 0), else [R, N_importance] uniform numbers;
 *                            merge = 1: z_vals / weights are the coarse depths and their weights [R,S], z_out [R, S+N_importance]
 *                            is the sorted union; merge = 0: plain sample_pdf(bins [R,S], weights [R,S-1]) -> z_out [R, N_importance];
 *                            samples_out (optional) the N new depths (for z_std)
 * ---------------------------------------------------------------------------------- */
GF_API int gf_adnerf_get_rays(uint32_t H, uint32_t W, float focal, float cx, float cy, const float* c2w, float* rays_o,
                              float* rays_d, float* viewdirs, gf_stream_t stream);
GF_API int gf_adnerf_embed(const float* x, uint32_t n, uint32_t D, uint32_t multi_res, float* out, uint32_t ld,
                           gf_stream_t stream);
GF_API int gf_adnerf_embed_points(const float* rays_o, const float* rays_d, const float* z_vals, uint32_t R, uint32_t S,
                                  uint32_t multi_res, float* out, uint32_t ld, gf_stream_t stream);
GF_API int gf_adnerf_raw2outputs(const float* raw, const float* z_vals, const float* rays_d, const float* bc_rgb, uint32_t R,
                                 uint32_t S, int white_bkgd, float* rgb_map, float* disp_map, float* acc_map, float* weights,
                                 float* depth_map, float* rgb_map_fg, gf_stream_t stream);
GF_API int gf_adnerf_sample_pdf(const float* z_vals, const float* weights, const float* u, uint32_t R, uint32_t S,
                                uint32_t N_importance, int merge, float* z_out, float* samples_out, gf_stream_t stream);

/* ---- the AD-NeRF backbone on tensor cores (modules/nerfs/adnerf/backbone.py:82-135: NeRFBackbone, num_density_linears = 8,
 *      skip_layer_indices = [4], num_color_linears = 3; weights in torch nn.Linear layout [out, in], row-major, fp32, DEVICE) ------------- */
typedef struct GfAdnerfDesc {
    uint32_t hid;                 /* hid_dim (128 or 256); colour head = hid / 2 */
    uint32_t cond_dim;            /* audio / condition feature size (64) */
    uint32_t pos_multires;        /* frequency bands of the position embedding (10 -> 63 columns) */
    uint32_t view_multires;       /* frequency bands of the view embedding (4 -> 27 columns) */
    const float* dens_w[8];       /* density_linears[i].weight: [hid, 63+cond] (i = 0), [hid, 63+cond+hid] (i = 5), else [hid, hid] */
    const float* dens_b[8];
    const float* dens_out_w;      /* density_out_linear.weight [1, hid] */
    const float* dens_out_b;
    const float* col_w[3];        /* color_linears[i].weight: [hid/2, hid+27] (i = 0), else [hid/2, hid/2] */
    const float* col_b[3];
    const float* col_out_w;       /* color_out_linear.weight [3, hid/2] */
    const float* col_out_b;
} GfAdnerfDesc;
typedef struct GfAdnerfMlp GfAdnerfMlp;

/* Packs the weights into fp16 tensor-core images (copies: the caller's tensors need not outlive the call). */
GF_API int gf_adnerf_mlp_create(const GfAdnerfDesc* desc, GfAdnerfMlp** out, gf_stream_t stream);
GF_API void gf_adnerf_mlp_destroy(GfAdnerfMlp* m);
GF_API uint64_t gf_adnerf_mlp_workspace_bytes(const GfAdnerfMlp* m, uint32_t n_samples);
/* raw[R,S,4] = (rgb logits, sigma) of the network at the points rays_o + rays_d * z_vals[R,S], viewdirs [R,3] (unit), cond [cond_dim]
 * (one frame): volume_rendering.py:153-155 run_network + backbone.py:99-135, embeddings included.  workspace: caller-owned,
 * 1024-byte aligned, gf_adnerf_mlp_workspace_bytes(m, R*S) bytes. */
GF_API int gf_adnerf_mlp_forward(const GfAdnerfMlp* m, const float* rays_o, const float* rays_d, const float* z_vals,
                                 const float* viewdirs, const float* cond, uint32_t R, uint32_t S, float* raw, void* workspace,
                                 uint64_t workspace_bytes, gf_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Tensor-core linear layers of the TRAINING step.  Replace the library GEMMs behind the bias-free MLPs of the field
 * (modules/radnerfs/cond_encoder.py:92-111: nn.Linear(bias=False) + ReLU; called from radnerf.py:73-105 under
 * tasks/radnerfs/radnerf.py:185-216) in forward, data-gradient and weight-gradient form; fp16 operands, fp32 accumulation
 * (= the reference's `amp: true` arithmetic).  Tensors travel as 128-row tiles of 64-column fp16 chunks
 * ([tile][chunk][128 rows x 128 B, 16-byte units XOR-swizzled by row & 7]); gf_tl_tiles_bytes gives the size.
 * ------------------------------------------------------------------------------------ */
GF_API size_t gf_tl_tiles_bytes(uint32_t M, uint32_t chunks);
/* rows [M][ld] (fp32, or fp16 if src_f16; ld = 0: one row broadcast to all samples) columns [0, K) (x *scale if non-NULL, a device scalar) -> columns
 * [col0, col0 + K) of tiles with `chunks` chunks; the rest of [col0, col1) is zero filled (col1 = 0: up to the tile width); col0, col1 % 8 == 0.
 * Calls with adjacent column ranges assemble torch.cat([...], dim=1) inputs (radnerf.py:79,90,99) without materialising them. */
GF_API int gf_tl_pack(const void* src, int src_f16, uint32_t ld, uint32_t K, uint32_t M, uint32_t chunks, uint32_t col0, uint32_t col1,
                      const float* scale, void* tiles, gf_stream_t stream);
/* W [N][K] fp32 (nn.Linear.weight) -> fp16 image of `chunks` blocks [rows_pad x 128 B]; rows_pad % 16 == 0, >= N, <= 256 */
GF_API int gf_tl_weight_image(const float* W, uint32_t N, uint32_t K, uint32_t rows_pad, uint32_t chunks, void* img, gf_stream_t stream);
/* dgrad = 0: D = A W^T (F.linear forward; D has rows_pad columns); dgrad = 1: D = A W (grad_input; D has 64 * w_chunks columns).
 * D (x ReLU mask of the saved activation tiles `mask` if non-NULL) (ReLU if relu) -> fp16 tiles `out` and / or fp32 rows
 * out_f32 [M][ld_f32] columns [0, n_f32) x *out_scale. */
GF_API int gf_tl_gemm(const void* a, uint32_t a_chunks, const void* w_img, uint32_t w_rows, uint32_t w_chunks, int dgrad, uint32_t M, void* out,
                      uint32_t out_chunks, int relu, const void* mask, uint32_t mask_chunks, float* out_f32, uint32_t ld_f32, uint32_t n_f32,
                      const float* out_scale, gf_stream_t stream);
/* grad_weight: dw += *scale * P[:, 64 p_c0 : 64 p_c0 + 128]^T Q[:, 0:N] over the M samples (P, Q tiles); transposed = 0: dw[m * ld + n],
 * 1: dw[n * ld + m]; entries m < rows_m, n < cols_n.  dw (fp32) is accumulated into with reductions: zero it first. */
GF_API int gf_tl_wgrad(const void* p, uint32_t p_chunks, uint32_t p_c0, const void* q, uint32_t q_chunks, uint32_t N, uint32_t M, float* dw,
                       uint32_t ld, uint32_t rows_m, uint32_t cols_n, int transposed, const float* scale, gf_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Fused frame renderer: replaces the eval branch of NeRFRenderer.render()
 * (modules/radnerfs/renderer.py:263-367) and RADNeRFTorso.render()
 * (modules/radnerfs/radnerf_torso.py:86-198) -- ray generation, aabb test, occupancy
 * marching, 3D grid -> ambient MLP -> 2D grid -> sigma MLP -> SH -> colour MLP, alpha
 * compositing, torso layer and background mix -- without the host-driven loop.
 * ---------------------------------------------------------------------------------- */
typedef struct GfModel GfModel;

/* Raw device pointers to the reference's state_dict tensors (SURVEY.md section 8a).  Not retained
 * after gf_model_create returns (weights are repacked into the model's own buffers, and the
 * position and ambient grid tables are copied into padded model-owned images);
 * the torso grid table and the bitfields ARE referenced in place (no copy). */
typedef struct GfModelDesc {
    /* geometry / hyper-parameters */
    float bound;                 /* hparams['bound']                       renderer.py:66 */
    uint32_t cascade;            /* 1 + ceil(log2(bound))                  renderer.py:67 */
    uint32_t grid_size;          /* H, hparams['grid_size']                renderer.py:68 */
    float min_near;              /* renderer.py:71 */
    float aabb[6];               /* aabb_infer                             renderer.py:78-81 */
    uint32_t gridtype;           /* 0 hash, 1 tiled                        grid.py:14-17 */
    uint32_t interp;             /* 0 linear, 1 smoothstep                 grid.py:19-22 */
    uint32_t hidden_dim;         /* 128 (64 also supported)                base.yaml:91-98 */
    uint32_t cond_dim;           /* cond_out_dim = 64 */
    uint32_t ind_dim;            /* individual_embedding_dim (0 or 4) */
    /* head field */
    const uint8_t* density_bitfield;   /* [cascade*H^3/8] */
    const float* pos_embeddings;  const int32_t* pos_offsets;  float pos_S; uint32_t pos_H;   /* 3D grid, L=16,C=2 */
    const float* amb_embeddings;  const int32_t* amb_offsets;  float amb_S; uint32_t amb_H;   /* 2D grid */
    const float* ambient_w0; const float* ambient_w1; const float* ambient_w2;   /* [h,32+cond] [h,h] [2,h] */
    const float* sigma_w0;   const float* sigma_w1;   const float* sigma_w2;     /* [h,64] [h,h] [1+geo,h] */
    const float* color_w0;   const float* color_w1;                              /* [h,16+geo+ind] [3,h] */
    uint32_t geo_feat_dim;       /* 128 */
    const float* ind_code;       /* individual_embeddings[0]  [ind_dim] or NULL */
    /* torso (all NULL/0 for head-only) */
    uint32_t has_torso;
    const float* density_grid_torso;   /* [H*H] */
    float density_thresh_torso;        /* min(density_thresh_torso, mean_density_torso)  radnerf_torso.py:166 */
    float torso_shrink;                /* hparams['torso_shrink'] */
    const float* torso_embeddings; const int32_t* torso_offsets; float torso_S; uint32_t torso_H;
    const float* torso_deform_w0; const float* torso_deform_w1; const float* torso_deform_w2;  /* [64,104] [64,64] [2,64] */
    const float* torso_canon_w0;  const float* torso_canon_w1;  const float* torso_canon_w2;   /* [32,136] [32,32] [4,32] */
    uint32_t torso_ind_dim;            /* 8 */
    const float* torso_ind_code;       /* torso_individual_codes[0] */
} GfModelDesc;

GF_API int gf_model_create(const GfModelDesc* desc, GfModel** out, gf_stream_t stream);
GF_API void gf_model_destroy(GfModel* m);
/* bytes of the packed parameter blob (what rank 0 broadcasts once, SURVEY.md section 8e) */
GF_API uint64_t gf_model_packed_bytes(const GfModel* m);

/* Per-frame inputs.  Either give explicit rays (drop-in for render(rays_o, rays_d, ...)) or
 * set rays_o = rays_d = NULL and give pose + intrinsics (rays are generated in-kernel,
 * utils.py:282-363).  bg_color may be NULL (=> 1.0, renderer.py:354-355). */
typedef struct GfFrame {
    uint32_t H, W;               /* N = H*W rays */
    const float* rays_o;         /* [N,3] or NULL */
    const float* rays_d;         /* [N,3] or NULL */
    float pose[12];              /* c2w rows 0..2 of the 4x4 (used when rays are NULL) */
    float intrinsics[4];         /* fx, fy, cx, cy */
    const float* cond_feat;      /* [cond_dim] device: output of cal_cond_feat (radnerf.py:61-71) */
    const float* bg_color;       /* [N,3] device or NULL */
    const float* bg_coords;      /* [N,2] device or NULL (=> generated, utils.py:273-278) */
    float torso_pose[6];         /* convert_poses(pose)  (utils.py:263-269) */
    float dt_gamma;              /* render(dt_gamma=...) */
    uint32_t max_steps;          /* render(max_steps=...) */
    float T_thresh;              /* 1e-4 default */
    uint32_t precision;          /* 0 = fp32 SIMT (reference arithmetic), 1 = fp16 tensor cores (tcgen05) */
    const float* dyn;            /* NULL, or DEVICE float[22] = pose[12] | intrinsics[4] | torso_pose[6]: the per-frame scalars are then
                                    read from device memory at execution time instead of travelling by value in the launch, so that
                                    ONE captured CUDA graph of gf_render_frame replays for every frame of a sequence (the host
                                    only rewrites these 88 bytes and cond_feat's source) */
} GfFrame;

typedef struct GfOut {
    float* rgb_map;              /* [N,3] clamped composite            renderer.py:357-365 */
    float* depth_map;            /* [N]                                renderer.py:361-364 */
    float* weights_sum;          /* [N] or NULL */
    float* torso_alpha_map;      /* [N] or NULL                        radnerf_torso.py:187 */
    float* torso_rgb_map;        /* [N,3] or NULL                      radnerf_torso.py:188 */
    int32_t* n_samples;          /* [N] per-ray composited sample count or NULL (parity/diagnostics) */
    uint8_t* rgb8;               /* [N,3] uint8 (rgb*255) or NULL      base_nerf_infer.py:97-101 */
    uint64_t* counters;          /* device uint64[4]: samples evaluated, torso pixels, S_total, launches; or NULL */
    uint32_t* term_hist;         /* device uint32[max_steps+1] or NULL: term_hist[k] = number of rays whose termination
                                    slot is k (1..max_steps); replaying renderer.py:326-351 over it yields the reference
                                    host loop's (n_alive, n_step) sequence.  term_hist[0] = S_total. */
    int32_t* term_slot;          /* [N] or NULL: per-ray termination slot (1-based: T < T_thresh at sample j -> j; ran dry after m
                                    samples -> m+1; missed the aabb -> 1), 0 for a ray still alive after the last round.  The
                                    reference marks the ray dead (rays_alive = -1, raymarching.cu:1017) in the host-loop
                                    iteration whose offered slots contain it; a slot > S_total was never observed by that loop. */
} GfOut;

/* get_rays (modules/radnerfs/utils.py:282-363): pixel-centre pinhole rays of B poses (device [B,4,4] c2w) for N flat pixel indices
 * (inds == NULL: N = H*W, every pixel in row-major order).  Outputs caller-allocated: rays_o, rays_d [B,N,3]; i, j [N] or NULL. */
GF_API int gf_get_rays(const float* poses, uint32_t B, float fx, float fy, float cx, float cy, uint32_t H, uint32_t W,
                       const int64_t* inds, uint32_t N, float* rays_o, float* rays_d, float* i, float* j, gf_stream_t stream);

/* Standalone field evaluation = the `self(xyzs, dirs, cond_feat, ind_code)` call inside the reference
 * loop (renderer.py:342 -> radnerf.py:73-105).  xyzs, dirs [M,3]; sigmas [M]; rgbs [M,3]; ambient [M,2] or NULL. */
/* Measurement aid (not on the render path): the field's hash-grid gathers alone -- 16 levels x 8 corners of the 3-D position grid at
 * xyzs [M,3] and 16 x 4 of the 2-D ambient grid at amb_pos [M,2] -- folded into out [M,2]; 1,536 algorithmic bytes per sample. */
GF_API int gf_gather_probe(const GfModel* model, const float* xyzs, const float* amb_pos, uint32_t M, float* out, gf_stream_t stream);

/* rgbs == NULL: density query (NeRFRenderer.density, radnerf.py:107-127): the colour net is skipped, dirs may be NULL.
 * workspace: caller-owned device scratch of gf_field_workspace_bytes(M, precision) bytes, 256-byte aligned. */
GF_API uint64_t gf_field_workspace_bytes(uint32_t M, uint32_t precision);
GF_API int gf_field_forward(const GfModel* model, const float* xyzs, const float* dirs, const float* cond_feat, uint32_t M,
                            float* sigmas, float* rgbs, float* ambient, uint32_t precision, void* workspace,
                            uint64_t workspace_bytes, gf_stream_t stream);

/* Profiling: when enabled, gf_render_frame brackets every field-kernel launch with CUDA events on the launching
 * stream; after synchronising, gf_profile_field_ms returns their summed duration for the last frame. */
GF_API int gf_profile_enable(GfModel* model, int enable);
GF_API int gf_profile_field_ms(GfModel* model, float* total_ms, int* n_launches);

/* Diagnostics for the tcgen05 field kernel: when dbg != NULL the next precision-1 launches dump the fp32
 * accumulators of sample tile 0 after each MMA stage into dbg (device float[9*128*144]). */
GF_API int gf_tc_debug(GfModel* model, float* dbg);

/* workspace the caller owns: gf_render_workspace_bytes(N) bytes of device memory */
GF_API uint64_t gf_render_workspace_bytes(uint32_t N);
GF_API int gf_render_frame(const GfModel* model, const GfFrame* frame, const GfOut* out, void* workspace,
                           uint64_t workspace_bytes, gf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GFRENDER_H_ */
