/*
 * nvsf_b200.h — C-ABI of the B200-native NVSF ray-rendering hot path.
 *
 * This is the drop-in boundary.  Every entry point takes plain device pointers,
 * sizes and a CUDA stream handle (`void*` == cudaStream_t, NULL = legacy default
 * stream) and returns an int status (0 = ok, >0 = cudaError_t of the launch,
 * <0 = NVSF_E_*).  No torch types appear in any signature; the caller allocates
 * every buffer (the reference's ownership rule, raymarching.py:40-41,235-250).
 *
 * Part 1 replaces the ten functions of the reference's pybind module
 * `_raymarching` (reference nvsf/nerf/raymarching/src/bindings.cpp:7-20, C++
 * declarations nvsf/nerf/raymarching/src/raymarching.h:6-96).  Argument order
 * follows raymarching.h; only fp32 is supported ("scalar_t should always be
 * float in use", raymarching.cu:103).
 *
 * Part 2 (nvsf_field_*, nvsf_render_*) replaces the per-sample field
 * evaluation NeRFNetwork.density / .color (network_dynamic.py:213-332) with its
 * tcnn encodings / MLPs and the uniform-sample renderer NeRFRenderer.run
 * (renderer_dynamic.py:109-265).
 */
#ifndef NVSF_B200_H_
#define NVSF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NVSF_OK 0
#define NVSF_E_INVALID (-1)   /* bad argument (null pointer, size, unsupported config) */
#define NVSF_E_WORKSPACE (-2) /* workspace too small */

/* ABI version of this header; bumped on any signature change. */
#define NVSF_B200_ABI_VERSION 14
int nvsf_abi_version(void);
/* Human-readable text for a status returned by any nvsf_* call. */
const char* nvsf_status_string(int status);

/* ------------------------------------------------------------------------- */
/* Part 1 — raymarching operators                                             */
/* ------------------------------------------------------------------------- */

/* replaces near_far_from_aabb (raymarching.h:6-12, kernel raymarching.cu:105-157).
 * rays_o/rays_d [N,3], aabb [6] (device), nears/fars [N]. */
int nvsf_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb,
                            uint32_t N, float min_near, float* nears, float* fars,
                            void* stream);

/* replaces sph_from_ray (raymarching.h:13-17, raymarching.cu:183-217). coords [N,2]. */
int nvsf_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N,
                      float* coords, void* stream);

/* replaces morton3D (raymarching.h:18, raymarching.cu:237-253). coords [N,3] i32 -> indices [N] i32. */
int nvsf_morton3D(const int32_t* coords, uint32_t N, int32_t* indices, void* stream);

/* replaces morton3D_invert (raymarching.h:19-21, raymarching.cu:257-280). */
int nvsf_morton3D_invert(const int32_t* indices, uint32_t N, int32_t* coords, void* stream);

/* replaces packbits (raymarching.h:22-25, raymarching.cu:287-320).
 * grid [N*8] f32 -> bitfield [N] u8, bit i of byte n = grid[8n+i] > density_thresh. */
int nvsf_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield,
                  void* stream);

/* Scratch bytes needed by nvsf_march_rays_train* for N rays. */
size_t nvsf_march_rays_train_workspace_bytes(uint32_t N);

/* replaces march_rays_train (raymarching.h:27-44, kernel raymarching.cu:332-534).
 *
 * Same inputs/outputs as the reference plus a caller-owned scratch buffer.
 * Differences, all inside what the reference leaves unspecified:
 *   - `rays` rows are written in ray-id order and sample offsets are the
 *     exclusive prefix sum of the per-ray counts in that order (the reference's
 *     order comes from atomicAdd and is scheduling dependent, raymarching.cu:445-454);
 *   - `counter` (int32[2]) is accumulated exactly like the reference: offsets
 *     start at counter[0], ray rows at counter[1]; on return
 *     counter[0] += sum(counts), counter[1] += N;
 *   - rays whose slice would end beyond M are dropped (row still written), as in
 *     raymarching.cu:457 — here deterministically the trailing ones.
 * xyzs/dirs [M,3], deltas [M,2] must be zero-filled by the caller where the
 * reference requires zeros (rows not covered by any ray). */
int nvsf_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid,
                          float bound, float dt_gamma, uint32_t max_steps, uint32_t N,
                          uint32_t C, uint32_t H, uint32_t M, const float* nears,
                          const float* fars, float* xyzs, float* dirs, float* deltas,
                          int32_t* rays, int32_t* counter, const float* noises,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Two-phase form of the same operator (lets the host size the sample buffers
 * from counter[0] instead of allocating N*max_steps rows):
 *   phase 1 `_count`: first pass of raymarching.cu:377-439 for every ray, prefix
 *            sum, writes `rays` [N,3] and accumulates `counter`;
 *   phase 2 `_write`: second pass of raymarching.cu:463-533 into xyzs/dirs/deltas
 *            (M rows available).  If zero_tail_end > 0, rows
 *            [min(M, counter[0]), min(M, zero_tail_end)) are zero-filled so the
 *            caller may pass uninitialised buffers. */
int nvsf_march_rays_train_count(const float* rays_o, const float* rays_d, const uint8_t* grid,
                                float bound, float dt_gamma, uint32_t max_steps, uint32_t N,
                                uint32_t C, uint32_t H, const float* nears, const float* fars,
                                int32_t* rays, int32_t* counter, const float* noises,
                                void* workspace, size_t workspace_bytes, void* stream);
int nvsf_march_rays_train_write(const float* rays_o, const float* rays_d, const uint8_t* grid,
                                float bound, float dt_gamma, uint32_t max_steps, uint32_t N,
                                uint32_t C, uint32_t H, uint32_t M, const float* nears,
                                const float* fars, float* xyzs, float* dirs, float* deltas,
                                const int32_t* rays, const int32_t* counter,
                                const float* noises, uint32_t zero_tail_end, void* stream);

/* Phase 2 given the workspace phase 1 (`_count`) filled for the SAME rays: phase 1 keeps (t, dt)
 * of the first 16 samples of every ray there, so rays with <= 16 samples are emitted without a
 * second walk through the occupancy grid and longer rays resume behind their 16th sample.
 * workspace == NULL behaves exactly like nvsf_march_rays_train_write.  Results are bit-identical
 * either way. */
int nvsf_march_rays_train_write_ws(const float* rays_o, const float* rays_d, const uint8_t* grid,
                                   float bound, float dt_gamma, uint32_t max_steps, uint32_t N,
                                   uint32_t C, uint32_t H, uint32_t M, const float* nears,
                                   const float* fars, float* xyzs, float* dirs, float* deltas,
                                   const int32_t* rays, const int32_t* counter,
                                   const float* noises, uint32_t zero_tail_end,
                                   const void* workspace, size_t workspace_bytes, void* stream);

/* replaces composite_rays_train_forward (raymarching.h:45-54, kernel raymarching.cu:578-655). */
int nvsf_composite_rays_train_forward(const float* sigmas, const float* rgbs,
                                      const float* deltas, const int32_t* rays, uint32_t M,
                                      uint32_t N, float T_thresh, float* weights_sum,
                                      float* depth, float* image, void* stream);

/* replaces composite_rays_train_backward (raymarching.h:55-67, kernel raymarching.cu:691-772).
 * grad_sigmas [M], grad_rgbs [M,3] must be zero-filled by the caller (raymarching.py:338-339). */
int nvsf_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image,
                                       const float* sigmas, const float* rgbs,
                                       const float* deltas, const int32_t* rays,
                                       const float* weights_sum, const float* image,
                                       uint32_t M, uint32_t N, float T_thresh,
                                       float* grad_sigmas, float* grad_rgbs, void* stream);

/* replaces march_rays (raymarching.h:69-86, kernel raymarching.cu:809-928).
 * xyzs/dirs [>= n_alive*n_step, 3], deltas [.., 2].  Unlike the reference the
 * kernel writes EVERY slot of rows [0, n_alive*n_step) (zeros where the ray
 * produced no sample) and zero-fills rows [n_alive*n_step, M_padded), so the
 * caller does not have to pre-zero. */
int nvsf_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t* rays_alive,
                    const float* rays_t, const float* rays_o, const float* rays_d, float bound,
                    float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                    const uint8_t* grid, const float* nears, const float* fars, float* xyzs,
                    float* dirs, float* deltas, const float* noises, uint32_t M_padded,
                    void* stream);

/* replaces composite_rays (raymarching.h:87-96, kernel raymarching.cu:967-1053). In place. */
int nvsf_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* rays_alive,
                        float* rays_t, const float* sigmas, const float* rgbs,
                        const float* deltas, float* weights_sum, float* depth, float* image,
                        void* stream);

/* ------------------------------------------------------------------------- */
/* Part 2 — field (encoders + heads) and uniform-sample renderer               */
/* ------------------------------------------------------------------------- */

/* One level of a tcnn-style multiresolution grid (tiny-cuda-nn GridEncoding: scale =
 * exp2(l*log2(per_level_scale))*base-1, res = ceil(scale)+1, size = min(align8(res^D), 2^log2T)
 * entries, offset = first entry of the level, hashed = res^D > size).  Computed on the host. */
#define NVSF_MAX_LEVELS 16
#define NVSF_MAX_PLANE_SCALES 8
typedef struct {
    float scale;
    uint32_t res, size, offset, hashed;
} nvsf_grid_level_t;

/* Architecture of the reference field (network_dynamic.py:13-192, hash_field.py:92-141,
 * flow_field.py:41-103, planes_field.py:142-194).  Fixed by this build (checked, else
 * NVSF_E_INVALID): 4 features per hash level (= the 4 temporal basis functions of HashGridT),
 * 8 features per flow-grid level, 8 features per plane, 64 hidden units, 15 geometry features,
 * sigma net 120->64->16, head nets (87|31)->64->64->(1|3), flow MLP 32->64->64->6. */
typedef struct {
    float bound;              /* scene box [-bound, bound]^3 */
    float density_scale;      /* NeRFRenderer.density_scale */
    uint32_t active_sensor;   /* doubles the exponent (renderer_dynamic.py:187-189) */
    uint32_t num_frames;      /* frame_idx = int(t*(num_frames-1)) */
    uint32_t time_resolution; /* time slices of HashGridT == time rows of the planes */
    uint32_t hs_levels;       /* static 3-D hash grid (HashGrid4D.hash_static), must be 8 */
    uint32_t hs_entries;
    nvsf_grid_level_t hs[NVSF_MAX_LEVELS];
    uint32_t hd_levels;       /* dynamic 2-D hash grids, planes xy / xz / yz, must be 8 */
    uint32_t hd_entries[3];   /* entries per time slice */
    nvsf_grid_level_t hd[3][NVSF_MAX_LEVELS];
    uint32_t fl_levels;       /* flow 3-D hash grid (FlowField.grid_enc), must be 16 */
    uint32_t fl_entries;
    nvsf_grid_level_t fl[NVSF_MAX_LEVELS];
    uint32_t pl_scales;       /* K-planes scales, must be 4 */
    uint32_t pl_res[NVSF_MAX_PLANE_SCALES]; /* spatial resolution per scale */
} nvsf_field_config_t;

/* fp32 master parameters of ONE modality (lidar or camera) in the reference's own layouts
 * (tcnn flat `params`, Planes4D [1,F,H,W] tensors concatenated scale-major then plane-major in
 * itertools.combinations(range(4),2) order, nn.Linear [out,in] weights). */
typedef struct {
    const float* hash_static;  /* hash_encoder_*.hash_static.params */
    const float* hash_dynamic; /* hash_encoder_*.hash_dynamic.{0,1,2}.hash_t.{k}.params, concatenated */
    const float* planes;       /* planes_encoder_*.planes.{s}.{c} */
    const float* flow_grid;    /* flow_net.grid_enc.params */
    const float* flow_mlp;     /* flow_net.mlp.{0,2,4}.weight */
    const float* sigma_net;    /* sigma_net.params */
    const float* head_a;       /* lidar: intensity_net.params ; camera: color_net.params */
    const float* head_b;       /* lidar: raydrop_net.params   ; camera: NULL */
} nvsf_field_params_t;

/* Bytes of the packed-field workspace for this config (device memory, caller-owned). */
size_t nvsf_field_workspace_bytes(const nvsf_field_config_t* cfg);

/* Re-pack the fp32 master parameters into the kernel layouts (fp16 static hash table, channel-
 * last planes, fp16 MLP weights).  Call after every parameter update. lidar != 0 selects the
 * LiDAR heads (Frequency direction encoding, intensity + raydrop nets). */
int nvsf_field_pack_params(const nvsf_field_config_t* cfg, const nvsf_field_params_t* params,
                           uint32_t lidar, void* workspace, size_t workspace_bytes, void* stream);

/* Collapse everything that depends only on the frame time t (device scalar `time`, the [1,1]
 * tensor the reference passes around) into small tables: the time-slice blend + cubic temporal
 * basis of HashGridT (hash_field.py:65-88) and of FlowField.interpT (flow_field.py:105-114), and
 * the time rows of the (x,t),(y,t),(z,t) planes, for the three query times t, (f+1)/F, (f-1)/F
 * of network_dynamic.py:242-271.  Call after nvsf_field_pack_params and whenever t changes. */
int nvsf_field_pack_time(const nvsf_field_config_t* cfg, const nvsf_field_params_t* params,
                         const float* time, void* workspace, size_t workspace_bytes, void* stream);

/* replaces NeRFNetwork.density (network_dynamic.py:213-287) for n points x [n,3] in
 * [-bound,bound]: sigma [n] f32, geo [n,16] f16 (column 0 = raw sigma logit, 1..15 = geo_feat).
 * Optional debug outputs (may be NULL): features [n,128] f16 (the 120 sigma-net inputs in the
 * reference's concat order, network_dynamic.py:276, zero padded) and flow [n,6] f32.
 * scratch (nvsf_field_density_scratch_bytes(n), may be NULL -> fused kernel). */
size_t nvsf_field_density_scratch_bytes(uint32_t n);
int nvsf_field_density(const nvsf_field_config_t* cfg, const void* workspace, const float* x,
                       uint32_t n, float* sigma, void* geo, void* features, float* flow,
                       void* scratch, size_t scratch_bytes, void* stream);

/* replaces NeRFNetwork.color (network_dynamic.py:290-332) for n samples with their own view
 * directions dirs [n,3]: LiDAR = Frequency(12) of (d+1)/2 (72) + geo_feat (15) -> intensity_net,
 * raydrop_net -> sigmoid, columns [raydrop, intensity]; camera = SH(4) (16) + geo_feat -> color_net
 * -> sigmoid, 3 columns.  geo: fp16 matrix [n, geo_ld] whose columns geo_off .. geo_off+14 are
 * geo_feat (the geo16 rows written by nvsf_field_density: geo_ld = 16, geo_off = 1).  mask [n]
 * (bytes, NULL = all): rows with mask == 0 are written as zeros (network_dynamic.py:297-307,327).
 * out f32 [n, out_ld], out_ld in [channels, 4]; extra columns are zero (out_ld = 3 feeds the
 * 3-channel compositors directly for LiDAR).  workspace must be packed for the same modality. */
int nvsf_field_color(const nvsf_field_config_t* cfg, const void* workspace, uint32_t lidar,
                     const float* dirs, const void* geo, uint32_t geo_ld, uint32_t geo_off,
                     const uint8_t* mask, uint32_t n, float* out, uint32_t out_ld, void* stream);

/* Tuning switches.  "density_mode": 2 (default) = staged density evaluation on fp16 table mirrors:
 * flow stage, the 72 time-collapsed 2-D hash tables gathered from shared memory (TMA-staged,
 * k_dyn_stage), gather stage, sigma MLP; 1 = staged on the fp32 collapsed tables without the dyn stage
 * (what the training forward runs); 0 = single fused mma.sync kernel.
 * Mode-2 sub-switches (all default 1): "flow_tc" = flow stage on tcgen05 / TMEM, "fuse_sigma" = gather
 * stage fused with the sigma MLP on tcgen05 (feature rows stay on the SM), "sigma_tc" = stand-alone
 * sigma stage on tcgen05 (when not fused).  "enc_pair" (default 0) = paired static-hash corner loads.
 * "dyn_tile" (samples per work item), "dyn_overhead", "split_chunk" (units of 64 K samples) tune
 * the staged evaluation.  "flow_ts" (default 0) = hidden activations of the flow MLP kept in tensor memory.
 * "heads_tc" = head MLPs of the compositor: 0 mma.sync; 1 tcgen05, four warpgroups, the two LiDAR nets
 * overlapped; 2..5 eight / six / five / seven warpgroups, nets in turn, direction term through a second layer-1
 * MMA; 6 (default) = five warpgroups with the activations as the A operand from tensor memory.
 * Backward: "mlp_bwd_tc" (default 1) = MLP backward on tcgen05 with the weight gradients accumulated in tensor
 * memory, 0 = mma.sync; "enc_bwd_h16" (default 1) = product-rule texels from the fp16 plane mirrors;
 * "enc_bwd_ctas" (2 | 3); "bwd_shift_flow" / "_sigma" / "_heads" = extra binades of the fp16 gradient scale.
 * "march_mode", "composite_mode", "composite_bwd_mode" pick the operator kernel variants (default: per size).
 * In the C ABI these are process-wide switches that the launch code reads on the host at launch time (the
 * defaults are the fastest measured configuration).  The host mirror gives them per-model meaning: a
 * NeRFNetwork carries its own `options` and every one of its entry points (autograd backward included) runs
 * inside `_lib.option_scope(model.options)` — one re-entrant lock around "apply the overrides, enqueue the
 * launches, restore" — so two models / worker threads in one process never see each other's settings.
 * nvsf_get_option returns the current value (NVSF_E_INVALID: unknown name). */
int nvsf_set_option(const char* name, int value);
int nvsf_get_option(const char* name);
int nvsf_density_mode_get(void); /* current "density_mode" */
/* "stage_timing": 1 records CUDA events on the launching stream around the kernels of every
 * chunk of the staged density evaluation; nvsf_stage_timing_read sums them since the last read:
 * ms4 = {flow stage, dyn stage (0 unless density_mode 2), encode (gather) stage, sigma stage} in
 * milliseconds, *launches = chunks. */
int nvsf_stage_timing_read(float* ms4, uint32_t* launches);

/* replaces NeRFRenderer.run (renderer_dynamic.py:109-265) for N rays with S uniform samples.
 * nears/fars [N]; noise [N,S] in [0,1) or NULL (perturb=False); bg_color used for camera only.
 * scratch: nvsf_render_uniform_scratch_bytes(N,S) = N*S*(4+32) bytes (sigma f32 + geo f16[16] per
 * sample) + the staged-density intermediates of one chunk.
 * Outputs: depth [N], image [N,2|3], weights_sum [N]; weights/z_vals [N,S] optional (NULL ok). */
size_t nvsf_render_uniform_scratch_bytes(uint32_t N, uint32_t S);
/* The two phases of nvsf_render_uniform, callable separately (bench.py times them apart):
 * phase 1 evaluates the field for all N*S samples into scratch, phase 2 composites. */
int nvsf_render_uniform_density(const nvsf_field_config_t* cfg, const void* workspace,
                                const float* rays_o, const float* rays_d, const float* nears,
                                const float* fars, const float* noise, uint32_t N, uint32_t S,
                                void* scratch, size_t scratch_bytes, void* stream);
int nvsf_render_uniform_composite(const nvsf_field_config_t* cfg, const void* workspace,
                                  uint32_t lidar, const float* rays_d, const float* nears,
                                  const float* fars, const float* noise, uint32_t N, uint32_t S,
                                  float bg_color, const void* scratch, size_t scratch_bytes,
                                  float* depth, float* image, float* weights_sum, float* weights,
                                  float* z_vals, void* stream);
int nvsf_render_uniform(const nvsf_field_config_t* cfg, const void* workspace, uint32_t lidar,
                        const float* rays_o, const float* rays_d, const float* nears,
                        const float* fars, const float* noise, uint32_t N, uint32_t S,
                        float bg_color, void* scratch, size_t scratch_bytes, float* depth,
                        float* image, float* weights_sum, float* weights, float* z_vals,
                        void* stream);

/* ------------------------------------------------------------------------- */
/* Part 3 — training: forward that keeps its intermediates, and the backward     */
/* ------------------------------------------------------------------------- */

/* fp32 gradient buffers of ONE modality, same layouts and sizes as nvsf_field_params_t.  The
 * backward ACCUMULATES into them (+=); the caller zero-fills (or keeps accumulating, like
 * autograd's .grad).  This is what loss.backward() leaves in the `.grad` of the reference's
 * tcnn `params`, Planes4D parameters and nn.Linear weights (trainer.py:1332). */
typedef struct {
    float* hash_static;
    float* hash_dynamic;
    float* planes;
    float* flow_grid;
    float* flow_mlp;
    float* sigma_net;
    float* head_a; /* lidar: intensity_net ; camera: color_net */
    float* head_b; /* lidar: raydrop_net   ; camera: NULL */
} nvsf_field_grads_t;

/* Bytes of the per-call buffer in which the training forward keeps, per sample: sigma f32,
 * sigma-net output f16[16], flow f32[8], the 120 sigma-net inputs f16[128], the flow-MLP inputs
 * f16[32] and the head colours f32[4]  (444 B per sample), plus the density_mode-2 intermediates of
 * one chunk (84 B per sample). */
size_t nvsf_render_uniform_saved_bytes(uint32_t N, uint32_t S);
/* Bytes of backward scratch (bf16 weight images, time-collapsed gradient tables, per-chunk
 * activation gradients; rays are processed in chunks of ~6 M samples). */
size_t nvsf_render_uniform_backward_scratch_bytes(const nvsf_field_config_t* cfg, uint32_t N,
                                                  uint32_t S);

/* Test/debug aid: byte offsets of the per-sample arrays inside `saved` (sigma, geo, flow, feats,
 * flowfeat, rgbs) and inside the backward scratch (dgeo16 f32[.,16], dfeat f32[.,128], dflow
 * f32[.,8], dflowfeat f32[.,32] of the LAST chunk), then rays per chunk and total scratch bytes:
 * out[12]. */
void nvsf_render_uniform_debug_layout(const nvsf_field_config_t* cfg, uint32_t N, uint32_t S,
                                      size_t* out);

/* NeRFRenderer.run (renderer_dynamic.py:109-265) in training mode: same outputs as
 * nvsf_render_uniform (weights and z_vals are mandatory), intermediates kept in `saved`. */
int nvsf_render_uniform_train_forward(const nvsf_field_config_t* cfg, const void* workspace,
                                      uint32_t lidar, const float* rays_o, const float* rays_d,
                                      const float* nears, const float* fars, const float* noise,
                                      uint32_t N, uint32_t S, float bg_color, void* saved,
                                      size_t saved_bytes, float* depth, float* image,
                                      float* weights_sum, float* weights, float* z_vals,
                                      void* stream);

/* Backward of the above: given dL/d(depth) [N], dL/d(image) [N,2|3], dL/d(weights_sum) [N] and
 * dL/d(weights) [N,S] (each may be NULL = zero), accumulates dL/d(parameters) into `grads`.
 * `workspace` must still hold the tables packed for the forward's time; `params` are the fp32
 * masters (MLP weights are re-packed to bf16); `weights` is the forward's output. */
int nvsf_render_uniform_backward(const nvsf_field_config_t* cfg, const void* workspace,
                                 const nvsf_field_params_t* params, uint32_t lidar,
                                 const float* rays_o, const float* rays_d, const float* nears,
                                 const float* fars, const float* noise, uint32_t N, uint32_t S,
                                 float bg_color, const void* saved, size_t saved_bytes,
                                 const float* weights, const float* g_depth, const float* g_image,
                                 const float* g_weights_sum, const float* g_weights,
                                 const nvsf_field_grads_t* grads, void* scratch,
                                 size_t scratch_bytes, void* stream);

/* NeRFNetwork.flow (network_dynamic.py:197-211 -> FlowField.forward, flow_field.py:116-133) with its
 * backward: what the scene-flow loss of train_step differentiates (trainer.py:237-265:
 * `self.model.flow(pc, time_ego)` -> Chamfer distance of the warped cloud + |flow|.mean()).
 * forward: x [n,3] in [-bound,bound] -> flow [n,8] f32 (forward xyz, backward xyz, 2 unused) and the
 * kept flow-MLP inputs flowfeat [n,32] f16; `workspace` packed for the frame time.
 * backward: dflow [n,8] f32 (columns 6,7 zero) -> accumulates into grads_flow_grid / grads_flow_mlp
 * (layouts of nvsf_field_params_t.flow_grid / .flow_mlp). */
size_t nvsf_field_flow_scratch_bytes(const nvsf_field_config_t* cfg, uint32_t n);
int nvsf_field_flow_forward(const nvsf_field_config_t* cfg, const void* workspace, const float* x,
                            uint32_t n, float* flow, void* flowfeat, void* scratch,
                            size_t scratch_bytes, void* stream);
int nvsf_field_flow_backward(const nvsf_field_config_t* cfg, const void* workspace,
                             const float* flow_mlp, const float* x, uint32_t n,
                             const void* flowfeat, const float* dflow, float* grads_flow_grid,
                             float* grads_flow_mlp, void* scratch, size_t scratch_bytes,
                             void* stream);

/* torch.optim.Adam step as the reference configures it (main_nvsf.py:350-352: betas (0.9, 0.99),
 * eps 1e-15, no weight decay) over one flat fp32 segment of n parameters (16-byte aligned
 * pointers): m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 * with g = grad_scale * grads[i] (1/world_size and the inverse loss scale fold in here).
 * `step` is the 1-based step count t. */
int nvsf_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n,
                   float lr, float beta1, float beta2, float eps, uint32_t step, float grad_scale,
                   void* stream);

/* The same step with the AMP skip decision of `scaler.step(optimizer)` (trainer.py:1332-1334) kept on
 * the device — no host read of found_inf:
 *   nvsf_grad_found_inf:   *found_inf = 1.0f if any of grads[0..n) is inf / nan (the flag only rises; n a
 *                          multiple of 4, 16-byte aligned).  With several ranks the 4-byte flag is
 *                          all-reduced (MAX) so every replica takes the same decision (SURVEY 8e).
 *   nvsf_adam_begin:       state = device float[4] {applied steps t, 1/(1-b1^t), 1/sqrt(1-b2^t), skip}
 *                          (zero-initialised by the caller): advances t unless *found_inf != 0
 *                          (found_inf may be NULL: never skip).
 *   nvsf_adam_step_guarded: nvsf_adam_step over one segment with t / the bias corrections / the skip flag
 *                          read from `state`; a skipped step leaves p, m, v untouched. */
int nvsf_grad_found_inf(const float* grads, size_t n, float* found_inf, void* stream);
int nvsf_adam_begin(float* state, const float* found_inf, float beta1, float beta2, void* stream);
int nvsf_adam_step_guarded(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                           size_t n, float lr, float beta1, float beta2, float eps, const float* state,
                           float grad_scale, void* stream);

/* Exponential moving average of the parameters over one flat fp32 segment, replacing the reference's
 * torch_ema.ExponentialMovingAverage.update() (trainer.py:112-114):
 *   shadow[i] = shadow[i] - (shadow[i] - params[i]) * one_minus_decay
 * with every operation rounded on its own (no FMA), bit-identical to torch_ema's tensor ops.  The caller
 * computes one_minus_decay = float(1 - min(decay, (1 + t) / (10 + t))) for update number t as torch_ema
 * does.  n a multiple of 4, 16-byte aligned pointers. */
int nvsf_ema_update(float* shadow, const float* params, size_t n, float one_minus_decay, void* stream);

/* ------------------------------------------------------------------------- */
/* Part 4 — callers either side of the marcher: ray generation, occupancy grid  */
/* ------------------------------------------------------------------------- */

/* replaces get_lidar_rays (dataset/dataset_utils.py:369-536) for one pose [4,4] (row-major,
 * device): pixel id p = row*W + col from inds [n] (int64, NULL = all pixels 0..n-1 in row-major
 * order), beta = -(col - W/2)/W * fov_hoz/180*pi, alpha = (fov_up - row/H*fov)/180*pi,
 * d = (cos a cos b, cos a sin b, sin a) R^T, o = translation.  rays_o / rays_d [n,3]. */
int nvsf_get_lidar_rays(const float* pose, const int64_t* inds, uint32_t n, uint32_t H, uint32_t W,
                        float fov_up, float fov, float fov_hoz, float* rays_o, float* rays_d,
                        void* stream);

/* replaces get_rays (dataset/dataset_utils.py:539-687): d = normalize((col+0.5-cx)/fx,
 * (row+0.5-cy)/fy, 1) R^T. */
int nvsf_get_rays(const float* pose, const int64_t* inds, uint32_t n, uint32_t H, uint32_t W,
                  float fx, float fy, float cx, float cy, float* rays_o, float* rays_d,
                  void* stream);

/* Occupancy-grid maintenance producing the `density_bitfield` that march_rays_train / march_rays
 * read (raymarching.py:179,379).  The reference ships only morton3D / packbits and no update
 * loop; this follows torch-ngp's update_extra_state, whose raymarching extension the reference
 * carries.  All steps stay on the device.
 *
 * nvsf_grid_cell_points: sample point of every cell, xyz [C*H^3,3] in the grid's own [C][Morton]
 *   order: (2*coords/(H-1) - 1) * (b_c - b_c/H) + (noise*2 - 1) * b_c/H with b_c = min(2^c, bound);
 *   noise [C*H^3,3] in [0,1) or NULL (cell centres).
 * nvsf_grid_accumulate: tmp = sigma*density_scale (first != 0) or max(tmp, sigma*density_scale)
 *   (union over several frame times of a dynamic scene).
 * nvsf_grid_update: grid = max(grid*decay, tmp) where grid >= 0 and tmp >= 0; stats[0] =
 *   mean(clamp(grid, 0)), stats[1] = min(stats[0], density_thresh); bitfield = packbits(grid,
 *   stats[1]).  n = C*H^3 (multiple of 8), workspace nvsf_grid_update_workspace_bytes(n). */
int nvsf_grid_cell_points(uint32_t C, uint32_t H, float bound, const float* noise, float* xyz,
                          void* stream);
/* The same for cells [first, first + count) of the C*H^3 only; noise / xyz rows are relative to the
 * slice.  Multi-GPU update (SURVEY 8e): each rank evaluates one slice of the cells and the ranks
 * all_gather the per-cell sigmas before nvsf_grid_update. */
int nvsf_grid_cell_points_range(uint32_t C, uint32_t H, float bound, const float* noise, uint64_t first,
                                uint64_t count, float* xyz, void* stream);
int nvsf_grid_accumulate(float* tmp_grid, const float* sigma, uint32_t n, float density_scale,
                         uint32_t first, void* stream);
size_t nvsf_grid_update_workspace_bytes(uint32_t n);
int nvsf_grid_update(float* density_grid, const float* tmp_grid, uint32_t n, float decay,
                     float density_thresh, uint8_t* bitfield, float* stats, void* workspace,
                     size_t workspace_bytes, void* stream);

/* Order-preserving compaction out = rays_alive[rays_alive >= 0] of the inference loop around
 * march_rays / composite_rays (composite_rays marks finished rays with -1, raymarching.cu:1049);
 * *n_out (device int32) receives the number kept. */
size_t nvsf_compact_alive_workspace_bytes(uint32_t n);
int nvsf_compact_alive(const int32_t* rays_alive, uint32_t n, int32_t* out, int32_t* n_out,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------- */
/* Part 5 — loss head on the composited outputs (SURVEY 8f rank 3)              */
/* ------------------------------------------------------------------------- */

/* element-wise criteria of main_nvsf.py:205-212 (all reduction="none") */
#define NVSF_LOSS_L1 0       /* torch.nn.L1Loss */
#define NVSF_LOSS_MSE 1      /* torch.nn.MSELoss */
#define NVSF_LOSS_SMOOTHL1 2 /* torch.nn.SmoothL1Loss(beta = param; reference 0.1) */
#define NVSF_LOSS_HUBER 3    /* torch.nn.HuberLoss(delta = param; reference 0.2 * scale) */

typedef struct nvsf_lidar_loss_cfg {
    float alpha_d, alpha_r, alpha_i; /* main_nvsf.py:93-95 (1, 0.01, 0.1) */
    float smooth;                    /* --smooth_factor (main_nvsf.py:76, 0.0) */
    int32_t depth_kind, raydrop_kind, intensity_kind; /* --depth_loss l1, --raydrop_loss mse, --intensity_loss mse */
    float depth_param, raydrop_param, intensity_param; /* beta / delta of smoothl1 / huber */
} nvsf_lidar_loss_cfg_t;

/* replaces the LiDAR supervision of Trainer.train_step (trainer.py:188-219):
 *   m = gt[:,0]; loss[i] = alpha_d * crit_d(depth*m, gt[:,2]*m) + alpha_r * crit_r(image[:,0],
 *   clamp(m, smooth, 1-smooth)) + alpha_i * crit_i(image[:,1]*m, gt[:,1]*m)
 * depth [n] = outputs["depth_lidar"], image [n,2] = outputs["image_lidar"] (raydrop, intensity),
 * gt [n,3] = images_lidar (raydrop mask, intensity, depth).  loss [n] is the per-ray lidar_loss the
 * trainer keeps for its error map; g_depth [n] / g_image [n,2] are d loss[i] / d depth[i], d image[i]
 * (the backward of loss.sum()). */
int nvsf_loss_lidar(const float* depth, const float* image, const float* gt, uint32_t n,
                    const nvsf_lidar_loss_cfg_t* cfg, float* loss, float* g_depth, float* g_image,
                    void* stream);

/* replaces alpha * criterion(pred, gt) with reduction="none" (trainer.py:503 rgb_loss, :514-518
 * rgb_depth_loss on pre-masked inputs): loss [n], g_pred [n] = d loss[i] / d pred[i]. */
int nvsf_loss_elementwise(const float* pred, const float* gt, size_t n, int kind, float param,
                          float alpha, float* loss, float* g_pred, void* stream);

/* Urban-Radiance-Fields line-of-sight loss of train_step (trainer.py:276-296) on the renderer's
 * `weights` [R,T] and `z_vals` [R,T] with gt_depth [R] (= images_lidar[:,:,2] * raydrop mask) and
 * eps = 0.02 * 0.1^min(step/iters, 1):  loss[0] = 0.1 * (sum (mask_empty w)^2 + sum (mask_near w -
 * distr)^2) / #(gt_depth > 0), distr = the normal density of (z - gt_depth) with sigma = eps/3 divided
 * by its maximum over all elements; g_weights [R,T] = d loss / d weights.  workspace: 16 bytes. */
int nvsf_loss_los(const float* weights, const float* z_vals, const float* gt_depth, uint32_t R, uint32_t T,
                  float eps, float* loss, float* g_weights, void* workspace, size_t workspace_bytes,
                  void* stream);

#define NVSF_LOSS_COS 4 /* torch.nn.CosineSimilarity() over the flattened patch (--depth_grad_loss cos) */

/* options of the structural regularisation (main_nvsf.py:86,90,100-107; trainer.py:297-462) */
typedef struct nvsf_patch_loss_cfg {
    float scale;                                          /* opt.scale */
    int32_t sobel, grad_norm_smooth, spatial_smooth, tv_loss, grad_loss;  /* flags */
    float alpha_grad_norm, alpha_spatial, alpha_tv, alpha_grad;
    int32_t grad_kind;                                    /* --depth_grad_loss: NVSF_LOSS_* */
    float grad_param;
} nvsf_patch_loss_cfg_t;

/* ground-truth side of the gradient loss (trainer.py:392-428): from the range image pano_depth [H,W]
 * (data['pano_frame'][0,...,2]) and the pixel ids rays_pano_inds [P*h*w] (int64) of P patches of h x w
 * rays: mask_x / mask_y [P,h,w] = |second difference of the range image| < thresh (0.05). */
int nvsf_patch_grad_masks(const float* pano_depth, uint32_t H, uint32_t W, const int64_t* rays_pano_inds,
                          uint32_t P, uint32_t h, uint32_t w, float scale, float thresh, float* mask_x,
                          float* mask_y, void* stream);

/* structural regularisation of P depth patches of h x w rays (trainer.py:306-462): pred_depth [P,h,w]
 * (= depth_lidar * raydrop mask), and for the gradient loss gt_depth, gt_raydrop, mask_x, mask_y
 * [P,h,w].  Forward pass (g_pred NULL): loss_map [P,h,w] = the element-wise terms (grad_norm / spatial
 * / tv), grad_loss [P] = each patch's share of `grad_loss.sum()`.  Backward pass (g_pred given; loss_map /
 * grad_loss may be NULL): g_pred [P,h,w] = sum_i g_map[i] d loss_map[i] / d pred + sum_p g_grad[p]
 * d grad_loss[p] / d pred for the incoming gradients g_map [P,h,w] / g_grad [P] (NULL = zero). */
int nvsf_loss_patch(const float* pred_depth, const float* gt_depth, const float* gt_raydrop, const float* mask_x,
                    const float* mask_y, uint32_t P, uint32_t h, uint32_t w, const nvsf_patch_loss_cfg_t* cfg,
                    float* loss_map, float* grad_loss, const float* g_map, const float* g_grad, float* g_pred,
                    void* stream);

/* replaces the reference's Chamfer extension (nvsf/nerf/chamfer3D/chamfer3D.cu; pybind
 * chamfer_cuda.cpp `forward` / `backward`; wrapper dist_chamfer_3D.py:42-95), called by train_step
 * on predicted vs ground-truth LiDAR points (trainer.py:229-233) and on flow-warped clouds
 * (:246-265).  xyz1 [b,n,3], xyz2 [b,m,3]; dist1 [b,n] / idx1 [b,n] = squared distance to and index
 * of the nearest point of xyz2 (first minimum, bit-identical to the reference kernel), dist2 / idx2
 * the other direction.  Backward ACCUMULATES into grad_xyz1 / grad_xyz2 (the reference wrapper
 * zero-fills them, dist_chamfer_3D.py:76-80); either may be NULL. */
size_t nvsf_chamfer_workspace_bytes(uint32_t b, uint32_t n, uint32_t m);
int nvsf_chamfer_forward(const float* xyz1, const float* xyz2, uint32_t b, uint32_t n, uint32_t m,
                         float* dist1, float* dist2, int32_t* idx1, int32_t* idx2, void* workspace,
                         size_t workspace_bytes, void* stream);
int nvsf_chamfer_backward(const float* xyz1, const float* xyz2, uint32_t b, uint32_t n, uint32_t m,
                          const float* grad_dist1, const float* grad_dist2, const int32_t* idx1,
                          const int32_t* idx2, float* grad_xyz1, float* grad_xyz2, void* stream);

/* ------------------------------------------------------------------------- */
/* Part 6 — evaluation of rendered frames                                     */
/* ------------------------------------------------------------------------- */
/* Replaces the host-side scoring of Trainer.evaluate_one_epoch / test_step (trainer.py:817-903,
 * 1458-1846): the meters of nvsf/lib/error_matrices.py and the range image -> point cloud conversion of
 * nvsf/lib/convert.py.  Metric definitions: DESIGN.md §3.5.  Reductions run in a fixed order, so the same
 * inputs give a bit-identical result; nothing is read back to the host. */

/* Chamfer forward with the cloud sizes in device memory: xyz1 [cap_n,3], xyz2 [cap_m,3] hold *n / *m
 * (device int32, clamped to [0, capacity]) points followed by padding.  dist / idx of the first *n / *m rows
 * are bit-identical to nvsf_chamfer_forward on the trimmed clouds (same arithmetic, same first minimum); rows
 * past a count get 0 / -1, and every query gets +inf / -1 when the other cloud is empty.  workspace:
 * nvsf_chamfer_workspace_bytes(1, cap_n, cap_m). */
int nvsf_chamfer_forward_counted(const float* xyz1, const float* xyz2, uint32_t cap_n, uint32_t cap_m,
                                 const int32_t* n, const int32_t* m, float* dist1, float* dist2, int32_t* idx1,
                                 int32_t* idx2, void* workspace, size_t workspace_bytes, void* stream);

/* Range image -> point cloud (convert.py): for every pixel p = j*W + i of depth [H,W] whose masked depth
 * depth * (raydrop > raydrop_threshold) is non-zero (raydrop [H,W] may be NULL: no mask), the row
 * lidar_dir(i, j) * (masked depth / scale), with lidar_dir the direction of nvsf_get_lidar_rays at the
 * identity pose; plus intensity[p] as a 4th column when intensity [H,W] is given.  points [H*W, 3 or 4]: kept
 * pixels in row-major order, then zero rows; *count (device int32) = number kept.  Order-preserving prefix sums,
 * no atomics.  H*W <= 2^26. */
size_t nvsf_lidar_points_workspace_bytes(uint32_t H, uint32_t W);
int nvsf_lidar_points(const float* depth, const float* raydrop, float raydrop_threshold, const float* intensity,
                      uint32_t H, uint32_t W, float fov_up, float fov, float fov_hoz, float scale, float* points,
                      int32_t* count, void* workspace, size_t workspace_bytes, void* stream);

/* One LiDAR frame's metric row (NVSF_EVAL_LIDAR_K floats, column order below).  depth [H,W] and image [H,W,2]
 * (raydrop probability, intensity) are render_frame's outputs; gt [H,W,3] = (raydrop mask, intensity, depth)
 * as for nvsf_loss_lidar.  workspace (16-byte aligned): nvsf_eval_lidar_workspace_bytes(H, W). */
#define NVSF_EVAL_LIDAR_K 15
#define NVSF_EVAL_DEPTH_RMSE 0
#define NVSF_EVAL_DEPTH_MEDAE 1
#define NVSF_EVAL_DEPTH_PSNR 2
#define NVSF_EVAL_DEPTH_SSIM 3
#define NVSF_EVAL_INTENSITY_RMSE 4
#define NVSF_EVAL_INTENSITY_MEDAE 5
#define NVSF_EVAL_INTENSITY_PSNR 6
#define NVSF_EVAL_INTENSITY_SSIM 7
#define NVSF_EVAL_RAYDROP_RMSE 8
#define NVSF_EVAL_RAYDROP_ACC 9
#define NVSF_EVAL_RAYDROP_F1 10
#define NVSF_EVAL_CHAMFER 11
#define NVSF_EVAL_FSCORE 12
#define NVSF_EVAL_POINTS_PRED 13
#define NVSF_EVAL_POINTS_GT 14
size_t nvsf_eval_lidar_workspace_bytes(uint32_t H, uint32_t W);
int nvsf_eval_lidar(const float* depth, const float* image, const float* gt, uint32_t H, uint32_t W, float fov_up,
                    float fov, float fov_hoz, float scale, float max_depth, float fscore_threshold, float* row,
                    void* workspace, size_t workspace_bytes, void* stream);

/* One camera frame's row (PSNR, SSIM) of pred / gt [H,W,3] in [0,1]: PSNR = -10 log10(MSE), SSIM = mean of
 * the per-channel SSIMs with data range 1.  workspace (16-byte aligned): nvsf_eval_camera_workspace_bytes. */
#define NVSF_EVAL_CAMERA_K 2
size_t nvsf_eval_camera_workspace_bytes(uint32_t H, uint32_t W);
int nvsf_eval_camera(const float* pred, const float* gt, uint32_t H, uint32_t W, float* row, void* workspace,
                     size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NVSF_B200_H_ */
