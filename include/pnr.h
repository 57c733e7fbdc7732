/* pnr.h — C ABI of libpnr (PanopticNeRF render hot path, sm_100a).
 *
 * The reference exposes this path only as a Python plugin surface in lib/networks
 * (make_network, Renderer.render, batchify_rays, raw2outputs, sample_pdf; SURVEY.md 8(b)); it has
 * no native/FFI boundary of its own, and its source is not in the mount (/root/reference holds the
 * landing branch only: README.md:7, README.md:13), so no reference file:line can be cited per entry
 * point.  Each entry point below names the SURVEY.md 8(a) row (a1..a10) it implements; the
 * reference-side binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every function returns 0 on success, <0 on error; pnr_last_error() gives a thread-local text.
 *  - all array arguments are DEVICE pointers unless the name ends in _host.
 *  - buffers are caller-owned; nothing is allocated on the stage entry points; all work is
 *    enqueued asynchronously on `stream` (a cudaStream_t passed as void*).
 *  - a context belongs to one device (cfg.device); every entry point that takes a context makes that
 *    device current for the call and restores the caller's current device before it returns; the
 *    context-free stage entry points run on the caller's current device (the one their pointers and
 *    stream belong to).  Several contexts, devices and streams may be used from one process; a single
 *    context is not thread-safe.  Outputs are deterministic (no atomics on outputs), so any ray
 *    sharding reproduces the single-GPU result bit for bit.
 */
#ifndef PNR_H_
#define PNR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PNR_VERSION 100

enum { PNR_OK = 0, PNR_ERR_ARG = -1, PNR_ERR_CUDA = -2, PNR_ERR_STATE = -3, PNR_ERR_UNSUPPORTED = -4 };

/* MLP arithmetic mode: element format of the tensor-core operands (accumulation is always fp32).
 * The x3 modes split every operand x = hi + lo in that format and issue A_hi*B_hi + A_lo*B_hi + A_hi*B_lo. */
enum { PNR_PREC_BF16X3 = 0, /* ~2^-17 per product, fp32 exponent range; ~1e-4 end to end (marginal)       */
       PNR_PREC_BF16 = 1,   /* 1 pass, ~1e-2 end to end: fast mode, outside the tolerance                 */
       PNR_PREC_FP16X3 = 2, /* ~2^-21 per product, needs |activation| < 65504; meets 1e-4 with margin     */
       PNR_PREC_FP16 = 3    /* 1 pass, ~1e-3 end to end: fast mode, outside the tolerance                 */ };

typedef struct pnr_ctx pnr_ctx;

typedef struct pnr_config {
  int32_t D;             /* trunk depth (8)                           a8 */
  int32_t W;             /* trunk width (256); 64, 128 or 256         a8 */
  int32_t xyz_res;       /* Lx, positional-encoding octaves for xyz   a7 */
  int32_t view_res;      /* Ld, octaves for the view direction        a7 */
  int32_t num_classes;   /* C semantic logits, 0 = no head            a8 */
  int32_t num_instances; /* K instance logits, 0 = no head            a8 */
  int32_t precision;     /* PNR_PREC_*                                   */
  int32_t device;        /* CUDA ordinal                                 */
} pnr_config;

int pnr_version(void);
const char* pnr_last_error(void);

/* a1/a2: context = packed weights + kernel attributes for one Network on one device. */
int pnr_create(const pnr_config* cfg, pnr_ctx** out);
int pnr_destroy(pnr_ctx* ctx);

/* a8 range check: sticky status of the fused-MLP launches enqueued so far on `stream` (synchronises it).
 * bit 0 (PNR_STATUS_RANGE): an activation left the range of the 16-bit operand format (fp16 modes: |x| > 65504)
 * or was not finite - the outputs of that launch are not trustworthy, re-run with PNR_PREC_BF16X3.
 * reset != 0 clears the word after reading it. */
#define PNR_STATUS_RANGE 1u
int pnr_status(pnr_ctx* ctx, uint32_t* status_host, int32_t reset, void* stream);

/* a2: load a Network state_dict.  `tensors_host[i]` are HOST fp32 pointers in this fixed order:
 *   pts_linears.{0..D-1}.weight/.bias (interleaved w,b), alpha_linear.w/.b, feature_linear.w/.b,
 *   views_linears.0.w/.b, rgb_linear.w/.b, [semantic_linears.0.w/.b, semantic_linears.1.w/.b],
 *   [instance_linears.0.w/.b, instance_linears.1.w/.b]
 * `shapes[2*i], shapes[2*i+1]` = (out, in) for weights, (out, 1) for biases.  Weights are split
 * into 16-bit hi/lo parts of the context's operand format (fp16 or bf16, cfg.precision), laid out as
 * no-swizzle K-major UMMA stage images and uploaded.  In the fp16 modes a weight with |w| > 65504 is
 * rejected (PNR_ERR_UNSUPPORTED): use a bf16 mode. */
int pnr_load_weights(pnr_ctx* ctx, const float* const* tensors_host, const int64_t* shapes, int32_t n);

/* a5: ray / oriented-box slab test.  rays [R,6] (o||d); box_center, box_half [B,3]; box_rot [B,3,3]
 * row-major, columns = box axes.  Out: hit_mask [R] u8, box_id [R,M] i32 (-1 pad), t_in/t_out [R,M]. */
int pnr_intersect(const float* rays, int64_t R, const float* box_center, const float* box_half,
                  const float* box_rot, int32_t B, int32_t M, uint8_t* hit_mask, int32_t* box_id,
                  float* t_in, float* t_out, void* stream);

/* a5 (AABB special case): per-ray near = max(tmin, near_min), far = tmax, or
 * (near_min, far_default) when the scene box is missed.  aabb_host = {lo.xyz, hi.xyz}. */
int pnr_scene_near_far(const float* rays, int64_t R, const float* aabb_host, float near_min,
                       float far_default, float* near, float* far, void* stream);

/* a5 helper (cfg.bound_by_primitives): clamp near/far to the hull of the hit intervals, in place. */
int pnr_bound_by_primitives(const uint8_t* hit_mask, const int32_t* box_id, const float* t_in,
                            const float* t_out, int64_t R, int32_t M, float* near, float* far,
                            void* stream);

/* a6: z[R,N] = near*(1-t)+far*t (t_vals [N]); if perturb>0, jittered with u [R,N].
 * sample_box (nullable) [R,N] i32 = id of the first hit interval containing the sample, else -1. */
int pnr_sample_stratified(const float* near, const float* far, const float* t_vals, const float* u,
                          int64_t R, int32_t N, float perturb, const int32_t* box_id,
                          const float* t_in, const float* t_out, int32_t M, float* z,
                          int32_t* sample_box, void* stream);

/* a6, interval mode: the N samples are placed inside the ray's hit intervals (clipped to [near, far]):
 * n_m = floor(N * len_m / sum len) samples for interval m, the remainder one by one to the nearest intervals,
 * sample j of an interval at a + (b-a)*(j+0.5)/n_m (or (j+u)/n_m when perturb > 0, u [R,N] per allocation slot),
 * the depths sorted ascending; rays without a hit interval fall back to the uniform rule of pnr_sample_stratified.
 * Same arguments as pnr_sample_stratified (box_id/t_in/t_out required).  The reference's own allocation rule is
 * not in the mount (SURVEY 8(c) question 4): this one is chosen here and documented in DESIGN.md. */
int pnr_sample_intervals(const float* near, const float* far, const float* t_vals, const float* u,
                         int64_t R, int32_t N, float perturb, const int32_t* box_id,
                         const float* t_in, const float* t_out, int32_t M, float* z,
                         int32_t* sample_box, void* stream);

/* a6: re-tag an existing depth array (after the coarse+fine merge). */
int pnr_tag_samples(const float* z, int64_t R, int32_t N, const int32_t* box_id, const float* t_in,
                    const float* t_out, int32_t M, int32_t* sample_box, void* stream);

/* 8(f) rank 3 (the step before the path): camera rays for image rows [row0, row0+rows) of an H x W image,
 * rays [rows*W, 6] = origin || unnormalised direction, row-major over (v, u).
 * camera 0 = pinhole: d_cam = ((u-cx)/fx, (v-cy)/fy, 1); camera 1 = equirectangular:
 * lon = (u/W-0.5)*2pi, lat = (0.5-v/H)*pi, d_cam = (cos lat sin lon, -sin lat, cos lat cos lon).
 * camera 2 = KITTI-360 fisheye (unified / MEI model), intr_host = {gamma1, gamma2, u0, v0, xi, k1, k2}: the pixel's
 * distorted normalised point is undistorted radially (rd = ro (1 + k1 ro^2 + k2 ro^4), 8 Newton steps from ro = rd)
 * and lifted to the unit sphere, d_cam = (f x, f y, f - xi), f = (xi + sqrt(1 + (1 - xi^2) r^2)) / (1 + r^2).
 * intr_host = {fx, fy, cx, cy} otherwise; c2w_host = row-major 3x4 [R|t]: d = R d_cam, o = t. */
int pnr_generate_rays(int32_t H, int32_t W, int32_t row0, int32_t rows, int32_t camera, const float* intr_host,
                      const float* c2w_host, float* rays, void* stream);

/* a7: standalone positional encoding, out [n, 3+6L]. */
int pnr_encode(const float* x, int64_t n, int32_t L, float* out, void* stream);

/* a8: Network.forward.  Either (pts, viewdirs) [n,3] each, or (rays [R,6], z [R,N]) with pts and the
 * normalised view direction formed in-kernel (pass pts = NULL).  raw [n or R*N, 4+C+K]. */
int pnr_mlp_forward(pnr_ctx* ctx, const float* pts, const float* viewdirs, const float* rays,
                    const float* z, int64_t R, int32_t N, float* raw, void* stream);

/* Development aid: as pnr_mlp_forward(rays, z) but block 0 also records a clock64 timeline of its third
 * tile into timeline[8192] (i64, device): [3*stage+{0,1,2}] MMA issuer (arrive / ready / issued),
 * [4096 + 3*(2*step+half)+{0,1,2}] epilogue (wait / accumulator ready / done), [6144 + stage] TMA issue. */
int pnr_mlp_forward_timeline(pnr_ctx* ctx, const float* rays, const float* z, int64_t R, int32_t N,
                             float* raw, int64_t* timeline, void* stream);
/* Development aid: the pnr_mlp_composite and pnr_mlp_backward_trunk launches of `ctx` record the same timeline into timeline[8192] (device i64)
 * until this is called again with NULL (-DPNR_TIMELINE builds only; ignored otherwise). */
int pnr_debug_timeline(pnr_ctx* ctx, int64_t* timeline);

/* a9: raw2outputs.  raw [R,N,4+C+K], z [R,N], rays [R,6].  Any output pointer may be NULL.
 * sem_softmax: composite softmax(logits) instead of logits.  sample_box/box_sem/box_inst nullable. */
typedef struct pnr_composite_out {
  float* rgb_map;    /* [R,3] */
  float* depth_map;  /* [R]   */
  float* acc_map;    /* [R]   */
  float* disp_map;   /* [R]   */
  float* weights;    /* [R,N] */
  float* semantic_map;        /* [R,C] */
  float* instance_map;        /* [R,K] */
  float* fixed_semantic_map;  /* [R,C] */
  float* fixed_instance_map;  /* [R,K] */
} pnr_composite_out;
int pnr_composite(const float* raw, const float* z, const float* rays, int64_t R, int32_t N,
                  int32_t C, int32_t K, int32_t white_bkgd, int32_t sem_softmax, int32_t mask_outside,
                  const int32_t* sample_box, const int32_t* box_sem, const int32_t* box_inst,
                  int32_t B, const pnr_composite_out* out, void* stream);

/* 8(e) label tiles / 8(f) rank 4 (panoptic label fusion): what a rank contributes to the all-gather when labels,
 * not logits, are wanted - rgb8 [R,3] u8 = round(255*clamp(rgb)), depth_out [R] f32, sem_label / inst_label [R] i16 =
 * argmax of the composited semantic / instance maps (ties -> lowest index, NaN counts as -inf).
 * 13 bytes per ray instead of 4*(5+C+K).  Any output pointer may be NULL. */
int pnr_label_tiles(const float* rgb_map, const float* depth_map, const float* semantic_map,
                    const float* instance_map, int64_t R, int32_t C, int32_t K, uint8_t* rgb8,
                    float* depth_out, int16_t* sem_label, int16_t* inst_label, void* stream);

/* 8(f) rank 2, the loss side: the per-ray terms of the training objective on the rendered maps and their gradients
 * w.r.t. those maps, in one pass (inputs any subset; NULL skips a term / an output):
 *   photometric  sum_c (rgb_map - rgb_gt)^2  (+ the same for the coarse map rgb_map0)
 *   depth        |depth_map - depth_gt| where depth_gt > 0
 *   semantic     label >= 0: cross-entropy of semantic_map [R,C] against label - softmax CE when the map holds rendered
 *                logits (sem_is_prob = 0), -log(max(p_label, eps)) when it holds rendered probabilities - times
 *                label_weight[r] (optional confidence)
 *   fixed        -log(max(fixed_semantic_map[label], eps)) * label_weight
 * per_ray [R,4] receives the four unweighted values; the caller sums them.  Every gradient is already multiplied by
 * the term's weight w_* and normaliser inv_n_* (1 / number of elements or valid rays, which the caller knows), i.e.
 * it is dL/dmap of L = w_rgb*mean_rgb + w_depth*mean_depth + w_sem*mean_sem + w_fix*mean_fix, ready for
 * pnr_composite_backward.  (Terms as in the paper; the reference's NetworkWrapper is not in the mount.) */
typedef struct pnr_loss_args {
  int64_t R; int32_t C; int32_t sem_is_prob;
  const float* rgb_map; const float* rgb_map0; const float* rgb_gt;
  const float* depth_map; const float* depth_gt;
  const float* semantic_map; const float* fixed_semantic_map; const int32_t* label; const float* label_weight;
  float w_rgb, w_depth, w_sem, w_fix;
  float inv_n_rgb, inv_n_depth, inv_n_sem;
  float eps;
  float* per_ray;
  float* d_rgb_map; float* d_rgb_map0; float* d_depth_map; float* d_semantic_map; float* d_fixed_semantic_map;
} pnr_loss_args;
int pnr_losses(const pnr_loss_args* args, void* stream);

/* 8(f) rank 4: panoptic label fusion + colour mapping of the composited maps (the step after the path).
 * s = argmax semantic_map [R,C] (ties -> lowest index, NaN = -inf).  A stuff class (is_thing[s] == 0, or no instance
 * map) gives id(s)*1000 with id(s) = class_id[s] (or s when class_id is NULL).  A thing class takes the best instance
 * slot among the slots k with inst_class[k] == s: panoptic = inst_id[k] (or id(s)*1000 + k + 1 when inst_id is NULL);
 * without such a slot it falls back to id(s)*1000.  color [R,3] u8: palette[s], for instances averaged with a colour
 * hashed from the panoptic id.  Outputs are optional.  (Rule chosen here; the reference's is not in the mount.) */
int pnr_panoptic_fuse(const float* semantic_map, const float* instance_map, int64_t R, int32_t C, int32_t K,
                      const uint8_t* is_thing, const int32_t* inst_class, const int32_t* inst_id,
                      const int32_t* class_id, const uint8_t* palette, int32_t* panoptic, int16_t* sem_label,
                      int16_t* inst_slot, uint8_t* color, void* stream);

/* 8(f) rank 4: multi-resolution hash-grid features (the 360 model's extra encoder; published algorithm of
 * Mueller et al. 2022): level l has resolution floor(base_resolution * per_level_scale^l) (double, on the host);
 * x [n,3] is mapped to [0,1]^3 by aabb (DEVICE {lo.xyz, hi.xyz}; NULL: already normalised) and clamped; the 8 corners
 * of its cell are read from table [L, 2^T_log2, F] fp32 - dense index x + y*(res+1) + z*(res+1)^2 while the level fits,
 * else (x*1) ^ (y*2654435761) ^ (z*805459861) mod 2^T_log2 - and blended trilinearly (corner order x fastest).
 * out [n, L*F], level-major.  F in {1,2,4,8}. */
int pnr_hashgrid_encode(const float* x, int64_t n, const float* aabb, const float* table, int32_t L, int32_t F,
                        int32_t T_log2, float base_resolution, float per_level_scale, float* out, void* stream);

/* Gradient of pnr_hashgrid_encode w.r.t. its table: grad_table [L, 2^T_log2, F] += scatter of grad_out [n, L*F] with the
 * forward's corner weights (fp32 atomic adds: ACCUMULATES - zero grad_table first; the summation order, hence the last
 * bits, vary between runs).  Same arguments as the forward. */
int pnr_hashgrid_backward(const float* x, int64_t n, const float* aabb, const float* grad_out, int32_t L, int32_t F,
                          int32_t T_log2, float base_resolution, float per_level_scale, float* grad_table, void* stream);

/* a8 + a9 in ONE kernel: Network.forward with the compositing done in the MLP's epilogue - per-sample alpha /
 * transmittance / weight right after the sigma-producing layer, colours and logits reduced on chip per ray - so the
 * network outputs `raw` [R,N,4+C+K] (456 B per sample with both heads) are never written to memory; only
 * out->weights [R,N] (REQUIRED) and the per-ray maps leave the SM.  Same maps as pnr_mlp_forward + pnr_composite
 * (weights bit-identical, sums in a different but fixed order); fixed_* maps come from the weights and the id
 * tables (a small second kernel).  Needs N % 32 == 0 and rays mode; sem_softmax is not available here
 * (PNR_ERR_UNSUPPORTED: use the two-call path). */
int pnr_mlp_composite(pnr_ctx* ctx, const float* rays, const float* z, int64_t R, int32_t N,
                      int32_t white_bkgd, int32_t mask_outside, const int32_t* sample_box,
                      const int32_t* box_sem, const int32_t* box_inst, int32_t B,
                      const pnr_composite_out* out, void* stream);

/* a9 backward (SURVEY 8(f) rank 2, first stage of the backward chain): d(loss)/d(raw) [R,N,4+C+K] from the
 * gradients of the composited maps (any pointer may be NULL = zero gradient; disp_map is not differentiated).
 * Same arguments as pnr_composite.  sem_softmax != 0 returns PNR_ERR_UNSUPPORTED. */
typedef struct pnr_composite_grads {
  const float* rgb_map;    /* [R,3] */
  const float* depth_map;  /* [R]   */
  const float* acc_map;    /* [R]   */
  const float* weights;    /* [R,N] */
  const float* semantic_map;        /* [R,C] */
  const float* instance_map;        /* [R,K] */
  const float* fixed_semantic_map;  /* [R,C] */
  const float* fixed_instance_map;  /* [R,K] */
} pnr_composite_grads;
int pnr_composite_backward(const float* raw, const float* z, const float* rays, int64_t R, int32_t N,
                           int32_t C, int32_t K, int32_t white_bkgd, int32_t sem_softmax, int32_t mask_outside,
                           const int32_t* sample_box, const int32_t* box_sem, const int32_t* box_inst,
                           int32_t B, const pnr_composite_grads* g, float* d_raw, void* stream);

/* a8 backward, first slice (SURVEY 8(f) rank 2; replaces autograd through Network.forward's trunk - the D
 * `pts_linears` with their ReLUs and the skip concatenation): dL/d(embedded xyz) (the first 3 + 6*xyz_res columns
 * of grad_emb [R*N, ld_emb]; ld_emb = 64 on a 16-byte aligned base lets the kernel use 16-byte stores) from
 * grad_h = dL/dh of the trunk output [R*N, W].  One kernel on the same 128-sample tiles as pnr_mlp_forward: the
 * forward trunk is recomputed (ReLU sign patterns stay in shared memory), then the layers run in reverse with the
 * transposed weight stream on the tensor cores, gradients split hi/lo like activations.  Samples are given as pts
 * [R*N,3] or as (rays [R,6], z [R,N]).  x3 precisions only; D <= 9.  grad_scale: a power of two applied to grad_h on
 * load and removed from everything the kernel writes (exact): pick it so that max |grad_h| * grad_scale is a few
 * hundred, or the fp16 operand parts of small gradients go subnormal (1.0 when grad_h is already O(1)). */
int pnr_mlp_backward_trunk(pnr_ctx* ctx, const float* pts, const float* rays, const float* z, int64_t R, int32_t N,
                           const float* grad_h, float grad_scale, float* grad_emb, int32_t ld_emb, float* stash,
                           uint32_t* stash_absmax, void* stream);
/* The weight gradients of the trunk come from `stash` [2D-1, R*N, W] fp32 (NULL: not kept): every A operand the
 * kernel produces on the way - slot i < D-1: H_i, the activations of forward layer i; slot 2D-2-j: dZ_j, the gradient
 * w.r.t. layer j's pre-activation - so that dW_j = dZ_j^T [H_{j-1} (, gamma(x))], db_j = sum_s dZ_j are GEMMs over
 * the samples: pnr_wgrad.  pnr_mlp_trunk_forward returns the trunk's output h [R*N, W] (16-byte
 * aligned), the input of the layers after the trunk (alpha / feature / view / rgb / heads), which the caller
 * differentiates itself to obtain grad_h.
 * stash_absmax (nullable; needs stash) [2D-1] u32, zeroed by the call: slot k receives the largest magnitude written
 * to stash slot k, as the bit pattern of its 16-bit hi part in the context's operand format (fp16 / bf16) and for
 * the gradient slots BEFORE the division by grad_scale - enough to pick pnr_wgrad's power-of-two dz_scale without
 * another pass over the stash. */
int pnr_mlp_trunk_forward(pnr_ctx* ctx, const float* pts, const float* rays, const float* z, int64_t R, int32_t N,
                          float* h_out, void* stream);

/* a8 backward, weight gradients (SURVEY 8(f) rank 2): dW [No, Ni] (row stride ld_w) (+)= dZ^T X and db [No] (+)= column
 * sums of dZ (NULL: skipped), for dZ [S, No] (row stride ld_dz) and X [S, Ni] (row stride ld_x), fp32, No, Ni <= 256
 * (wider layers - the skip layer's [gamma(x), h], the view layer's [feature, gamma(d)] - are split by columns into
 * two calls on the same dZ).  A split-K GEMM over the samples on the tensor cores: every CTA accumulates its share of
 * the samples in tensor memory (operands split into 16-bit hi / lo parts on the fly, hi.hi + lo.hi + hi.lo, fp32
 * accumulation), the partial products are added in a fixed order by a second kernel (deterministic).
 * precision = PNR_PREC_BF16X3 (~2^-17 per product, fp32 exponent range: gradients need no scaling) or PNR_PREC_FP16X3
 * (~2^-21 per product; dz_scale - DEVICE scalar or NULL - is a power of two dZ is multiplied by on load and dW divided
 * by, exact, so that the fp16 parts of ~1e-6 gradients stay normal; |X| and |dZ * scale| must stay below 65504).
 * accumulate != 0 adds to dW / db instead of overwriting them.
 * workspace: pnr_wgrad_workspace_bytes(No, Ni) bytes of device scratch (16-byte aligned) on the current device.
 * Replaces the trunk's dW_j = dZ_j^T [H_{j-1}] on pnr_mlp_backward_trunk's stash and the weight gradients of the
 * layers after the trunk; the reference gets them from torch.autograd through nn.Linear. */
size_t pnr_wgrad_workspace_bytes(int32_t No, int32_t Ni);
int pnr_wgrad(const float* dz, int64_t ld_dz, int32_t No, const float* x, int64_t ld_x, int32_t Ni, int64_t S,
              int32_t precision, const float* dz_scale, float* dW, int64_t ld_w, float* db, int32_t accumulate,
              void* workspace, size_t workspace_bytes, void* stream);

/* a8 on the training path, the layers AFTER the trunk (alpha / feature / view / rgb / heads; SURVEY 8(f) rank 2):
 * y [S, N] (row stride ld_y) = act(x W^T + bias) for x [S, K] (row stride ld_x), fp32, N <= 256, K <= 512, on the
 * tensor cores with the 3-product 16-bit operand split of the fused MLP kernel (precision = PNR_PREC_FP16X3 or
 * PNR_PREC_BF16X3), fp32 accumulation in tensor memory.  W is [N, K] (row stride ld_w), or with transposed != 0 a
 * [K, N] matrix read transposed: dL/dx = g W of a layer y = x W^T is pnr_linear(g, W, transposed = 1).  bias [N] or
 * NULL; relu != 0 applies max(., 0).  in_scale: DEVICE scalar or NULL - a power of two the rows of x are multiplied
 * by on load, the result divided by it (exact): gradients of a mean-reduced loss are ~1e-6 and their fp16 parts would
 * go subnormal unscaled.  workspace: pnr_linear_workspace_bytes(N, K) bytes, 16-byte aligned (the packed weights).
 * The render path does not use this (there these layers are steps of the fused kernel); the reference runs
 * nn.Linear / autograd here. */
size_t pnr_linear_workspace_bytes(int32_t N, int32_t K);
int pnr_linear(const float* x, int64_t ld_x, int32_t K, const float* W, int64_t ld_w, int32_t transposed,
               const float* bias, int32_t N, int64_t S, int32_t relu, int32_t precision, const float* in_scale,
               float* y, int64_t ld_y, void* workspace, size_t workspace_bytes, void* stream);

/* a10: sample_pdf + merge.  z [R,N] coarse depths, weights [R,N] coarse weights; bins are the mid
 * points, the pdf is weights[1:-1]+1e-5.  u [R,Ni] is required (deterministic sampler: the host's
 * linspace(0,1,Ni) broadcast over rays, so the values are the caller's, bit for bit).
 * Out (nullable each): z_fine [R,Ni], idx [R,Ni] i64 (searchsorted right), z_all [R,N+Ni] sorted. */
int pnr_sample_pdf(const float* z, const float* weights, int64_t R, int32_t N, int32_t Ni,
                   const float* u, float* z_fine, int64_t* idx, float* z_all, void* stream);

/* Refresh the weights of a loaded context from DEVICE tensors (same list, order and shapes as pnr_load_weights; fp32,
 * contiguous), stream-ordered on `stream`: what a training loop calls after every optimiser step.  The structure of
 * the per-tile programs does not depend on the values, so nothing is rebuilt or copied through the host: the packed
 * 16-bit streams and constant tables of the forward program (and of the trunk-forward / backward programs once they
 * exist) are rewritten by kernels, including the feature_linear fold.  Bit-identical to a fresh pnr_load_weights of the
 * same values.  A weight outside the fp16 range sets bit 1 of the status word (pnr_status) in the fp16 modes. */
int pnr_update_weights(pnr_ctx* ctx, const float* const* device_tensors, int32_t n, void* stream);

/* Host-only twin of pnr_load_weights (no CUDA call, no context): builds the per-tile program of the fused MLP
 * kernel, the packed 16-bit weight stream and the constant table for `cfg` and returns them in caller buffers
 * (each may be NULL to query sizes only).  `program` receives the MlpProgram struct of csrc/mlp_program.h.
 * For the CPU test tier: tests/test_cpu_program.py replays the program on the host and compares it with
 * the oracle's Network.forward. */
#define PNR_PROGRAM_SPLIT_E1 4  /* flags: E1 signalled in two blocks */
#define PNR_PROGRAM_NO_SPLIT 8  /* flags: start from one-block epilogues instead of the precision's default */
#define PNR_PROGRAM_BACKWARD 16 /* flags: the backward program of the trunk (pnr_mlp_backward_trunk) instead */
#define PNR_PROGRAM_VIEW_PRODUCERS 32 /* flags: the variant whose view epilogue runs on the producer warps (no heads) */
int pnr_program_host(const pnr_config* cfg, const float* const* tensors_host, const int64_t* shapes, int32_t n,
                     int32_t flags, void* program, size_t program_cap, size_t* program_bytes,
                     void* wpacked, size_t wpacked_cap, size_t* wpacked_bytes,
                     float* consts, size_t consts_cap, size_t* n_consts);

/* a3/a4: Renderer.render / batchify_rays as ONE call.  Everything render_rays does for R rays - scene near/far,
 * ray/primitive intersection, stratified sampling + per-sample ids, Network.forward, raw2outputs and, when
 * Ni > 0, sample_pdf + merge + the fine pass - is enqueued on `stream` in ray chunks sized by the caller's
 * workspace, so the big intermediate (raw [chunk, N+Ni, 4+C+K]) never exceeds it (size it with
 * pnr_workspace_bytes).
 * Results do not depend on the chunking (every kernel is per-ray and deterministic).
 * All pointers are DEVICE pointers except aabb_host; outputs and most inputs are optional (NULL). */
enum { PNR_SAMPLE_UNIFORM = 0,    /* z = near*(1-t) + far*t over [near, far], samples tagged with the interval they fall in */
       PNR_SAMPLE_INTERVALS = 1   /* a6: the N samples are placed inside the ray's M hit intervals (pnr_sample_intervals) */ };
typedef struct pnr_render_args {
  const float* rays;            /* [R,6] origin || direction                                                      */
  int64_t R;
  const float* near;            /* [R] and                                                                        */
  const float* far;             /* [R]; or both NULL: from aabb_host (pnr_scene_near_far) or near_min/far_default  */
  const float* aabb_host;       /* {lo.xyz, hi.xyz} HOST floats, or NULL                                          */
  float near_min, far_default;
  const float* box_center;      /* [B,3]   bounding primitives (B = 0: none)                                      */
  const float* box_half;        /* [B,3]                                                                          */
  const float* box_rot;         /* [B,3,3]                                                                        */
  const int32_t* box_sem;       /* [B] class id per primitive (fixed_semantic_map), nullable                      */
  const int32_t* box_inst;      /* [B] instance id per primitive (fixed_instance_map), nullable                   */
  int32_t B, M;                 /* M = hits kept per ray (<= 8)                                                   */
  int32_t N, Ni;                /* coarse samples, importance samples (0: single pass)                            */
  const float* t_vals;          /* [N] linspace(0,1,N) computed by the caller (host linspace, bit for bit)        */
  const float* u;               /* [R,N] jitter, required when perturb > 0                                        */
  float perturb;
  const float* u_fine;          /* [R,Ni] (row stride u_fine_stride floats; 0 = one row shared by all rays)       */
  int64_t u_fine_stride;
  int32_t sample_mode;          /* PNR_SAMPLE_*                                                                   */
  int32_t white_bkgd, sem_softmax, mask_outside, bound_by_primitives;
  pnr_composite_out out;        /* maps of the final pass                                                         */
  pnr_composite_out out0;       /* maps of the coarse pass (only used when Ni > 0)                                */
  float* z_vals;                /* [R,N+Ni] depths of the final pass                                              */
  float* z_vals0;               /* [R,N] coarse depths (Ni > 0)                                                   */
  uint8_t* hit_mask;            /* [R]                                                                            */
  int32_t* box_id;              /* [R,M]                                                                          */
  float* t_in;                  /* [R,M]                                                                          */
  float* t_out;                 /* [R,M]                                                                          */
  int32_t* sample_box;          /* [R,N+Ni] primitive id per sample of the final pass (-1 = none)                 */
  float* near_out;              /* [R] near / far actually used                                                   */
  float* far_out;               /* [R]                                                                            */
  void* workspace;              /* device scratch, caller-owned                                                   */
  size_t workspace_bytes;
} pnr_render_args;
/* ctx_fine: the network of the fine pass (NULL = ctx). */
int pnr_render_fused(pnr_ctx* ctx, pnr_ctx* ctx_fine, const pnr_render_args* args, void* stream);

/* Bytes of device scratch pnr_render_fused wants for R rays: enough for one chunk of min(R, rays_per_chunk) rays
 * with every optional output absent, where rays_per_chunk puts `raw` near 1.5 GB and never below ~64 tiles of the
 * fused MLP per SM (smaller chunks cost more in kernel ramp-up than they save).  Any workspace that holds at
 * least one ray works (more chunks). */
size_t pnr_workspace_bytes(const pnr_ctx* ctx, int64_t R, int32_t N, int32_t Ni);

/* 8(e) multi-GPU entry: one NCCL communicator per rank (NCCL is bound at run time: pnr_comm_available() == 0
 * when libnccl.so.2 cannot be loaded) and ONE all-gather of the rendered per-ray tiles.  Rays shard across ranks
 * with no data-path collective; this gather of image / label tiles is the only exchange step of the path.
 * Rank 0 creates the id with pnr_comm_unique_id and hands its PNR_COMM_ID_BYTES bytes to the other ranks over any
 * out-of-band channel (the host application's launcher; torch.distributed.broadcast in the Python layer).
 * pnr_allgather_outputs: recv [world * bytes_per_rank] <- each rank's send [bytes_per_rank], in rank order,
 * asynchronously on `stream` (in place when send == recv + rank * bytes_per_rank). */
#define PNR_COMM_ID_BYTES 128
typedef struct pnr_comm pnr_comm;
int pnr_comm_available(void);
int pnr_comm_unique_id(uint8_t* id_out);
int pnr_comm_init(pnr_comm** out, const uint8_t* id, int32_t rank, int32_t world, int32_t device);
int pnr_comm_destroy(pnr_comm* comm);
int pnr_allgather_outputs(pnr_comm* comm, const void* send, void* recv, size_t bytes_per_rank, void* stream);

/* Evaluation of rendered frames (the reference's `run.py --type evaluate` / lib/evaluators): every frame passed to
 * pnr_eval_frame is ACCUMULATED into a caller-owned device statistics buffer; nothing is copied to the host per frame.
 * Every input pair is optional (both NULL skips that metric family); all arrays are device pointers, R rays per frame.
 *   semantic   sem_pred [R] i16 (pnr_label_tiles / pnr_panoptic_fuse labels), sem_gt [R] i32: confusion matrix, row =
 *              GT, column = prediction; GT outside [0, C) and predictions outside [0, C) (-1) are ignored.  C <= 64.
 *   panoptic   pan_pred / pan_gt [R] i32, ids category * label_divisor + instance (pnr_panoptic_fuse's convention with
 *              label_divisor 1000), is_thing [C] u8.  A pixel is void when its id is negative or its category is
 *              outside [0, C).  A stuff category (is_thing 0) has one segment: the instance part is dropped.  GT pixels of
 *              a thing category with instance 0 are that category's crowd region.  A predicted segment p and a non-crowd
 *              GT segment g of the same category match iff IoU = |p∩g| / (|p| + |g| - |p∩g| - |p ∩ GT-void|) > 0.5
 *              (strict; the match is then unique).  TP = matches, FN = unmatched non-crowd GT segments, FP = unmatched
 *              predicted segments except those with (|p ∩ GT-void| + |p ∩ crowd(category)|) / |p| > 0.5.  Per category:
 *              TP / FP / FN and the sum of the TPs' IoUs.  At most PNR_EVAL_MAX_SEGMENTS distinct segments per side and
 *              frame: a frame with more adds no PQ terms and increments the overflow word instead.
 *   image      rgb_pred / rgb_gt [R,3] f32: PSNR = -10 log10(mean squared error over the R*3 values), per frame.  With
 *              H * W == R (rays row-major; H = W = 0 skips it): SSIM (Wang et al. 2004) with an 11x11 Gaussian window
 *              (sigma 1.5, separable, normalised), valid region only, c1 = 0.01^2, c2 = 0.03^2, data range 1, variances
 *              clamped at 0, mean over the valid pixels and the 3 channels, window moments in fp64.
 *   depth      depth_pred / depth_gt [R] f32: pixels with 0 < gt <= max_depth count, the prediction is clamped to
 *              [min_depth, max_depth] (min_depth > 0); sums in fp64 of |d|/gt, d^2/gt, d^2, (log p - log gt)^2 and the
 *              counts of valid pixels and of max(p/gt, gt/p) < 1.25, 1.25^2, 1.25^3.
 * Statistics layout (pnr_eval_stats_bytes(C) bytes, 8-byte words; zero it once, then pass frames): the words
 * PNR_EVAL_* below (i64 counts, f64 sums), then from word PNR_EVAL_HEADER_WORDS: conf i64 [C*C], tp i64 [C], fp i64 [C],
 * fn i64 [C], iou_sum f64 [C].  Integer statistics are added with integer atomics, floating-point sums in a fixed order
 * (per-block partials summed by one thread; frames added in call order): the buffer is bit-identical from run to run.
 * workspace: pnr_eval_workspace_bytes(R, C, label_divisor) bytes (256-byte aligned; label_divisor <= 0 when no panoptic
 * inputs are passed), reused by every frame on the same stream.  Arguments are checked before any CUDA call. */
#define PNR_EVAL_MAX_CLASSES 64
#define PNR_EVAL_MAX_SEGMENTS 1024
#define PNR_EVAL_MAX_KEYS (1 << 24)   /* C * label_divisor */
#define PNR_EVAL_HEADER_WORDS 16
enum { PNR_EVAL_OVERFLOW = 0,      /* i64: frames whose segments exceeded PNR_EVAL_MAX_SEGMENTS (no PQ terms added) */
       PNR_EVAL_PQ_FRAMES = 1,     /* i64: frames that added PQ terms                                          */
       PNR_EVAL_PSNR_FRAMES = 2,   /* i64 */
       PNR_EVAL_SSIM_FRAMES = 3,   /* i64 */
       PNR_EVAL_DEPTH_VALID = 4,   /* i64, then DELTA1..3 (i64) in words 5..7                                    */
       PNR_EVAL_DEPTH_DELTA1 = 5, PNR_EVAL_DEPTH_DELTA2 = 6, PNR_EVAL_DEPTH_DELTA3 = 7,
       PNR_EVAL_PSNR_SUM = 8,      /* f64: sum of the per-frame PSNRs (dB)                                     */
       PNR_EVAL_SSIM_SUM = 9,      /* f64: sum of the per-frame SSIMs                                           */
       PNR_EVAL_ABS_REL_SUM = 10, PNR_EVAL_SQ_REL_SUM = 11, PNR_EVAL_SQ_ERR_SUM = 12, PNR_EVAL_SQ_LOG_SUM = 13
       /* words 14, 15: reserved, zero */ };
typedef struct pnr_eval_args {
  int64_t R; int32_t C; int32_t H, W;                  /* H*W == R enables SSIM, else 0, 0                          */
  const int16_t* sem_pred; const int32_t* sem_gt;
  const int32_t* pan_pred; const int32_t* pan_gt; const uint8_t* is_thing; int32_t label_divisor;
  const float* rgb_pred; const float* rgb_gt;
  const float* depth_pred; const float* depth_gt; float min_depth, max_depth;
  void* stats;                                         /* pnr_eval_stats_bytes(C), zeroed once, accumulated         */
  void* workspace; size_t workspace_bytes;             /* pnr_eval_workspace_bytes(R, C, label_divisor)             */
} pnr_eval_args;
size_t pnr_eval_stats_bytes(int32_t C);
size_t pnr_eval_workspace_bytes(int64_t R, int32_t C, int32_t label_divisor);
int pnr_eval_frame(const pnr_eval_args* args, void* stream);

/* Number of kernels this library has launched on this thread since the last reset (bench evidence). */
int64_t pnr_launch_count(int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* PNR_H_ */
