/*
 * rangeclip_b200 -- C ABI of the B200 (sm_100a) kernels behind the DepthCLIP loss / evaluation
 * hot path of jinryan/RangeCLIP.
 *
 * The reference has no FFI: its boundary for this path is the Python call surface
 *   DepthUNet.compute_loss            RangeCLIP/src/depth_segmentation_model/model.py:178-355
 *   masked_average_pooling            model.py:15-56
 *   prepare_image_contrast_data       dataloader.py:205-305  (area pooling: 286-304)
 *   DepthUNet.predict                 model.py:119-175
 *   validate_model metric loop        validate.py:88-139, finalisation 194-214
 * Those signatures are mirrored in Python by the package `rangeclip_b200` (losses.py, pooling.py,
 * evaluation.py); every one of them bottoms out in the entry points declared here, bound with
 * ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless named `h_*`;
 *   - the library never allocates or frees caller-visible memory and never synchronises the
 *     host; every call enqueues work on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = success, negative = rc_status; rc_last_error() gives the text for the
 *     calling thread; no C++ exception crosses the ABI;
 *   - pixel embeddings are the reference's NCHW tensor viewed as [B][D][HW] (HW contiguous),
 *     element type given by an rc_dtype; `ld_b` = elements between images (normally D*HW).
 */
#ifndef RANGECLIP_B200_H_
#define RANGECLIP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RC_ABI_VERSION 1

typedef enum { RC_F32 = 0, RC_BF16 = 1 } rc_dtype;

typedef enum {
  RC_OK = 0,
  RC_ERR_INVALID = -1,      /* bad argument (shape, alignment, null pointer)          */
  RC_ERR_UNSUPPORTED = -2,  /* shape outside what the kernel family supports          */
  RC_ERR_CUDA = -3,         /* CUDA runtime / driver error at launch                  */
  RC_ERR_NO_DEVICE = -4     /* no sm_100 device / driver entry point not available    */
} rc_status;

int rc_abi_version(void);
const char* rc_last_error(void);
/* Number of kernel launches this library has enqueued since load (bench.py's gpu_launches). */
int64_t rc_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Pixel-text / area-image InfoNCE  (replaces model.py:272-291 fwd and its autograd; 304-321)
 *
 *   z[p,k] = <x_p / max(|x_p|, 1e-12), t_k> * inv_tau         t = L2-normalised rows [K][D]
 *   loss   = sum_p w_p (lse_p - z[p, y_p]) / sum_p w_p          y_p = -1 or w_p = 0: ignored
 *
 * `w` carries the reference's sampling-with-replacement multiplicities (model.py:220-228).
 * Accumulators (`loss_sum`, `w_sum`, `dlogtau`) are double[1] each and are ADDED to (zero them).
 * ------------------------------------------------------------------------------------------- */

/* Workspace bytes rc_infonce_* needs for the given problem (bf16 tensor-core path only). */
int64_t rc_infonce_workspace_bytes(int B, int D, int64_t HW, int K, rc_dtype x_dtype);
/* Same, including the bf16 [B][HW][Kp] tensor G the tensor-core dText path needs (rc_infonce_bf16 with dt). */
int64_t rc_infonce_workspace_bytes_dt(int B, int D, int64_t HW, int K, rc_dtype x_dtype);

/* fp32 CUDA-core path (any K >= 1, D % 8 == 0, D <= 512).  Parity path: 1e-5 relative.
 *   dx (nullable) [B][D][HW] f32 = grad_scale * d(loss)/dx, dt (nullable) [K][D] f32 ADDED to.
 *   w_sum_in: device double[1] holding sum_p w_p (needed when dx/dt/dlogtau are requested);
 *   grad_scale: device float[1] upstream gradient (nullable = 1).                             */
int rc_infonce_f32(const float* x, int B, int D, int64_t HW, int64_t ld_b,
                   const float* t, int K, const int32_t* y, const float* w, float inv_tau,
                   float* lse, double* loss_sum, double* w_sum,
                   const double* w_sum_in, const float* grad_scale,
                   float* dx, float* dt, double* dlogtau, void* stream);

/* bf16 tcgen05/TMEM path (K <= 256, D % 64 == 0, D <= 512, HW % 8 == 0).
 *   x        [B][D][HW] f32 or bf16 (x_dtype); f32 input is rounded to bf16 by the pre-pass
 *   t_bf16   [Kp][D] bf16 normalised rows, Kp = K rounded up to 64, pad rows zero
 *   tt_bf16  [D][Kp] bf16 = transpose of t_bf16 (operand of the dX GEMM)
 *   dx       nullable; ALWAYS bf16 [B][D][HW] whatever x_dtype (the tensor cores' gradient; rc_scale_to / rc_tv_bwd_from widen
 *            it in the pass that applies the upstream scale); = grad_scale * w_p/sum(w) * d(lse_p - z_py)/dx
 *   dt       nullable [K][D] f32, ADDED to; needs dx, D = 256 or 512 and a workspace of
 *            rc_infonce_workspace_bytes_dt: the fused kernel also writes G = rs (P - sum onehot)
 *            (bf16 [B][HW][Kp]) and a second tensor-core kernel adds G^T X (split-K over pixels)
 *   workspace from rc_infonce_workspace_bytes; holds bf16 copy of x (f32 input) and 1/|x|.
 *   flags    RC_INFONCE_PREPASS_DONE: the workspace already holds the pre-pass results for this
 *            x (written by rc_infonce_prepass or an earlier call); skip the pre-pass kernel.
 * D = 256 / 512 run the CTA-pair kernel, which computes 1/|x_p| itself from the operand tiles in
 * shared memory: a bf16 x then needs no pre-pass at all.  D = 128 / 384 run the single-CTA kernel
 * (pre-pass + fused kernel).                                                                      */
#define RC_INFONCE_PREPASS_DONE 1
/* More than 256 candidates (e.g. the area-image loss at thousands of objects): split the candidate rows into launches of
 * <= 256 (D = 256 / 512, no dt).  y is then the target index RELATIVE to the launch's first row and may fall outside
 * [0, K); ignored rows are encoded by w = 0 only.
 *   RC_INFONCE_KEEP_WEIGHT  a row whose target is outside this launch keeps its weight (its one-hot term is dropped);
 *                           round 1 = forward launches with this flag: lse per block, loss_sum = sum w lse_blk - sum_{y in blk} w z_y
 *   RC_INFONCE_LSE_GIVEN    `lse` is an INPUT: the row's logsumexp over all candidates (logsumexp of the per-block values);
 *                           round 2 = backward launches with both flags: dx and dlogtau of each block add up to the full gradient
 * rc_infonce_bf16_rep4 takes the same flags (D = 256 / 512, no dt): y4 holds each target relative to the launch's first
 * row, w4 is 0 for every ignored target, lse is [B*hw] (one value per shared row: per block out, or in), and round 1's
 * loss_sum = sum_q wtot_q lse_blk - sum_{y_qj in blk} w_qj z_qy with wtot_q = sum_j w_qj.  rc_infonce_bf16_dyn rejects
 * these flags (its K-blocked form is rc_infonce_bf16_dyn_kblock); rc_infonce_bf16_kblocks takes one target per row only. */
#define RC_INFONCE_KEEP_WEIGHT 2
#define RC_INFONCE_LSE_GIVEN 4
/* Backward launches (dx given, no dt) of D = 256 / 512 with K and log tau given by the host (rc_infonce_bf16, _rep4 and the
 * K-blocked rounds), and those of rc_infonce_bf16_dyn_kblock, run the kernel whose softmax tile is a tensor-memory operand of the dX GEMM (TS-mode tcgen05.mma,
 * csrc/infonce_ts.cu).  Forward-only launches, launches with dt and rc_infonce_bf16_dyn run the kernel with both operands in
 * shared memory (SS, csrc/infonce_umma2.cu).  Both give the same results bit for bit; DESIGN.md records their speed.
 *   RC_INFONCE_SS_KERNEL  run the SS kernel for a backward launch too (A/B measurements)
 *   RC_INFONCE_TS_KERNEL  the default for the launches above; kept so that callers that asked for TS keep working */
#define RC_INFONCE_TS_KERNEL 8
#define RC_INFONCE_SS_KERNEL 32
/* RC_INFONCE_ACCUMULATE_DX: dx += this launch's gradient instead of dx = (TMA reduce-add stores, bf16 accumulation).  The
 * backward launches of the K-blocked scheme after the first one: the per-block gradients add up in ONE bf16 tensor. */
#define RC_INFONCE_ACCUMULATE_DX 16
int rc_infonce_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                    const void* t_bf16, const void* tt_bf16, int K,
                    const int32_t* y, const float* w, float inv_tau,
                    float* lse, double* loss_sum, double* w_sum,
                    const double* w_sum_in, const float* grad_scale,
                    void* dx, float* dt, double* dlogtau,
                    void* workspace, int64_t workspace_bytes, int flags, void* stream);
/* Shared-embedding form (SURVEY 8f-1, decoder.py:113-114): the decoder emits `normalize(nearest_x2(conv))`, so the four
 * pixels of every 2x2 block share one embedding (quirk Q8).  Here a row of x is that shared embedding (x is the
 * PRE-upsample tensor [B][D][hw], normalised or not) and carries four targets / multiplicities:
 *   y4, w4   [B*hw][4] (16-byte aligned), the block's pixels in any fixed order; y = -1 or w = 0: ignored
 *   loss   = sum_q sum_j w_qj (lse_q - z[q, y_qj]) / sum w        (the reference loss on the upsampled tensor)
 *   dx     = gradient with respect to the shared row = the sum of the four pixel gradients -- what autograd
 *            returns below F.interpolate(mode='nearest')
 *   lse    [B*hw]; w_sum_in = sum of all 4 B hw weights (rc_weight_sum over the flat arrays).
 * One quarter of the tensor-core work and HBM traffic of rc_infonce_bf16 on the upsampled tensor.  D = 256 or 512
 * (CTA-pair kernel); everything else as rc_infonce_bf16. */
int rc_infonce_bf16_rep4(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                         const void* t_bf16, const void* tt_bf16, int K,
                         const int32_t* y4, const float* w4, float inv_tau,
                         float* lse, double* loss_sum, double* w_sum,
                         const double* w_sum_in, const float* grad_scale,
                         void* dx, float* dt, double* dlogtau,
                         void* workspace, int64_t workspace_bytes, int flags, void* stream);
/* All candidate blocks of the K-blocked scheme in ONE launch (K > 256 candidates against ONE image of rows, HW % 256 == 0,
 * D = 256 / 512): the kernel's image index runs over the n_blocks = ceil(K / 256) blocks of candidate rows.
 *   t_bf16_all [n_blocks*256][D], tt_bf16_all [D][n_blocks*256] (zero pad rows / columns past K)
 *   y_rel, w_rep [n_blocks][HW]: target index relative to the block's first row (any value outside [0,256) when the
 *       target lives in another block), the row weight repeated per block (0 = ignored row)
 *   round 1 (dx_blocks = NULL): lse [n_blocks][HW] OUT per-block logsumexp; loss_sum += sum_b (sum_p w lse_b - sum_{y in b} w z_y)
 *   round 2 (flags has RC_INFONCE_LSE_GIVEN): lse [HW] IN = logsumexp over the blocks; dx_blocks [n_blocks][D][HW] bf16 OUT,
 *       their sum over the blocks is dx; dlogtau += the full gradient. */
int rc_infonce_bf16_kblocks(const void* x, rc_dtype x_dtype, int D, int64_t HW,
                            const void* t_bf16_all, const void* tt_bf16_all, int K, int n_blocks,
                            const int32_t* y_rel, const float* w_rep, float inv_tau,
                            float* lse, double* loss_sum, double* w_sum, const double* w_sum_in, const float* grad_scale,
                            void* dx_blocks, double* dlogtau, void* workspace, int64_t workspace_bytes, int flags, void* stream);
/* rc_infonce_bf16 / rc_infonce_bf16_rep4 (rep = 1 / 4) for callers that must not synchronise with the host (SURVEY 8f-2):
 * the number of valid candidate rows and the temperature are read from DEVICE memory when the kernel starts.
 *   K        rows of t_bf16 / tt_bf16 the launch is shaped for (<= 256; rows past *k_dev are zero pad rows)
 *   k_dev    device int32[1], valid rows in [1, K] (nullable = K); e.g. k_out[0] of rc_contrast_build
 *   log_tau_dev device float[1] = log(tau) (model.py:99-103 `log_temperature_text`); replaces inv_tau = exp(-log tau)
 * D = 256 or 512 (CTA-pair kernel), no dText, no K-blocked flags; everything else as rc_infonce_bf16. */
int rc_infonce_bf16_dyn(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                        const void* t_bf16, const void* tt_bf16, int K, const int32_t* k_dev,
                        const int32_t* y, const float* w, const float* log_tau_dev, int rep,
                        float* lse, double* loss_sum, double* w_sum,
                        const double* w_sum_in, const float* grad_scale,
                        void* dx, double* dlogtau,
                        void* workspace, int64_t workspace_bytes, int flags, void* stream);
/* rc_infonce_bf16_dyn for one block of the K-blocked rounds (more than 256 rows in the contrast set of the sync-free loss,
 * e.g. rc_contrast_build with k_cap up to 1024): the launch is shaped for rows [k0, k0 + K) of the set, K <= 256, and
 * reads the set's valid row count from k_dev and log(tau) from log_tau_dev (both required) when it starts.
 *   valid rows of the launch = min(K, *k_dev - k0); for k0 = 0 at least 1, as rc_infonce_bf16_dyn
 *   t_bf16 / tt_bf16 the block's rows as [Kp][D] / [D][Kp] (rows past the valid ones are zero pad rows)
 *   y, w     every launch runs the RC_INFONCE_KEEP_WEIGHT form: y is relative to k0 and may fall outside [0, K); w is 0 for
 *            every ignored target.  rep = 1 or 4 (y, w [B*HW] or [B*HW][4])
 *   lse      [B*HW], one value per embedding row: OUT per block in round 1, IN with RC_INFONCE_LSE_GIVEN in round 2
 *   flags    RC_INFONCE_KEEP_WEIGHT, RC_INFONCE_LSE_GIVEN, RC_INFONCE_ACCUMULATE_DX, RC_INFONCE_SS_KERNEL,
 *            RC_INFONCE_PREPASS_DONE.  Backward launches run the TS kernel unless RC_INFONCE_SS_KERNEL (bit-identical).
 * EMPTY LAUNCH: when no row of the block is valid (k0 > 0 and *k_dev <= k0) the kernel returns at once.  It writes no lse
 * and no dx and adds nothing to loss_sum, w_sum or dlogtau, so an RC_INFONCE_ACCUMULATE_DX launch leaves dx as it was.
 * The block at k0 = 0 is never empty; it should be the launch that stores dx.  A caller shapes its launches for the
 * capacity of the set (ceil(capacity / 256) blocks) and combines the per-block results on the device, treating an empty
 * block's lse as -inf.  D = 256 or 512, no dText; everything else as rc_infonce_bf16_dyn. */
int rc_infonce_bf16_dyn_kblock(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                               const void* t_bf16, const void* tt_bf16, int K, const int32_t* k_dev, int k0,
                               const int32_t* y, const float* w, const float* log_tau_dev, int rep,
                               float* lse, double* loss_sum, double* w_sum,
                               const double* w_sum_in, const float* grad_scale,
                               void* dx, double* dlogtau,
                               void* workspace, int64_t workspace_bytes, int flags, void* stream);
/* The pre-pass alone: 1/|x_p| of the bf16-rounded rows (+ bf16 copy of an f32 x) into workspace. */
int rc_infonce_prepass(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                       void* workspace, int64_t workspace_bytes, void* stream);
/* f32 x [B][D][H][W] with W % 8 == 0: the same pre-pass AND the smoothness sums of rc_tv_fwd (model.py:332-334; ADDED to
 * tv_sums[0] = sum |x[h][w+1] - x[h][w]|, tv_sums[1] = sum |x[h+1][w] - x[h][w]|) from ONE read of x; follow with
 * rc_infonce_bf16(..., flags | RC_INFONCE_PREPASS_DONE) on the same workspace. */
int rc_infonce_prepass_tv(const float* x, int B, int D, int H, int W, void* workspace,
                          int64_t workspace_bytes, double* tv_sums, uint32_t* tv_codes, void* stream);
/* tv_codes (nullable, [B][D][H][W/8] words) keeps the SIGNS of those differences, 4 bits per element: pixel j of an 8-pixel
 * group at bits 4j .. 4j+3 = {sgn(x[h][w] - x[h][w+1]) + 1, sgn(x[h][w] - x[h+1][w]) + 1}, two bits each
 * (an opaque format between these two entry points).
 * rc_tv_bwd_codes is rc_tv_bwd_from computed from them instead of from x (the autograd of model.py:332-334 needs nothing
 * else): dx_out (f32) = dx_scale[0] * dx_in (f32 | bf16, nullable) + scale[0] d(sum_w)/dx + scale[1] d(sum_h)/dx. */
int rc_tv_bwd_codes(const uint32_t* codes, int64_t planes, int H, int W, const float* scale,
                    const void* dx_in, rc_dtype dx_in_dtype, const float* dx_scale, float* dx_out, void* stream);

/* Helpers used by both paths.
 * rc_text_prepare: rows of `text[idx[k]]` (idx nullable = identity; `text` has n_rows rows, an index outside [0, n_rows)
 *   yields a row of NaN instead of an out-of-bounds read -- the reference raises an index error there; the pad value -1
 *   of rc_contrast_build yields a zero row) are L2-normalised
 *   (F.normalize, eps 1e-12; model.py:272) and written as f32 [K][D] (nullable), bf16 [Kp][D]
 *   (nullable) and transposed bf16 [D][Kp] (nullable), Kp = round_up(K, 64), pads zeroed.
 * rc_weight_sum: w_sum[0] += sum_p w_p * (y_p >= 0)  (double).
 * rc_sample_weights: w[b][p] = multiplicity of p in rand_idx[b][:] * (seg[b][p] > 0), and
 *   y[b][p] = map[seg[b][p]] (or -1 where seg == 0) -- the dense form of model.py:220-228,276-278.
 * rc_scale: in-place x *= s[0] (device scalar) for a late upstream gradient. */
int rc_text_prepare(const float* text, int64_t ld_text, int64_t n_rows, const int64_t* idx, int K, int D,
                    float* t_f32, void* t_bf16, void* tt_bf16, void* stream);
int rc_weight_sum(const float* w, const int32_t* y, int64_t n, double* w_sum, void* stream);
int rc_sample_weights(const int64_t* seg, const int64_t* rand_idx, int B, int64_t HW, int64_t n_samples,
                      const int32_t* map, int C, float* w, int32_t* y, void* stream);
/* counts[label] += number of sampled pixels (rand_idx [B][n_samples], nullable = every pixel once) carrying that label, labels
 * outside [0, C) skipped; counts int32[C] is ADDED to.  The sampled foreground labels of model.py:222-233 (gather, drop 0,
 * torch.unique) are the nonzero entries from 1 on -- no gather, no sort.  C <= 12000. */
/* Device-side contrast-set builder (model.py:234-268 without the .tolist() / np.random / randperm host round trips):
 *   counts     int32[C] label histogram of the sampled pixels (rc_sample_label_counts); labels >= 1 with counts > 0 are "present"
 *   sim_off / sim_items   CSR over labels (int32[C+1] / int32[nnz], nullable together): per label the union of the similarity
 *              lists in use (label_similarity_sets['medium'] if n_medium > 0, ['hard'] if n_hard > 0)
 *   n_curriculum = n_medium + n_hard candidates are drawn without replacement from the lists of the present labels (all of
 *              them if there are fewer), n_rand from every label that is neither present nor chosen (label 0 included)
 *   k_cap      rows the loss launch is shaped for: distractors are trimmed to fit (flag 2); present labels beyond it are
 *              dropped from the map (flag 1)
 *   seed       draws = the n smallest of key(c) = splitmix64(splitmix64(seed ^ phase << 56) + c), phase 1 / 2
 *   include_label0  0: label 0 is background and never "present" (compute_loss, model.py:226); 1: it is a label like any other
 *              (the reduced candidate set of predict, model.py:147-156: GT labels of the batch + num_negatives random others)
 *   seed_dev   nullable device int64[1]: XORed into `seed` by the kernel -- a seed produced on the device (e.g. by a graph-safe
 *              generator) gives every replay of a captured CUDA graph its own draw
 * Outputs: label_map int32[C] (position in the sorted contrast set or -1), contrast int64[k_cap] (sorted ids, -1 pads:
 * rc_text_prepare turns those into zero rows), k_out int32[4] = {K, flags, #present, #distractors}.  C <= 16384. */
int rc_contrast_build(const int32_t* counts, int C, const int32_t* sim_off, const int32_t* sim_items,
                      int n_curriculum, int n_rand, int k_cap, uint64_t seed, const int64_t* seed_dev,
                      int include_label0, int32_t* label_map, int64_t* contrast, int32_t* k_out, void* stream);
int rc_sample_label_counts(const int64_t* seg, const int64_t* rand_idx, int B, int64_t HW, int64_t n_samples, int C,
                           int32_t* counts, void* stream);
int rc_scale(void* x, rc_dtype dtype, int64_t n, const float* s, void* stream);
/* out[i] = s[0] * x[i] (s nullable = 1) into a separate buffer, converting x_dtype -> out_dtype: the late upstream scaling of a
 * saved gradient (autograd may run a backward twice; the saved tensor must stay intact) and the bf16 -> f32 widening of the
 * tensor-core gradient in one pass. */
int rc_scale_to(const void* x, rc_dtype x_dtype, void* out, rc_dtype out_dtype, int64_t n, const float* s, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Segment-masked average pooling  (replaces dataloader.py:286-304 and model.py:36-54)
 *   slot = lut[b * lut_ld + seg[b][p]]  (lut_ld = 0: one LUT for the whole batch, model.py:15)
 *   sum[slot][d] += x[b][d][p], count[slot] += 1; rc_pool_finish divides (zeros when empty).
 * ------------------------------------------------------------------------------------------- */
int rc_pool_fwd(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                const int64_t* seg, const int32_t* lut, int64_t lut_ld, int C, int n_slots,
                float* sum /*[n][D], zeroed*/, int32_t* count /*[n], zeroed*/, void* stream);
int rc_pool_finish(float* sum_inout, const int32_t* count, int n_slots, int D, void* stream);
/* dx[b][d][p] = g[slot][d] / count[slot] (0 where slot < 0); dx dtype = x_dtype. */
int rc_pool_bwd(const float* g, const int32_t* count, int B, int D, int64_t HW,
                const int64_t* seg, const int32_t* lut, int64_t lut_ld, int C, int n_slots,
                void* dx, rc_dtype x_dtype, int accumulate, void* stream);

/* ---------------------------------------------------------------------------------------------
 * L2-normalised pixel rows  (F.normalize(x, p=2, dim=1), the decoder tail utils/src/decoder.py:114, as one operator)
 *   fwd: out[b][:,p] = x[b][:,p] / max(|x[b][:,p]|, 1e-12) as f32 whatever x's dtype (F.normalize is an fp32 op under
 *        autocast), inv_norm[b][p] (nullable) = the factor
 *   bwd: dx (x's dtype) = (g - xhat (xhat . g)) * inv_norm, xhat and g f32
 * HW % 8 == 0, 32-byte aligned pointers.  Used where compute_loss_shared2x2 needs the normalised rows the decoder would
 * have emitted (smoothness, area pooling) without eager PyTorch's ~10 full-tensor passes.
 * ------------------------------------------------------------------------------------------- */
int rc_normalize_rows_fwd(const void* x, rc_dtype dtype, int B, int D, int64_t HW, float* out, float* inv_norm, void* stream);
int rc_normalize_rows_bwd(const float* xhat, const float* g, const float* inv_norm, rc_dtype dtype, int B, int D, int64_t HW,
                          void* dx, void* stream);

/* Backward of the smoothness term through the normalisation in ONE kernel (model.py:332-334 on decoder.py:114's output):
 *   dx = d/dx [ scale[0] * sum |xh[..,w]-xh[..,w+1]| + scale[1] * sum |xh[..,h,:]-xh[..,h+1,:]| ],  xh = x / max(|x|, 1e-12)
 * from the saved xhat / inv_norm of rc_normalize_rows_fwd; scale = device float[2]; sign(0) = 0; dx in `dtype`; W % 8 == 0.
 * (Instead of rc_tv_bwd -> a gradient tensor the size of xhat -> rc_normalize_rows_bwd.) */
int rc_tv_normalize_bwd(const float* xhat, const float* inv_norm, const float* scale, rc_dtype dtype, int B, int D, int H, int W,
                        void* dx, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Smoothness (TV-L1)  (replaces model.py:332-334 and its autograd)
 *   sums[0] += sum |x[..,w]-x[..,w+1]|, sums[1] += sum |x[..,h,:]-x[..,h+1,:]|  (double[2])
 *   bwd: dx (=|+=) scale_h * d(sum_h)/dx + scale_v * d(sum_v)/dx, sign(0) = 0;
 *        scales are device floats scale[2]; when dx_scale (device float[1], nullable) is given
 *        and accumulate != 0 the existing dx is first multiplied by it (fused late upstream
 *        scaling of the InfoNCE gradient).
 * ------------------------------------------------------------------------------------------- */
int rc_tv_fwd(const void* x, rc_dtype x_dtype, int64_t planes, int H, int W, double* sums, void* stream);
int rc_tv_bwd(const void* x, rc_dtype x_dtype, int64_t planes, int H, int W, const float* scale,
              void* dx, int accumulate, const float* dx_scale, void* stream);
/* Out-of-place / mixed-dtype form: dx_out (x_dtype) = dx_scale[0] * dx_in + scale_h d(sum_h)/dx + scale_v d(sum_v)/dx.
 * dx_in may be bf16 under an f32 x (the tensor-core InfoNCE gradient): the fused text + smoothness backward of an f32
 * embedding tensor then reads x once, dx_in once and writes dx once.  dx_in == dx_out (same dtype) is allowed. */
int rc_tv_bwd_from(const void* x, rc_dtype x_dtype, int64_t planes, int H, int W, const float* scale,
                   const void* dx_in, rc_dtype dx_in_dtype, const float* dx_scale, void* dx_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Evaluation  (replaces model.py:164-173 and validate.py:88-139)
 * rc_eval_topk_f32 / rc_eval_topk_bf16: top-k (k <= 8) text ids per pixel by cosine logit,
 *   ties broken towards the smaller reduced index; out[b][j][p] = index_map[arg] (int64).
 * rc_eval_hist: per-batch histograms over equivalence classes
 *   hist[0][L]=#(ge==L) hist[1][L]=#(p1==L) hist[2][L]=#(ge==L & p1==L)
 *   hist[3][L]=#(oracle==L) hist[4][L]=#(ge==L & oracle==L); counters {correct_top1,
 *   correct_topk, total}; all int64, ADDED to.
 * rc_eval_fold: fold one batch's hist into the running accumulators with the reference's
 *   per-batch label-presence rule (validate.py:108) and record first-seen batch per label.
 * ------------------------------------------------------------------------------------------- */
int rc_eval_topk_f32(const float* x, int B, int D, int64_t HW, int64_t ld_b, const float* t, int K,
                     const int64_t* index_map, int k, int64_t* out, void* stream);
int rc_eval_topk_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                      const void* t_bf16, int K, const int64_t* index_map, int k, int64_t* out,
                      void* workspace, int64_t workspace_bytes, void* stream);
/* Fused form: the top-k ids of a pixel go from the scan registers straight into the five class histograms and the
 * three counters of rc_eval_hist (same per-pixel function, warp-aggregated atomics); `out` is optional (NULL when only
 * the metrics are wanted).  hist / counters are ADDED to. */
int rc_eval_topk_hist_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                           const void* t_bf16, int K, const int64_t* index_map, int k, int64_t* out /*nullable*/,
                           const int64_t* gt /*[B*HW]*/, const uint8_t* E, const int64_t* cmap, int C,
                           int64_t* hist /*[5][C]*/, int64_t* counters /*[3]*/,
                           void* workspace, int64_t workspace_bytes, void* stream);
/* rc_eval_topk_bf16 / rc_eval_topk_hist_bf16 with the number of valid text rows read from DEVICE memory when the kernel starts
 * (a candidate set built by rc_contrast_build: model.py:147-161 without the unique().tolist() / random.sample round trip):
 * K = rows the launch is shaped for (t_bf16 has round_up(K, 64) rows, rows past *k_dev are pads), k_dev device int32[1] in
 * [1, K].  `out` and `hist` are both optional; at least one must be given. */
int rc_eval_topk_dyn_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW,
                          const void* t_bf16, int K, const int32_t* k_dev, const int64_t* index_map, int k,
                          int64_t* out /*nullable*/, const int64_t* gt, const uint8_t* E, const int64_t* cmap, int C,
                          int64_t* hist /*nullable [5][C]*/, int64_t* counters /*[3]*/,
                          void* workspace, int64_t workspace_bytes, void* stream);
/* rc_eval_topk_bf16 / _hist_bf16 / _dyn_bf16 on the decoder's half-resolution rows x [B][D][h*w] (the output_conv result,
 * SURVEY 8f-1): the top-k of row (i, j) is the top-k of the four full-resolution pixels (2i+a, 2j+b) of the nearest-x2
 * upsampled tensor; out [B][k][2h][2w] and gt [B][2h][2w] are FULL resolution.  k_dev nullable (NULL: K valid rows);
 * out and hist optional, at least one given; hist / counters are added to.  h*w % 8 == 0. */
int rc_eval_topk_bf16_rep4(const void* x, rc_dtype x_dtype, int B, int D, int h, int w, const void* t_bf16, int K,
                           const int32_t* k_dev, const int64_t* index_map, int k, int64_t* out, const int64_t* gt,
                           const uint8_t* E, const int64_t* cmap, int C, int64_t* hist, int64_t* counters,
                           void* workspace, int64_t workspace_bytes, void* stream);
int rc_eval_hist(const int64_t* gt, const int64_t* topk, int B, int64_t HW, int k,
                 const uint8_t* E, const int64_t* cmap, int C,
                 int64_t* hist /*[5][C]*/, int64_t* counters /*[3]*/, void* stream);
int rc_eval_fold(const int64_t* batch_hist /*[5][C]*/, int C, int32_t batch_index,
                 int64_t* acc /*[4][C]: I1,U1,IK,UK*/, int32_t* first_seen /*[C], init INT32_MAX*/,
                 void* stream);

/* ---------------------------------------------------------------------------------------------
 * Debug / bring-up: one 128 x N x Kd bf16 GEMM tile through the same TMA + tcgen05 + TMEM
 * building blocks (descriptor variants selected by `variant`), C[128][N] f32 row-major.
 *   variant 0: A K-major [128][Kd], B K-major [N][Kd]
 *   variant 1: A MN-major [Kd][128] (the NCHW pixel operand), B K-major [N][Kd]
 *
 * Bring-up entry points and environment switches (RANGECLIP_B200_ABLATE / _INFONCE / _DT) exist ONLY in
 * librangeclip_b200_bringup.so, built with -DRC_BRINGUP (`make -C rangeclip_b200/csrc bringup`); the shipped
 * librangeclip_b200.so exports none of them and reads no environment variable.
 * ------------------------------------------------------------------------------------------- */
/* ---------------------------------------------------------------------------------------------
 * Object crops for the CLIP image encoder  (replaces dataloader.py:254,276: the per-object slice
 * `image[:, ymin:ymax, xmin:xmax]` + `clip_processor(images=crops, return_tensors="pt", do_rescale=False)`,
 * i.e. transformers 5.5.0 TorchvisionBackend._preprocess: bicubic antialiased resize of the shortest edge to
 * `shortest_edge`, centre crop to crop_size x crop_size, (v - mean) / std) -- all crops of a batch in one launch.
 *   images [B][C][H][W] f32 or bf16; boxes int32 [n][4] = xmin, ymin, xmax, ymax (pixels, exclusive max);
 *   image_index int32 [n]; mean, stdv float[C]; out f32 [n][C][crop_size][crop_size].
 * A box outside its image (the reference skips those on the host) yields a zero crop. */
int rc_clip_crops(const void* images, rc_dtype dtype, int B, int C, int H, int W, const int32_t* boxes,
                  const int32_t* image_index, int n, int shortest_edge, int crop_size, const float* mean,
                  const float* stdv, float* out, void* stream);

#ifdef RC_BRINGUP
/* Bring-up instrumentation: when set (device int64[32]), CTA 0 of rc_infonce_bf16 records per-barrier
 * wait cycles of its producer / MMA / softmax / epilogue roles; index 0 = role lifetime. NULL disables. */
int rc_debug_set_timing_buffer(int64_t* dev_buf);
int rc_debug_umma_gemm(const void* a_bf16, const void* b_bf16, int N, int Kd, int variant,
                       float* c, void* stream);

/* Bring-up query: number of clusters of `cluster_size` CTAs (block size and dynamic shared memory as given) the device
 * keeps resident at once (cudaOccupancyMaxActiveClusters); negative = rc_status. */
int rc_debug_max_active_clusters(int cluster_size, int threads, int smem_bytes);

/* CTA-pair (cta_group::2) variant of the bring-up GEMM: C[256][N] = A[256][Kd] B[N][Kd]^T, both K-major. */
int rc_debug_umma_gemm_2sm(const void* a_bf16, const void* b_bf16, int N, int Kd, float* c, void* stream);
/* Same GEMM with A as a tensor-memory operand (TS mode): the threads write A [256][Kd] (Kd <= 256) to TMEM with tcgen05.st. */
int rc_debug_umma_gemm_ts_2sm(const void* a_bf16, const void* b_bf16, int N, int Kd, float* c, void* stream);
#endif /* RC_BRINGUP */

#ifdef __cplusplus
}
#endif
#endif /* RANGECLIP_B200_H_ */
