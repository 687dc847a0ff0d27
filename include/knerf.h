/* knerf.h -- C ABI of libknerf.so: the B200 (sm_100a) implementation of keras_nerf's per-ray hot path.
 *
 * The reference (naufalso/keras_nerf) is pure Python on TensorFlow and has NO FFI / custom-op
 * interface of its own; the drop-in boundary is its Python class API (SURVEY.md §8b).  The entry
 * points below are what a TF custom-op (`Compute(OpKernelContext*)` on TF's GPU stream) or the
 * ctypes/DLPack shim in keras_nerf_b200/ binds for each reference function; every declaration cites
 * the reference code it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *  - All pointers are CALLER-OWNED DEVICE memory unless the name ends in `_host`.  The library never
 *    frees or retains them.  Tensors are float32, row-major, last dim contiguous.
 *  - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it (no host sync).
 *  - Every function returns 0 on success or a negative knerf_status; knerf_last_error() gives the
 *    thread-local message.  No C++ exception crosses the ABI.
 *  - Stateless: no global mutable state and no process-wide mode switches (options travel with each call, see
 *    KNERF_TC_ORDERED below); safe to call from several host threads on distinct streams (the reference calls
 *    RaysGenerator from tf.data worker threads, keras_nerf/data/loader.py:96-98).  The only objects the library
 *    owns are the communicators of knerf_comm_* (multi-GPU), created and destroyed by the caller.
 *  - Randomness is explicit: functions that the reference feeds from tf.random.uniform take the
 *    uniforms as an argument (`u`), or NULL + a seed for the built-in counter-based Philox4x32-10.
 */
#ifndef KNERF_H
#define KNERF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KNERF_ABI_VERSION 2

typedef enum knerf_status {
  KNERF_OK = 0,
  KNERF_ERR_INVALID = -1,     /* bad argument (null pointer, size, unsupported shape) */
  KNERF_ERR_CUDA = -2,        /* CUDA runtime / launch error */
  KNERF_ERR_UNSUPPORTED = -3, /* configuration outside what the selected precision mode implements */
  KNERF_ERR_WORKSPACE = -4,   /* workspace too small (see knerf_workspace_bytes) */
  KNERF_ERR_NCCL = -5         /* NCCL not loadable, or an NCCL call failed (knerf_comm_*, knerf_allreduce_grads) */
} knerf_status;

/* out-of-range tf.gather in the fine sampler (keras_nerf/model/nerf/utils.py:87-88, SURVEY App. C-1) */
typedef enum knerf_oob_mode {
  KNERF_OOB_ZERO = 0,  /* TF-GPU kernel: out-of-range index reads 0   (parity default) */
  KNERF_OOB_CLAMP = 1, /* clamp to the last mid point */
  KNERF_OOB_COUNT = 2  /* as ZERO, and count offending samples into *oob_count (host raises: TF-CPU) */
} knerf_oob_mode;

/* OR-ed into every `oob_mode` argument.  tf.reduce_sum / tf.cumsum do not define a summation order
 * (TF-CPU is sequential, TF-GPU uses a cub scan).  The default is a warp-shuffle scan; with this flag the
 * pdf normaliser and the cdf are summed strictly left to right in fp32 (TF-CPU / NumPy order), which makes
 * the cdf -- and through it every fine depth -- bit-identical to the CPU oracle.  The fp32 parity mode of
 * the Python shim sets it: the out-of-range-gather quirk (App. C-1) turns a 1e-6 cdf difference into a
 * 5e-4 depth difference for the ~3% of samples that land in [0, near).                                  */
#define KNERF_SCAN_SEQUENTIAL 0x10

typedef enum knerf_precision {
  KNERF_FP32 = 0, /* SIMT FFMA, fp32 end to end: the 1e-5 parity mode                   */
  KNERF_BF16 = 1, /* tcgen05 tensor cores: bf16 operands, fp32 TMEM accumulation; models of dense_units <= 256
                   * (even), up to 8 layers, at most one skip concat (not into the heads), pos_emb_xyz <= 10,
                   * pos_emb_dir <= 4 (else KNERF_ERR_UNSUPPORTED) */
  KNERF_FP32_TC = 2 /* fp32-grade results ON the tensor cores: every fp32 operand is split into three bf16 values
                       (24 mantissa bits) and each product formed from its six leading bf16 x bf16 terms, fp32
                       accumulation in TMEM; one GEMM per Dense layer like KNERF_FP32, same 1e-5 parity bar, several
                       times its speed.  Layers whose width is not a multiple of 64 stay on the SIMT path.          */
} knerf_precision;

/* Per-call options, OR-ed into every `precision` argument (the library keeps NO process-wide mode switches).
 *  KNERF_TC_ORDERED     BF16 inference: the two MMA-issuing threads of the forward kernel hand over in ring
 *                       order like the training kernels do (bit-reproducible outputs, ~14 % slower).  Default:
 *                       they interleave freely (last-bit run-to-run differences).
 *  KNERF_BWD_DGRAD_ONLY / KNERF_BWD_WGRAD_ONLY   knerf_mlp_backward (BF16) launches only its dgrad chain kernel /
 *                       only its weight-gradient kernels, so that a benchmark can time them apart.
 *  KNERF_REC_FP8        BF16 training: the records the forward and the dgrad chain save for the weight-gradient GEMMs
 *                       are 8-bit floats (activations e4m3, pre-activation gradients e5m2 under one power-of-two scale
 *                       per backward call) instead of bf16: half the bytes through HBM, the forward outputs and the
 *                       dgrad chain unchanged.  The training forward and the backward of a step must both carry it
 *                       (knerf_train_chunk passes it to both).                                                  */
#define KNERF_PRECISION_MASK 0xff
#define KNERF_TC_ORDERED 0x100
#define KNERF_BWD_DGRAD_ONLY 0x200
#define KNERF_BWD_WGRAD_ONLY 0x400
#define KNERF_REC_FP8 0x800

/* The 7 ints of model_config.json (keras_nerf/model/nerf/nerf.py:47-55) + encoded widths.
 * dx/dd = width of the xyz / direction encodings fed to the MLP; 0 means 3+6*pos_emb_*.      */
typedef struct knerf_config {
  int32_t n_coarse, n_fine, pos_emb_xyz, pos_emb_dir, n_layers, dense_units, skip_layer;
  int32_t dx, dd;
} knerf_config;

int knerf_abi_version(void);
const char* knerf_last_error(void);
/* number of CUDA kernels this library has launched in the process so far (bench.py's gpu_launches) */
uint64_t knerf_launch_count(void);
/* 1 if the library contains the tcgen05 path and the current device is sm_100 */
int knerf_device_supports_bf16(void);

/* ---- a3  RaysGenerator.__call__  (keras_nerf/data/rays.py:69-130) ------------------------------
 * c2w_host: 16 floats row-major (HOST).  u: [H*W*n_samples] uniforms in [0,1) or NULL (then Philox(seed)).
 * Outputs o[H*W,3], d[H*W,3], t[H*W,n_samples]; ray id = y*W + x.                                */
int knerf_generate_rays(const float* c2w_host, int H, int W, float focal, float near_, float far_,
                        int n_samples, const float* u, uint64_t seed, float* o, float* d, float* t,
                        void* stream);

/* ---- random ray batches drawn across all training views (NeRF's N_rand; no counterpart in the reference) ----------
 * images[n_img, H, W, C] (C >= 3; rgb in channels 0..2, e.g. ImageLoader's RGBA fp32) and c2w[n_img, 4, 4] (DEVICE):
 * the prepared training views.  Pixel id p = (img*H + y)*W + x over P = n_img*H*W pixels.  Epoch `epoch` of key
 * `perm_seed` visits every pixel once, in the order of a bijection pi of [0, P) computed in the kernel (no buffer):
 * a 4-round balanced Feistel network on the smallest even bit width b >= 2 with 2^b >= P, cycle-walked until the
 * value is < P.  Round r maps (L, R) -> (R, L ^ (mix(R ^ k_r) & mask)), mix = the splitmix64 finaliser,
 * k_r = mix(mix(perm_seed) ^ (epoch*0x9E3779B97F4A7C15 + 0xD1B54A32D192ED03)) + r*0x9E3779B97F4A7C15, and the
 * output is (L << b/2) | R.  Any window of any epoch is computed independently, so data-parallel ranks take disjoint
 * windows of the same epoch without communicating.
 * This call writes rays first .. first+R-1 of that order: pixel p_j = pi(first + j) gives o[j,3], d[j,3] and
 * t[j, n_samples] -- the same bits knerf_generate_rays writes for pixel p_j of its view given the same uniforms --
 * and target[j,3] = images[p_j, 0..2]; pixel[j] = p_j (int64, may be NULL).  u: [R*n_samples] uniforms or NULL (then
 * Philox(seed) at counter j*n_samples + k, the batch-local convention of knerf_generate_rays).
 * KNERF_ERR_INVALID: null pointer, n_img/H/W/n_samples <= 0, C < 3, first < 0, first + R > P.                  */
int knerf_generate_ray_batch(const float* images, int n_img, int H, int W, int C, const float* c2w, float focal,
                             float near_, float far_, int n_samples, uint64_t perm_seed, uint64_t epoch,
                             int64_t first, int64_t R, const float* u, uint64_t seed, float* o, float* d, float* t,
                             float* target, int64_t* pixel, void* stream);

/* tf.random.uniform stand-in: n floats, multiples of 2^-24 in [0,1), Philox4x32-10(seed, offset) */
int knerf_uniform(float* out, int64_t n, uint64_t seed, uint64_t offset, void* stream);

/* ---- a4  NeRFUtils.positional_encoding  (keras_nerf/model/nerf/utils.py:176-186) ----------------
 * x[n_rows, dim] -> out[n_rows, ld_out] holding dim*(1+2L) columns (ld_out >= that; extra columns
 * are zero-filled).                                                                              */
int knerf_positional_encoding(const float* x, int64_t n_rows, int dim, int L, float* out, int ld_out,
                              void* stream);

/* ---- a5  NeRFUtils.encode_position_and_directions  (keras_nerf/model/nerf/utils.py:188-210) -----
 * o[R,3], d[R,3], t[R,S] -> xyz[R*S, ld_xyz] (3+6*L_xyz cols), dirs[R*S, ld_dir] (3+6*L_dir cols) */
int knerf_encode_position_and_directions(const float* o, const float* d, const float* t, int64_t R,
                                         int S, int L_xyz, int L_dir, float* xyz, int ld_xyz,
                                         float* dirs, int ld_dir, void* stream);

/* ---- a7  NeRFUtils.render_image_depth_chunk  (keras_nerf/model/nerf/utils.py:16-58) -------------
 * Inputs either packed rgbsigma[R,S,4] (r,g,b,sigma) or separate rgb[R,S,3] + sigma[R,S] (the other
 * NULL).  white/clip = 0 reproduces the test-only render_image_depth (utils.py:99-134).
 * Outputs image[R,3], depth[R], weights[R,S] (any may be NULL), acc[R] = sum of weights (may be NULL). */
int knerf_composite_forward(const float* rgbsigma, const float* rgb, const float* sigma, const float* t,
                            int64_t R, int S, int white_background, int clip, float epsilon,
                            float* image, float* depth, float* weights, float* acc, void* stream);

/* Fused backward of the above + MSE (what autodiff of keras_nerf/model/nerf/nerf.py:361-377 yields).
 * dL/dimage is either given (dimage[R,3]) or formed in-kernel as loss_scale*(image - target) with
 * target[R,3]; then sqerr[R] (may be NULL) receives sum_c (image-target)^2 per ray.
 * through_activations=1: outputs are gradients w.r.t. the PRE-activations of the heads
 * (rgb = sigmoid(.), sigma = relu(.)), packed d_out[R,S,4]; 0: w.r.t. rgb and sigma themselves.    */
int knerf_composite_backward(const float* rgbsigma, const float* t, int64_t R, int S,
                             int white_background, int clip, float epsilon, const float* dimage,
                             const float* target, float loss_scale, int through_activations,
                             float* d_out, float* sqerr, void* stream);

/* ---- a8 (+ sort of a9)  fine_hierarchical_sampling_chunk  (keras_nerf/model/nerf/utils.py:60-97,
 *      keras_nerf/model/nerf/nerf.py:182-191) ------------------------------------------------------
 * Either t_coarse[R,Nc] (mid points formed in-kernel, nerf.py:182-183, and t_sorted[R,Nc+Nf] =
 * sort(concat(t_coarse, samples)) written), or mid_points[R,Nc-1] given explicitly (t_coarse NULL,
 * t_sorted NULL).  weights[R,Nc]; u[R,Nf] or NULL (Philox(seed)); cdf_in[R,Nc+1] overrides the
 * in-kernel cdf (bin indices are bit-exact given the reference's cdf).  Optional outputs:
 * samples[R,Nf] (unsorted), indices[R,Nf] (searchsorted side='right'), cdf_out[R,Nc+1],
 * oob_count (single int32, KNERF_OOB_COUNT).                                                     */
int knerf_sample_fine(const float* t_coarse, const float* mid_points, const float* weights,
                      const float* u, uint64_t seed, const float* cdf_in, int64_t R, int Nc, int Nf,
                      int oob_mode, float* t_sorted, float* samples, int32_t* indices, float* cdf_out,
                      int32_t* oob_count, void* stream);

/* ---- a6  NeRFMLP  (keras_nerf/model/nerf/mlp.py:5-50) -------------------------------------------
 * Parameters live in ONE flat fp32 buffer per network in Keras variable order
 * (layer_0..layer_{n-1}, sigma, features, rgb_features, rgb; kernel[in,out] then bias[out]).       */
int64_t knerf_param_count(const knerf_config* cfg);
/* table of the n_layers+4 dense layers: offsets (in floats) of kernel and bias, fan_in, fan_out */
int knerf_layer_table(const knerf_config* cfg, int max_layers, int64_t* kernel_off, int64_t* bias_off,
                      int32_t* fan_in, int32_t* fan_out);

/* bytes of scratch the MLP / chunk entry points need for `rows` = R*S samples (`precision` with the option bits
 * the calls will carry: KNERF_REC_FP8 halves the training records) */
int64_t knerf_workspace_bytes(const knerf_config* cfg, int64_t rows, int precision, int training);

/* NeRFMLP.call on already-encoded inputs: xyz[rows, ld_xyz], dirs[rows, ld_dir] -> rgb[rows,3],
 * sigma[rows,1] (fp32 SIMT path, any widths; mirrors tests/model/nerf/test_nerf_mlp.py).            */
int knerf_mlp_forward_encoded(const knerf_config* cfg, const float* params, const float* xyz,
                              int ld_xyz, const float* dirs, int ld_dir, int64_t rows, float* rgb,
                              float* sigma, void* workspace, int64_t workspace_bytes, void* stream);

/* bf16 operand images of the weights for the tcgen05 path (re-run after every optimizer step) */
int64_t knerf_packed_weight_bytes(const knerf_config* cfg);
int knerf_pack_weights(const knerf_config* cfg, const float* params, void* packed, void* stream);

/* Fused PE + MLP + heads: (o[R,3], d[R,3], t[R,S]) -> rgbsigma[R,S,4].  `packed` is required for
 * KNERF_BF16 (NULL otherwise).  training=1 keeps the activations the backward needs in `workspace`. */
int knerf_mlp_forward(const knerf_config* cfg, const float* params, const void* packed, const float* o,
                      const float* d, const float* t, int64_t R, int S, int precision, int training,
                      float* rgbsigma, void* workspace, int64_t workspace_bytes, void* stream);

/* Backward of knerf_mlp_forward (same workspace, same R,S): d_pre[R,S,4] = gradient w.r.t. the head
 * pre-activations; grads (flat, Keras order) is ACCUMULATED into (grads += dL/dtheta).             */
int knerf_mlp_backward(const knerf_config* cfg, const float* params, const void* packed,
                       const float* d_pre, int64_t R, int S, int precision, float* grads,
                       void* workspace, int64_t workspace_bytes, void* stream);

/* ---- a9/a10  NeRF._predict_and_render_chunk x2  (keras_nerf/model/nerf/nerf.py:175-227) ----------
 * coarse pass then fine pass for R rays.  Outputs (any may be NULL): image_*[R,3], depth_*[R],
 * weights_c[R,Nc], weights_f[R,Nc+Nf], t_fine_sorted[R,Nc+Nf].                                    */
int knerf_render_chunk(const knerf_config* cfg, const float* params_coarse, const float* params_fine,
                       const void* packed_coarse, const void* packed_fine, const float* o,
                       const float* d, const float* t_coarse, int64_t R, const float* u_fine,
                       uint64_t seed, int white_background, int oob_mode, int precision,
                       float* image_c, float* depth_c, float* weights_c, float* image_f, float* depth_f,
                       float* weights_f, float* t_fine_sorted, void* workspace, int64_t workspace_bytes,
                       void* stream);

/* ---- a11/a12  one chunk of NeRF.train_step  (keras_nerf/model/nerf/nerf.py:351-421) --------------
 * coarse fwd+MSE+bwd, fine fwd+MSE+bwd.  grads_* += grad(mean-squared-error of this chunk) * grad_scale
 * (grad_scale = 1/sequential_chunks, nerf.py:383-384); losses[0], losses[1] += chunk MSE * grad_scale
 * (device floats).  image_c/image_f[R,3] may be NULL.                                             */
int knerf_train_chunk(const knerf_config* cfg, const float* params_coarse, const float* params_fine,
                      const void* packed_coarse, const void* packed_fine, const float* o, const float* d,
                      const float* t_coarse, const float* target_rgb, int64_t R, const float* u_fine,
                      uint64_t seed, int white_background, int oob_mode, int precision,
                      float grad_scale, float* grads_coarse, float* grads_fine, float* losses,
                      float* image_c, float* image_f, void* workspace, int64_t workspace_bytes,
                      void* stream);

/* ---- a13  Keras Adam  (keras_nerf/model/nerf/nerf.py:163-165,455-458) ----------------------------
 * theta -= lr*sqrt(1-b2^t)/(1-b1^t) * m/(sqrt(v)+eps); m,v updated in place; step = t (1-based).
 * zero_grads=1 clears `grads` afterwards (nerf.py:465-471).                                       */
int knerf_adam_step(float* params, float* grads, float* m, float* v, int64_t n, float lr, float beta1,
                    float beta2, float epsilon, int64_t step, int zero_grads, void* stream);

/* sum_c,rays (a-b)^2 / n  -> out[0] (device float); used for test_step losses / PSNR (nerf.py:306-330) */
int knerf_mse(const float* a, const float* b, int64_t n, float* out, void* stream);

/* ---- a18 / f1  per-image metrics of NeRF.update_and_return_metrics  (keras_nerf/model/nerf/nerf.py:306-330) ---
 * a, b: [B,H,W,C] float32.  mse[B] = mean (a-b)^2 per image (tf.image.psnr(max_val=1) = -10 log10 of it);
 * ssim[B] = tf.image.ssim(a, b, max_val) with its defaults (11x11 gaussian window, sigma 1.5, k1 .01, k2 .03,
 * VALID positions, mean over positions and channels).  Either output may be NULL.  H, W >= 11.  `workspace`:
 * knerf_image_metrics_workspace_floats(B,H,W,C) floats of device scratch.  Bit-reproducible (fixed-order sums). */
int64_t knerf_image_metrics_workspace_floats(int B, int H, int W, int C);
int knerf_image_metrics(const float* a, const float* b, int B, int H, int W, int C, float max_val, float* mse,
                        float* ssim, float* workspace, int64_t workspace_floats, void* stream);

/* ---- f3  ImageLoader.__call__ after the PNG decode  (keras_nerf/data/image.py:17-35) --------------------
 * rgba: [in_h, in_w, 4] uint8 (DEVICE; what tf.io.decode_image(channels=4) yields).  Fuses
 * convert_image_dtype (x * 1/255), tf.image.resize(bilinear, antialias=True) (ScaleAndTranslate, triangle
 * kernel, rows then columns, fp32 sums in span order), the alpha composite on a white (1) / black (0)
 * background, the alpha concat and the [0,1] clip.  out: [out_h, out_w, 4] float32.  Note that the reference
 * passes (image_width, image_height) as tf.image.resize's (height, width) (image.py:22-23).                */
int knerf_image_prepare(const uint8_t* rgba, int in_h, int in_w, int out_h, int out_w, int white_background,
                        float* out, void* stream);

/* ---- a14  cross-replica gradient SUM  (train.py:75,110; keras_nerf/model/nerf/nerf.py:455-458) --------------
 * tf.distribute.MirroredStrategy all-reduces (SUM) every gradient inside optimizer.apply_gradients.  Here: one
 * process per GPU, one NCCL communicator per process, and the flat fp32 gradient buffers of the two networks
 * (2 x 595,844 floats) are SUM-all-reduced in place over NVLink.  NCCL is bound at run time
 * (dlopen("libnccl.so.2"): the copy the host process already loaded, else the system one), so single-GPU users
 * need no NCCL at all.
 *   knerf_comm_unique_id    rank 0 fills id_host[KNERF_COMM_ID_BYTES] (HOST memory) and hands the bytes to the other
 *                           ranks through whatever the host has (MPI, a file, the host framework's own collectives).
 *   knerf_comm_create       collective over all ranks: builds the communicator for the CURRENT CUDA device.
 *   knerf_comm_adopt        wraps an existing ncclComm_t of the host framework instead (not destroyed by the library).
 *   knerf_comm_destroy      frees a communicator (and the NCCL one if knerf_comm_create made it).
 *   knerf_allreduce_grads   grads[n] (device) <- SUM over ranks, in place, asynchronous on `stream`.
 * A communicator is used by one host thread at a time (NCCL rule); all ranks issue the same calls in the same order. */
#define KNERF_COMM_ID_BYTES 128
typedef struct knerf_comm knerf_comm;
int knerf_comm_unique_id(void* id_host);
int knerf_comm_create(const void* id_host, int rank, int nranks, knerf_comm** comm);
int knerf_comm_adopt(void* nccl_comm, int rank, int nranks, knerf_comm** comm);
int knerf_comm_destroy(knerf_comm* comm);
int knerf_comm_rank(const knerf_comm* comm, int* rank, int* nranks);
int knerf_allreduce_grads(knerf_comm* comm, float* grads, int64_t n, void* stream);

/* knerf_train_chunk for ray-sharded data parallelism.  Same arguments and arithmetic; with reduce != 0 (the LAST
 * accumulation chunk of the step) the all-reduce of grads_coarse (n_params floats) is enqueued on `comm_stream` as
 * soon as the coarse network's backward has finished -- it travels over NVLink while the fine network is still in
 * its forward / backward on `stream` -- and the all-reduce of grads_fine follows the fine backward; `stream` waits
 * for both before the call's work is complete, so an Adam step enqueued on `stream` afterwards sees the reduced
 * gradients.  comm == NULL or reduce == 0: identical to knerf_train_chunk.  comm_stream must differ from stream.  */
int knerf_train_chunk_dp(const knerf_config* cfg, const float* params_coarse, const float* params_fine,
                         const void* packed_coarse, const void* packed_fine, const float* o, const float* d,
                         const float* t_coarse, const float* target_rgb, int64_t R, const float* u_fine,
                         uint64_t seed, int white_background, int oob_mode, int precision,
                         float grad_scale, float* grads_coarse, float* grads_fine, float* losses,
                         float* image_c, float* image_f, void* workspace, int64_t workspace_bytes,
                         void* stream, knerf_comm* comm, void* comm_stream, int reduce);

/* ---- mesh export: isosurface of a scalar grid (NeRF.extract_mesh; no counterpart in the reference) ---------------
 * Marching tetrahedra on the Kuhn split: every cell of field[nx,ny,nz] (index (i*ny + j)*nz + k, x slowest) is cut into
 * the 6 tets 0 -> e_a -> e_a+e_b -> (1,1,1), one per axis permutation (a,b,c) in the order 012, 021, 102, 120, 201, 210.
 * The split is the same in every cell, so the surface is watertight; there are no ambiguous cases.
 *  - a grid point is inside when f > iso (strict); the edge p -> p+delta (delta in 100, 010, 001, 110, 101, 011, 111, in
 *    that order) carries a vertex when exactly one endpoint is inside, at t = (iso - f_p) / (f_q - f_p),
 *    v = origin + spacing * (p + t*delta) (fp32), with the normal = -normalise(interpolated central-difference gradient,
 *    one-sided on the grid faces), pointing towards decreasing f; a zero gradient gives a zero normal.
 *  - a tet with 1 or 3 corners inside gives one triangle; 2 inside (a,b) and 2 outside (c,d) give the quad
 *    ac, ad, bd, bc split along ac-bd.  Counter-clockwise seen from outside: the normal of the triangle through the
 *    EDGE MIDPOINTS points from the inside corners' centroid towards the outside ones'.
 *  - vertices in the order (grid point, delta); triangles in the order (cell, tet, triangle).  No atomics: two runs
 *    give the same bytes.
 * Usage: the count pass writes counts[2] = {V, T} (DEVICE int64); the caller reads them back, allocates, then calls the
 * emit pass with the same field, iso and workspace (untouched in between).  vertices[V,3], normals[V,3] (may be NULL),
 * triangles[T,3] int32; nothing is written at or beyond max_vertices / max_triangles.  max_vertices >= 2^31 is
 * KNERF_ERR_UNSUPPORTED (int32 indices).  Workspace: knerf_isosurface_workspace_bytes, 256-byte aligned, about
 * 5 bytes per grid point.  nx, ny, nz >= 2.                                                                        */
int64_t knerf_isosurface_workspace_bytes(int nx, int ny, int nz);
int knerf_isosurface_count(const float* field, int nx, int ny, int nz, float iso, int64_t* counts, void* workspace,
                           int64_t workspace_bytes, void* stream);
int knerf_isosurface_emit(const float* field, int nx, int ny, int nz, float iso, const float* origin_host,
                          const float* spacing_host, float* vertices, float* normals, int32_t* triangles,
                          int64_t max_vertices, int64_t max_triangles, void* workspace, int64_t workspace_bytes,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KNERF_H */
