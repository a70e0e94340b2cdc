/*
 * ian_b200.h -- C-ABI of libian_b200.so: the B200-native (sm_100a) implementation of the IAN hot path
 * of ajbrock/Neural-Photo-Editor.
 *
 * The reference has NO native boundary for this path: its contract is the Python class API.IAN
 * (reference API.py:11-110), whose methods hand numpy arrays to Theano-compiled functions.  Each entry
 * point below replaces one of those compiled functions; the citation says which.  A host binding
 * (ctypes, cffi, cgo, JNI ...) needs nothing but this header: plain pointers and sizes, int status
 * codes, no C++/torch types.  The Python mirror of API.IAN that ships in this repo
 * (neural-photo-editor_b200/API.py) is such a binding; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every function returns IAN_OK (0) or a negative ian_status; ian_last_error() gives the text.
 *   - image tensors are float32 NCHW (n,3,64,64) in [-1,1]; latents are float32 (n,100); row-major.
 *   - *_dev entry points take DEVICE pointers valid on the handle's device and enqueue on `stream`
 *     (a cudaStream_t passed as void*, NULL = the handle's own stream) without synchronising.
 *   - *_host entry points take HOST pointers, do H2D, compute, D2H and return after the result landed
 *     (the numpy-in / numpy-out semantics of the reference's theano.function calls).
 *   - a handle is bound to one device and is not thread-safe (API.IAN is single-threaded: NPE.py calls
 *     it from the Tk main loop).
 *   - results are reproducible: a call repeated with the same batch size returns the same bits (split-K and
 *     stream-K partial sums are added in a fixed order; there are no atomics on the path).
 *   - environment, read by ian_create: IAN_CHUNK=<n> images per internal chunk (default 512); IAN_PATH=simt selects
 *     the FFMA verification kernels; IAN_STREAMK=0 disables stream-K scheduling; IAN_GRAPHS=0 disables the CUDA-graph
 *     replay that *_host calls with <= 32 images use; IAN_TC2=0 keeps every layer on the one-CTA tap-GEMM kernel
 *     (default: layers with >= IAN_TC2_MIN (37) whole pair-tiles run on CTA pairs, tcgen05 cta_group::2);
 *     IAN_SPLITK=0 disables split-K (tests); IAN_PUSH=kernel makes the pipelined all-gather push with a copy kernel
 *     (IAN_PUSH_CTAS=<n> CTAs) instead of copy engines + stream memory operations; IAN_PDL=0 launches the kernel chains
 *     plainly instead of with programmatic dependent launch; IAN_FINALIZE8=0 chooses the one-thread split-K finalize.
 *     All of these select schedules or launch forms of the same kernels (DESIGN.md section 5.8);
 *     results do not depend on IAN_GRAPHS, IAN_PDL or IAN_FINALIZE8 (bit-identical), the others change float32 summation
 *     order within the tolerances of the parity tests.
 *   - stream semantics of *_dev calls: kernels of one call are chained with programmatic dependent launch among themselves;
 *     towards the caller's own work on `stream` (kernels, copies, events before and after the call) the usual stream order
 *     holds -- the first kernel of a call waits for everything enqueued before it before it reads or writes any argument,
 *     and a kernel the caller launches afterwards without the programmatic attribute starts after the call's last kernel
 *     has completed.
 */
#ifndef IAN_B200_H_
#define IAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ian_handle ian_handle;

typedef enum ian_status {
  IAN_OK = 0,
  IAN_ERR_INVALID = -1,   /* bad argument (shape, NULL, non-integral box, empty box ...)        */
  IAN_ERR_CUDA = -2,      /* CUDA runtime / driver error                                        */
  IAN_ERR_STATE = -3,     /* call order: parameters missing, not finalized ...                  */
  IAN_ERR_UNSUPPORTED = -4
} ian_status;

/* Model graph selector.  Replaces `config_module.get_model(dnn=dnn)` (reference API.py:18-21). */
typedef enum ian_model_kind {
  IAN_MODEL_SIMPLE = 0,   /* reference IAN_simple.py:56-241                                                  */
  IAN_MODEL_FULL = 1,     /* reference IAN.py:67-228: MADE/IAF latent flow, MDC blocks, RGB-Beta head          */
  IAN_MODEL_V1 = 2        /* reference IANv1.py:63-222: MADE/IAF latent flow, plain deconv decoder, RGB-Beta   */
} ian_model_kind;

/* Compute path of the dense contractions (enc_conv2-4, dec_conv1-3, fully-connected layers).
 * Both are CUDA on the GPU; there is no CPU path.
 *   IAN_PATH_TC   : tcgen05 tensor-core kernels, fp32 emulated by a 3-pass bf16 split (default)
 *   IAN_PATH_SIMT : fp32 FFMA kernels (verification path, bit-for-bit independent of IAN_PATH_TC) */
typedef enum ian_path { IAN_PATH_TC = 0, IAN_PATH_SIMT = 1 } ian_path;

/* ---- lifecycle: replaces IAN.__init__ (reference API.py:12-64) --------------------------------- */

/* Create an empty model on CUDA device `device`. */
int ian_create(int model_kind, int device, ian_handle** out);

/* Upload one parameter under its reference checkpoint name ("enc_conv2.W", "bnorm2.inv_std", ...;
 * names and shapes: reference GANcheckpoints.py:33-57 + IAN_simple.py layer names).  `data` is a HOST
 * float32 array of `ndim` dims `shape`, in the reference's own layout (conv W (Cout,Cin,5,5); deconv W
 * (Cin,Cout,5,5); dense W (in,out)).  Unlike the reference loader (which only warns,
 * GANcheckpoints.py:45-52) a name outside ian_model_param_spec's list or a shape mismatch is an error, and so is a
 * parameter still missing at ian_finalize. */
int ian_set_param(ian_handle* h, const char* name, const float* data, const int64_t* shape, int ndim);

/* The model's OWN parameter list -- what `lasagne.layers.get_all_params(...)` hands GANcheckpoints.load_weights in the
 * reference (API.py:23-30; GANcheckpoints.py:33-57).  A loader iterates index 0..count-1, looks each `name` up in the
 * checkpoint and calls ian_set_param; keys of the file that are not in this list (the trainer's `log_sigma_theta`,
 * discriminator weights, `metadata`) are ignored exactly as the reference loader ignores them.  Handle-free (no GPU
 * needed).  ian_model_param_count returns the count (or a negative ian_status); `name` stays valid for the life of
 * the process; `shape` receives 4 entries (trailing ones are 1). */
int ian_model_param_count(int model_kind);
int ian_model_param_spec(int model_kind, int index, const char** name, int64_t* shape /*[4]*/, int* ndim);

/* IAN_MODEL_FULL / IAN_MODEL_V1: the MADE input ordering (a permutation of 0..99) from which the autoregressive masks are
 * derived by integer comparison (reference mask_generator.py:29-38,93-94).  Replaces the one
 * `shuffle_ordering` draw of `l_IAF_mu/ls.reset("Once")` (reference API.py:33-36).  Must precede ian_finalize. */
int ian_set_made_ordering(ian_handle* h, const int32_t* ordering, int n);

/* The 0/1 autoregressive mask the library derives from `ordering` for one MaskedLayer, as (in,out) bytes [100][100]:
 * which = 0 `<net>_input` (mask_generator.py:93 for layer 0), 1 `<net>_output_W`, 2 `<net>_output_D` (direct
 * input->output, layers.py:822-836).  Pure host integer logic (handle-free): lets a test compare the mask indexing
 * bit for bit with the reference's MaskGenerator. */
int ian_made_mask(const int32_t* ordering, int n, int which, uint8_t* mask_out);
/* Debug getter: the masked MADE weights W*M as uploaded, float32 [2 nets: mu, ls][3: input, output_W, output_D][100][100]. */
int ian_debug_made_weights(ian_handle* h, float* out);

/* Check that every parameter of the graph is present, fold BatchNorm (inference), re-lay weights for
 * the kernels and upload them.  Must precede any compute call. */
int ian_finalize(ian_handle* h);

int ian_destroy(ian_handle* h);
const char* ian_last_error(const ian_handle* h);   /* h may be NULL: last error of ian_create     */

int ian_get_zdim(const ian_handle* h);             /* replaces IAN.get_zdim (API.py:92-96) -> 100 */
int ian_set_path(ian_handle* h, int path);         /* ian_path                                    */
/* Arithmetic of the dense contractions.  IAN_PRECISION_FP32 (default): float32 semantics, every operand kept as
 * bf16 hi|lo planes, 3 tensor-core passes.  IAN_PRECISION_BF16 (full IAN only; BASELINE configs[2]): operands
 * rounded to bf16, one pass, fp32 accumulation -- about 1e-2 max-abs from the float32 result. */
typedef enum ian_precision { IAN_PRECISION_FP32 = 0, IAN_PRECISION_BF16 = 1 } ian_precision;
int ian_set_precision(ian_handle* h, int precision);
/* Number of kernels this library launched on the handle since creation (bench.py gpu_launches). */
int64_t ian_launch_count(const ian_handle* h);

/* ---- encode: replaces Z_hat_fn / IAN.encode_images (reference API.py:50-51, 78-90) ------------- */
/* z = mu(x) (deterministic=True, what API.py:50 compiles).  If eps != NULL the reparameterised
 * sample z = mu + exp(logsigma) * eps (reference layers.py:419-433, eps injected: (n,100)).       */
int ian_encode_dev(ian_handle* h, const float* x, int n, const float* eps, float* z, void* stream);
int ian_encode_host(ian_handle* h, const float* x, int n, const float* eps, float* z);

/* ---- decode: replaces X_hat_fn / IAN.sample_at (reference API.py:46-47, 98-110) ---------------- */
int ian_decode_dev(ian_handle* h, const float* z, int n, float* x, void* stream);
int ian_decode_host(ian_handle* h, const float* z, int n, float* x);

/* ---- encode -> decode in one call (BASELINE metric; no reference equivalent: NPE calls the two
 * functions back to back, NPE.py:257-261) ------------------------------------------------------- */
int ian_reconstruct_dev(ian_handle* h, const float* x, int n, float* z_out /*nullable*/, float* x_hat,
                        void* stream);
int ian_reconstruct_host(ian_handle* h, const float* x, int n, float* z_out /*nullable*/, float* x_hat);

/* ---- pipelined encode -> decode for streaming use (no reference equivalent; the reference is synchronous) --
 * ian_reconstruct_submit enqueues  H2D(x) -> encode -> decode -> D2H(x_hat[, z])  on three streams (copy-in,
 * compute, copy-out) and returns a ticket at once; up to two requests are in flight, so the copies of one request
 * overlap the compute of its neighbours.  ian_reconstruct_wait blocks until that request's outputs have landed in
 * the host buffers, which must stay valid until then.  n <= 512.  Pinned host memory (ian_host_alloc) is what
 * makes the copies asynchronous; pageable memory works but serialises. */
int ian_reconstruct_submit(ian_handle* h, const float* x, int n, float* z_out /*nullable*/, float* x_hat, int* ticket);
int ian_reconstruct_wait(ian_handle* h, int ticket);
/* Page-locked host memory owned by the handle (freed by ian_host_free or ian_destroy). */
int ian_host_alloc(ian_handle* h, size_t bytes, void** out);
int ian_host_free(ian_handle* h, void* p);

/* ---- data-parallel encode -> decode with the all-gather FUSED into the decoder's last kernel (no reference
 * equivalent: the reference is single-GPU).  One process per GPU; every rank calls, in order:
 *   ian_gather_create(h, world, rank, n_local, handle64)   allocate this rank's double gather buffer, get its 64-byte
 *                                                          CUDA IPC handle
 *   (exchange the handles between ranks with any transport, e.g. torch.distributed.all_gather)
 *   ian_gather_connect(h, all_handles)                     map every peer's buffer (NVLink peer access)
 *   ian_reconstruct_gather_dev(h, x, n_local, z, &gathered, stream)   per step
 * The decoder's last kernel stores each decoded image straight into slot `rank` of EVERY rank's gather buffer (st.global
 * on peer pointers): dec_out for IAN_MODEL_SIMPLE, the RGB-Beta head's last kernel for IAN_MODEL_FULL and IAN_MODEL_V1.
 * Every graph runs its gather in the handle's current precision (ian_set_precision), on the tensor-core path only
 * (IAN_PATH_SIMT returns IAN_ERR_UNSUPPORTED).  A flag barrier over peer memory then makes the step complete:
 * `gathered` (world*n_local,3,64,64) holds all ranks' images on return of the stream work.  n_local may exceed the
 * 512-image plan chunk (the shard then runs as consecutive chunks into the same gather buffer, one barrier at the end).
 * Lifetime of a result: the two gather buffers alternate, so step t+1 of ANY rank never touches the buffer that holds
 * step t -- but a peer that has passed the barrier of step t+1 may begin its step t+2 stores into it.  A result is
 * therefore valid until the stream work of THIS rank's next call has executed: enqueue every consumer of step t on
 * `stream` (or order it before) the call of step t+1.  tests/test_gpu_multi.py skews the ranks to check exactly this. */
int ian_gather_create(ian_handle* h, int world, int rank, int n_local, void* ipc_handle_out /*64 bytes*/);
int ian_gather_connect(ian_handle* h, const void* all_handles /*world x 64 bytes*/);
int ian_reconstruct_gather_dev(ian_handle* h, const float* x, int n_local, float* z_out /*nullable*/, float** gathered_out,
                               void* stream);
/* Pipelined form of the same all-gather, for streams of batches.  dec_out's peer stores are bound by the NVLink
 * egress (7 x 12.6 MB per GPU and step at 8 x 256 images: ~0.11 ms of link time behind a 0.04 ms kernel), so here the
 * shard is decoded into this rank's own buffer and a side stream pushes it to every peer WHILE the next step's tensor
 * kernels run -- by copy engines, with the free/pushed flag handshake that orders the buffer reuse across ranks done as
 * stream memory operations (cuStreamWriteValue32 / cuStreamWaitValue32) on peer-mapped flag words, so that no SM is taken
 * from the persistent tensor kernels (a copy-kernel form exists behind IAN_PUSH=kernel and measured slower for that
 * reason).  ian_reconstruct_gather_async_dev enqueues one step and returns; ian_gather_wait_dev makes `stream`
 * wait until the most recent step's images of ALL ranks have landed and returns that buffer.  A result must be
 * consumed (in stream order) before the call that submits the step after next.  Steps are collective: every rank
 * calls the same sequence of gather entry points. */
int ian_reconstruct_gather_async_dev(ian_handle* h, const float* x, int n_local, float* z_out /*nullable*/, void* stream);
int ian_gather_wait_dev(ian_handle* h, float** gathered_out, void* stream);

/* ---- the function set of the reference's sampling script (reference sample_IAN.py:86-94) ---------------------
 *   Zfn      : X -> l_Z_IAF (deterministic = mu, before the MADE/IAF flow)        -> ian_encode_pre_host
 *   Z_IAF_fn : l_Z_IAF -> l_Z = (z - MADE_mu(z)) / exp(MADE_ls(z))                 -> ian_flow_host(z_out)
 *   sample   : l_Z_IAF -> X (flow, then decoder)                                   -> ian_flow_host(x_out)
 *   sampleZ  : l_Z -> X                                                            -> ian_decode_host
 * For IAN_MODEL_SIMPLE there is no flow: Zfn == encode and Z_IAF_fn is the identity. */
int ian_encode_pre_host(ian_handle* h, const float* x, int n, float* z_iaf);
int ian_flow_host(ian_handle* h, const float* z_iaf, int n, float* z_out /*nullable*/, float* x_out /*nullable*/);

/* ---- latent-brush gradients: replace calculate_RGB_gradient / calculate_lighten_gradient
 * (reference API.py:59, 64; IAN.imgrad / IAN.imgradRGB API.py:66-76), batched per sample -------- */
/* boxes: (n,4) int32 rows [c1,r1,c2,r2], half-open box [r1:r2, c1:c2], 0<=c1<c2<=64, 0<=r1<r2<=64.
 * target: NULL -> lighten gradient d/dz mean(x_hat[k,:,box_k]);
 *         target_is_frame=0 -> (n,3) colour per sample, broadcast over the frame;
 *         target_is_frame=1 -> (n,3,64,64) frames (what NPE passes, NPE.py:205).
 * g: (n,100) = d/dz_k mean((target_k[:,box_k] - x_hat[k,:,box_k])^2).                              */
int ian_grad_dev(ian_handle* h, const float* z, const int32_t* boxes, const float* target,
                 int target_is_frame, int n, float* g, void* stream);
int ian_grad_host(ian_handle* h, const float* z, const int32_t* boxes, const float* target,
                  int target_is_frame, int n, float* g);

/* ---- latent edit loop: n_steps of the NPE paint rule (reference NPE.py:199-209) per sample:
 *        g = grad(z);  z <- z - weight * g * (1 + (c2 - c1))        (all float32)
 * in place on z (n,100).  `weight` = 0.05 in NPE.py:199.                                          */
int ian_edit_loop_dev(ian_handle* h, float* z, const int32_t* boxes, const float* target,
                      int target_is_frame, int n, int n_steps, float weight, void* stream);
int ian_edit_loop_host(ian_handle* h, float* z, const int32_t* boxes, const float* target,
                       int target_is_frame, int n, int n_steps, float weight);

/* ---- one NPE paint stroke in ONE call: replaces the body of paint() in photo mode (reference NPE.py:199-231):
 *   g = imgradRGB(box, rgb_frame, z);  z <- z - weight * g * (1 + (c2 - c1));  x_hat = sample_at(z)
 *   DELTA = x_hat - to_tanh(RECON);  MASK = gaussian_filter(min(mean_c|DELTA|, 1), 0.7)
 *   IM = uint8(from_tanh(to_tanh(RECON) + MASK*DELTA + (1-MASK)*ERROR))
 * z (1,100) in/out; box int32[4] = [c1,r1,c2,r2]; rgb_frame (1,3,64,64) float32 in [-1,1]; recon_u8 (3,64,64) uint8;
 * error (3,64,64) float32; im_u8 (3,64,64) uint8 out; display_u8 (256,256,3) uint8 out (nullable): IM upsampled 4x
 * nearest-neighbour in HWC order, what update_photo() hands to PIL (NPE.py:107-118).  IAN_MODEL_SIMPLE only. */
int ian_paint_stroke_host(ian_handle* h, float* z, const int32_t* box, const float* rgb_frame, float weight,
                          const uint8_t* recon_u8, const float* error, uint8_t* im_u8, uint8_t* display_u8);

/* ---- training-mode pieces (no trainer here: train_IAN*.py stay the reference's; these are the two forward ops whose
 * training form differs from the deterministic graphs everything above runs).  Device pointers, float32.
 *
 * BatchNorm with BATCH statistics = lasagne BatchNormLayer.get_output_for(deterministic=False), i.e. every BN(...) of
 * reference IAN_simple.py:84-170 / layers.py:411-416 in training.  x is (n, c, hw) (NCHW with hw = H*W; dense layers: hw = 1).
 *   ian_bn_batch_stats_dev      per-channel sum and sum of squares (float64 [c] each) over (n, hw): warp-shuffle reductions,
 *                               fixed order, bit-reproducible.  Data-parallel ranks all-reduce the two arrays here
 *                               (cross-GPU synchronised BN) and pass the GLOBAL element count to the second call.
 *   ian_bn_train_normalize_dev  mean = sum/count, inv_std = 1/sqrt(sumsq/count - mean^2 + eps)  (biased variance);
 *                               y = (x - mean) * (gamma * inv_std) + beta;  running_mean / running_inv_std (nullable) are
 *                               updated in place: r <- (1 - alpha) r + alpha * batch value.  lasagne: eps 1e-4, alpha 0.1.
 * ian_minibatch_discrim_dev     MinibatchLayer.get_output_for(init=False) of reference layers.py:486-524:
 *                               x (n,d), theta (d,K,P), log_weight_scale (K,P), b (K) -> out (n, d+K) = [x | f]. */
int ian_bn_batch_stats_dev(ian_handle* h, const float* x, int n, int c, int hw, double* sum, double* sumsq, void* stream);
int ian_bn_train_normalize_dev(ian_handle* h, const float* x, int n, int c, int hw, const double* sum, const double* sumsq,
                               double count, const float* gamma /*nullable*/, const float* beta /*nullable*/, float eps,
                               float alpha, float* running_mean /*nullable*/, float* running_inv_std /*nullable*/, float* y,
                               void* stream);
int ian_minibatch_discrim_dev(ian_handle* h, const float* x, int n, int d, const float* theta, const float* log_weight_scale,
                              const float* b, int num_kernels, int dim_per_kernel, float* out, void* stream);

/* ---- measurement helpers ----------------------------------------------------------------------- */
/* Average device time (ms, CUDA events on the launch stream) of the tap-GEMM kernel of layer
 * `layer_name` ("enc_conv2", "dec_conv1", ...) over the launches since the last reset; returns <0 if
 * the layer was never timed.  Timing is enabled with ian_set_layer_timing(h, 1). */
int ian_set_layer_timing(ian_handle* h, int enable);
double ian_layer_time_ms(ian_handle* h, const char* layer_name, int reset);

#ifdef __cplusplus
}
#endif
#endif /* IAN_B200_H_ */
