// edge.h -- launchers of the HBM-bound end kernels and glue (see edge_kernels.cu).
#pragma once
#include "tapgemm.h"

namespace ian {
constexpr int kMaxPeers = 8;

// where a decoder's last kernel stores the decoded images: one buffer (single GPU) or the same offset of every rank's
// gather buffer -- the all-gather of the data-parallel path is fused into the kernel's stores (peer pointers over NVLink).
// Written by decout_tc_kernel (IAN_simple) and head_b_out_kernel (IAN.py / IANv1.py).
struct DecOutDst {
  float* base[kMaxPeers];
  int n;
};

// every launcher returns the number of kernels launched (1) or <0 on a launch error
int launch_conv1(const float* x, const float* wt, const float* bias, __nv_bfloat16* out, long long plane, int n,
                 cudaStream_t st);
int launch_dec_out(const __nv_bfloat16* h3, long long plane, const float* wt, float* xhat, int n, cudaStream_t st);
int launch_sample(const float* head, const float* eps, float* z, __nv_bfloat16* zp, long long zplane, int n,
                  cudaStream_t st);
int launch_z_to_planes(const float* z, __nv_bfloat16* zp, long long zplane, int n, cudaStream_t st);
int launch_brush_seed_bwd(const float* xhat, const int32_t* boxes, const float* target, int target_is_frame,
                          const float* wt, const float* scale3, const __nv_bfloat16* h3, __nv_bfloat16* d3,
                          long long plane, int n, cudaStream_t st);
int launch_brush_update(const float* gpad, const int32_t* boxes, float weight, float* g_out, float* z,
                        __nv_bfloat16* zp, long long zplane, int n, cudaStream_t st);
// NPE photo-mode blend + display upsample after a stroke (NPE.py:107-118, 218-231)
int launch_npe_blend(const float* xhat, const uint8_t* recon, const float* error, uint8_t* im, uint8_t* display, cudaStream_t st);
// full IAN: MADE+IAF latent flow and the autoregressive RGB-Beta head
int launch_made_iaf(const float* z0, const float* mw, const float* mb, float* z, __nv_bfloat16* zp, long long zplane, int n,
                    cudaStream_t st);
int launch_head_gather(const float* tt, int tt_is_bf16, const int* taps, int ntaps, float* ha, int n, cudaStream_t st);
// dsts[0..ndst): destination base pointers of x_hat, as for launch_dec_out_tc
int launch_rgb_beta_head(const float* ha, int ha_planar, float* rg, const int* taps, const float* wgb, const float* wbb, int ntaps,
                         float* const* dsts, int ndst, float* bsave /*nullable*/, int n, cudaStream_t st);
// brush gradient through the RGB-Beta head: seed over the box, beta/sigmoid/autoregressive backward into dpre (n,64,64,8),
// then the im2col operand a2 (n,64,64,256 split planes) of the dense backward GEMM (see edge_kernels.cu)
int launch_head_bwd(const float* xhat, const float* rg, const float* bsave, const int32_t* boxes, const float* target,
                    int target_is_frame, const int* taps, const float* wgb, const float* wbb, int ntaps, float* dpre,
                    __nv_bfloat16* a2, long long a2_plane, int n, cudaStream_t st);
// RGB-Beta head on the tensor-core path (head_tc.cu): dense GEMM per (image, conv) + on-chip tap gather -> ha [n][6][4096]
// (the autoregressive sigmoid / Beta part stays the three per-pixel kernels of edge_kernels.cu)
struct HeadMaps;
HeadMaps* head_build_maps(const __nv_bfloat16* fh4, long long fh4_plane, int n_img, const __nv_bfloat16* wt, long long wt_plane,
                          char* err, int errlen);
void head_free_maps(HeadMaps*);
int launch_head_tc(const HeadMaps* maps, int passes, float* ha, int n, cudaStream_t st);
// enc_conv1 on the tensor-core path (conv1_tc.cu): thread-built im2col tile + tcgen05
struct Conv1Maps;
struct Conv1OutMap;
// wt: three blocks of [128 cout][64 k] bf16 (hi k<64 | lo k<64 | tail: hi k 64..79, lo k 64..79, zeros)
Conv1Maps* conv1_build_maps(const __nv_bfloat16* wt, char* err, int errlen);
void conv1_free_maps(Conv1Maps*);
// per plan: the TMA-store view of the a1 activation planes the kernel writes
Conv1OutMap* conv1_build_out_map(__nv_bfloat16* out, long long plane, int n, char* err, int errlen);
void conv1_free_out_map(Conv1OutMap*);
int launch_conv1_tc(const Conv1Maps* maps, const Conv1OutMap* omap, const float* x, const float* bias, int n, cudaStream_t st);
// dec_out on the tensor-core path (decout_tc.cu)
struct DecOutMaps;
DecOutMaps* decout_build_maps(const __nv_bfloat16* h3, long long h3_plane, int n_img, const __nv_bfloat16* wt,
                              long long wt_plane, char* err, int errlen);
void decout_free_maps(DecOutMaps*);
// dsts[0..ndst): destination base pointers (1 = local only; >1 = every rank's gather buffer incl. peers)
int launch_dec_out_tc(const DecOutMaps* maps, float* const* dsts, int ndst, int n, cudaStream_t st);
// signal + wait kernels of the peer-memory barrier (flag_ptrs[r] = rank r's flag array, int[8])
int launch_peer_barrier(float* const* flag_ptrs, int world, int rank, int epoch, cudaStream_t st);
// training-mode pieces (train_kernels.cu): BatchNorm batch statistics / normalisation, MinibatchLayer forward
size_t bn_workspace_bytes(int c);
int launch_bn_batch_stats(const float* x, int n, int c, int hw, double* sum, double* sumsq, void* ws, cudaStream_t st);
int launch_bn_train_normalize(const float* x, int n, int c, int hw, const double* sum, const double* sumsq, double count,
                              const float* gamma, const float* beta, float eps, float alpha, float* running_mean,
                              float* running_inv_std, float* y, void* ws, cudaStream_t st);
size_t mb_workspace_bytes(int n, int K, int P);
int launch_minibatch_discrim(const float* x, int n, int d, const float* theta, const float* lws, const float* b, int K, int P,
                             float* out, void* ws, cudaStream_t st);
// pipelined all-gather: copy this rank's decoded shard (src, n_floats) into every peer's gather buffer from a small
// side-stream kernel + free/pushed flag handshake (see decout_tc.cu); returns after enqueueing push + wait kernels
int launch_peer_push(const float* src, float* const* dsts, float* const* flag_ptrs, long long n_floats, int world, int rank,
                     int step, int ctas, cudaStream_t st);
}  // namespace ian
