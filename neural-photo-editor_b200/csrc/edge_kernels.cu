// edge_kernels.cu -- the HBM-bound ends of the IAN graph and the small glue kernels.
//   conv1   : enc_conv1  3->128 ch 5x5 s2 + bias + LeakyReLU  (reference IAN_simple.py:73-83)
//   dec_out : dec_out    128->3 ch 5x5 s2 transposed conv + tanh (IAN_simple.py:171-181, layers.py:436-483)
//   latent  : GaussianSampleLayer (layers.py:419-433) and float32 <-> split-plane conversion of z
//   brush   : loss seed (API.py:59,64) fused with dec_out's backward-data and the bnorm_dc3*ReLU mask,
//             and the NPE step rule (NPE.py:199-209)
// These have K<=75 or N<=3: no tensor-core shape exists for them, they are written as FFMA kernels
// with smem-staged weights, vectorised channel-contiguous global access and one fused pass.
#include "edge.h"

namespace ian {

namespace {

__device__ __forceinline__ float lrelu02(float v) { return 0.6f * v + 0.4f * fabsf(v); }

// ------------------------------------------------------------------------------------------------
// conv1: x (n,3,64,64) fp32 NCHW -> out (n,32,32,128) split planes.
// block = one image x 8x8 output pixels; 256 threads = 32 groups of 4 output channels x 8 rows;
// a thread computes 8 pixels (one tile row) x 4 channels.  Weights [75][128] fp32 in smem.
// ------------------------------------------------------------------------------------------------
constexpr int C1_TILE = 8;
constexpr int C1_PATCH = 2 * C1_TILE + 3;   // 19

__global__ void __launch_bounds__(256) conv1_kernel(const float* __restrict__ x, const float* __restrict__ wt /*[75][128]*/,
                                                    const float* __restrict__ bias, __nv_bfloat16* __restrict__ out,
                                                    long long out_plane, int n_img) {
  __shared__ __align__(16) float Ws[75 * 128];
  __shared__ float Xs[3][C1_PATCH][C1_PATCH + 1];
  const int tid = threadIdx.x;
  const int tiles = 32 / C1_TILE;                 // 4 x 4 tiles per image
  const int img = blockIdx.x / (tiles * tiles);
  const int trow = (blockIdx.x / tiles) % tiles, tcol = blockIdx.x % tiles;
  const int oy0 = trow * C1_TILE, ox0 = tcol * C1_TILE;

  for (int i = tid; i < 75 * 128 / 4; i += 256)
    reinterpret_cast<float4*>(Ws)[i] = reinterpret_cast<const float4*>(wt)[i];
  for (int i = tid; i < 3 * C1_PATCH * C1_PATCH; i += 256) {
    int c = i / (C1_PATCH * C1_PATCH), r = (i / C1_PATCH) % C1_PATCH, cc = i % C1_PATCH;
    int iy = 2 * oy0 - 2 + r, ix = 2 * ox0 - 2 + cc;
    float v = 0.f;
    if (iy >= 0 && iy < 64 && ix >= 0 && ix < 64) v = x[((long long)(img * 3 + c) * 64 + iy) * 64 + ix];
    Xs[c][r][cc] = v;
  }
  __syncthreads();

  const int cg = tid & 31;        // channel group: channels 4*cg .. 4*cg+3
  const int py = tid >> 5;        // tile row 0..7
  float acc[C1_TILE][4];
#pragma unroll
  for (int p = 0; p < C1_TILE; ++p)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[p][j] = 0.f;

  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      float xr[C1_PATCH];
#pragma unroll
      for (int k = 0; k < C1_PATCH; ++k) xr[k] = Xs[c][2 * py + i][k];   // warp-uniform: broadcast
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const float4 w4 = *reinterpret_cast<const float4*>(&Ws[((c * 5 + i) * 5 + j) * 128 + cg * 4]);
#pragma unroll
        for (int p = 0; p < C1_TILE; ++p) {
          const float xv = xr[2 * p + j];
          acc[p][0] = fmaf(xv, w4.x, acc[p][0]);
          acc[p][1] = fmaf(xv, w4.y, acc[p][1]);
          acc[p][2] = fmaf(xv, w4.z, acc[p][2]);
          acc[p][3] = fmaf(xv, w4.w, acc[p][3]);
        }
      }
    }
  }
  const float4 b4 = *reinterpret_cast<const float4*>(bias + cg * 4);
  const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
  for (int p = 0; p < C1_TILE; ++p) {
    const long long pix = (long long)(img * 32 + oy0 + py) * 32 + ox0 + p;
    __align__(8) __nv_bfloat16 hi4[4], lo4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) split_bf16(lrelu02(acc[p][j] + bb[j]), hi4[j], lo4[j]);
    *reinterpret_cast<uint2*>(out + pix * 128 + cg * 4) = *reinterpret_cast<uint2*>(hi4);
    *reinterpret_cast<uint2*>(out + out_plane + pix * 128 + cg * 4) = *reinterpret_cast<uint2*>(lo4);
  }
}

// ------------------------------------------------------------------------------------------------
// dec_out: h3 (n,32,32,128) split planes -> x_hat (n,3,64,64) fp32 NCHW, tanh.
//   y[co, 2p+r, 2q+s] = sum_{d,e,ci} h3[p+d, q+e, ci] * W[ci][co][2+2d-r][2+2e-s]
// block = one image x 8x8 input pixels (-> 16x16 output pixels); warp w handles output phase
// (r,s) = (w>>1 & 1 ... ) so weight reads are warp-uniform broadcasts.
// smem: patch [10*10][128+4] fp32 (joined hi+lo), weights [25][128][4] fp32 (co padded to 4).
// ------------------------------------------------------------------------------------------------
constexpr int DO_T = 8, DO_P = DO_T + 2, DO_LD = 132;

__global__ void __launch_bounds__(256) dec_out_kernel(const __nv_bfloat16* __restrict__ h3, long long plane,
                                                      const float* __restrict__ wt /*[25][128][4]*/,
                                                      float* __restrict__ xhat, int n_img) {
  extern __shared__ __align__(16) float smem[];
  float* Xs = smem;                          // [100][132]
  float* Ws = smem + DO_P * DO_P * DO_LD;    // [25*128*4]
  const int tid = threadIdx.x;
  const int img = blockIdx.x >> 4;
  const int py0 = ((blockIdx.x >> 2) & 3) * DO_T, px0 = (blockIdx.x & 3) * DO_T;

  for (int i = tid; i < 25 * 128; i += 256)
    reinterpret_cast<float4*>(Ws)[i] = reinterpret_cast<const float4*>(wt)[i];
  // patch: 100 pixels x 128 channels, 4 channels per thread-iteration
  for (int i = tid; i < DO_P * DO_P * 32; i += 256) {
    const int pix = i >> 5, c4 = (i & 31) * 4;
    const int iy = py0 - 1 + pix / DO_P, ix = px0 - 1 + pix % DO_P;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (iy >= 0 && iy < 32 && ix >= 0 && ix < 32) {
      const __nv_bfloat16* src = h3 + ((long long)(img * 32 + iy) * 32 + ix) * 128 + c4;
      uint2 h = *reinterpret_cast<const uint2*>(src);
      uint2 l = *reinterpret_cast<const uint2*>(src + plane);
      const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&h);
      const __nv_bfloat162* lp = reinterpret_cast<const __nv_bfloat162*>(&l);
      float2 h0 = __bfloat1622float2(hp[0]), h1 = __bfloat1622float2(hp[1]);
      float2 l0 = __bfloat1622float2(lp[0]), l1 = __bfloat1622float2(lp[1]);
      v = make_float4(h0.x + l0.x, h0.y + l0.y, h1.x + l1.x, h1.y + l1.y);
    }
    *reinterpret_cast<float4*>(&Xs[pix * DO_LD + c4]) = v;
  }
  __syncthreads();

  const int warp = tid >> 5, lane = tid & 31;
  const int r = (warp >> 1) & 1, s = warp & 1;          // output phase of this warp
  const int half = warp >> 2;                           // which 32 of the 64 input pixels
  const int ip = half * 32 + lane;                      // input pixel 0..63
  const int p = ip >> 3, q = ip & 7;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
  // r=0: d in {-1,0,1} -> k = 2+2d ; r=1: d in {0,1} -> k = 1+2d
  const int dlo_r = r ? 0 : -1, dlo_s = s ? 0 : -1;
  for (int d = dlo_r; d <= 1; ++d) {
    const int ki = 2 + 2 * d - r;
    for (int e = dlo_s; e <= 1; ++e) {
      const int kj = 2 + 2 * e - s;
      const float* xp = &Xs[((p + d + 1) * DO_P + (q + e + 1)) * DO_LD];
      const float* wp = &Ws[(ki * 5 + kj) * 128 * 4];
#pragma unroll 8
      for (int ci = 0; ci < 128; ci += 4) {
        const float4 xv = *reinterpret_cast<const float4*>(xp + ci);
        const float4 w0 = *reinterpret_cast<const float4*>(wp + (ci + 0) * 4);
        const float4 w1 = *reinterpret_cast<const float4*>(wp + (ci + 1) * 4);
        const float4 w2 = *reinterpret_cast<const float4*>(wp + (ci + 2) * 4);
        const float4 w3 = *reinterpret_cast<const float4*>(wp + (ci + 3) * 4);
        a0 = fmaf(xv.x, w0.x, a0); a1 = fmaf(xv.x, w0.y, a1); a2 = fmaf(xv.x, w0.z, a2);
        a0 = fmaf(xv.y, w1.x, a0); a1 = fmaf(xv.y, w1.y, a1); a2 = fmaf(xv.y, w1.z, a2);
        a0 = fmaf(xv.z, w2.x, a0); a1 = fmaf(xv.z, w2.y, a1); a2 = fmaf(xv.z, w2.z, a2);
        a0 = fmaf(xv.w, w3.x, a0); a1 = fmaf(xv.w, w3.y, a1); a2 = fmaf(xv.w, w3.z, a2);
      }
    }
  }
  const int oy = 2 * (py0 + p) + r, ox = 2 * (px0 + q) + s;
  float* o = xhat + (long long)img * 3 * 4096 + oy * 64 + ox;
  o[0] = tanhf(a0);
  o[4096] = tanhf(a1);
  o[8192] = tanhf(a2);
}

// ------------------------------------------------------------------------------------------------
// latent glue
// ------------------------------------------------------------------------------------------------
// head (n,256) fp32: mu at [0,100), logsigma at [100,200) -> z fp32 (n,100) and split planes (n,128)
__global__ void sample_kernel(const float* __restrict__ head, const float* __restrict__ eps, float* __restrict__ z,
                              __nv_bfloat16* __restrict__ zp, long long zplane, int n) {
  pdl_trigger();
  pdl_wait();                                           // tapgemm.h: PDL
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 128) return;
  const int k = i / 128, j = i % 128;
  float v = 0.f;
  if (j < 100) {
    v = head[k * 256 + j];
    if (eps) v = fmaf(expf(head[k * 256 + 100 + j]), eps[k * 100 + j], v);
    if (z) z[k * 100 + j] = v;
  }
  if (zp) {
    __nv_bfloat16 hi, lo;
    split_bf16(v, hi, lo);
    zp[i] = hi;
    zp[zplane + i] = lo;
  }
}

// z fp32 (n,100) -> split planes (n,128), zero padded
__global__ void z_to_planes_kernel(const float* __restrict__ z, __nv_bfloat16* __restrict__ zp, long long zplane, int n) {
  pdl_trigger();
  pdl_wait();                                           // tapgemm.h: PDL
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 128) return;
  const int k = i / 128, j = i % 128;
  const float v = j < 100 ? z[k * 100 + j] : 0.f;
  __nv_bfloat16 hi, lo;
  split_bf16(v, hi, lo);
  zp[i] = hi;
  zp[zplane + i] = lo;
}

// ------------------------------------------------------------------------------------------------
// brush: loss seed + dec_out backward-data + bnorm_dc3 scale * ReLU mask, fused.
//   seed[k,co,u,v] = coef * (x_hat - t) * (1 - x_hat^2)  inside box_k (coef = 2/(3*bh*bw)), or
//                    (1/(3*bh*bw)) * (1 - x_hat^2) for the lighten gradient           (API.py:59,64)
//   d3[k,a,b,ci]   = scale3[ci] * (h3[k,a,b,ci] > 0) * sum_{co,ki,kj} seed[k,co,2+2a-ki,2+2b-kj] * W[ci][co][ki][kj]
// One block per (sample k, feature-map row a), 8 warps; lane l owns channels 4l..4l+3, warp w the pixel pairs
// (2j, 2j+1), j = w, w+8.  Only rows / pixels within reach of the box (2a-2 < r2 && 2a+2 >= r1, same for columns: at
// most 11 x 11 of the 32 x 32 map for NPE's <= 17-pixel brush) do any work: the block stages the 5 seed rows it can touch
// in shared memory (zero outside the box), every in-reach pixel pair walks the valid taps with warp-uniform control flow
// (a warp is one pixel pair), and everything else is a coalesced zero fill that does not even read h3.  (Round 2's first
// form ran one thread per (pixel, 4 channels) over the whole map: 104 us at batch 128, 12 % of an edit step.)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) brush_seed_bwd_kernel(const float* __restrict__ xhat, const int32_t* __restrict__ boxes,
                                                             const float* __restrict__ target, int target_is_frame,
                                                             const float* __restrict__ wt /*[25][128][4]*/,
                                                             const float* __restrict__ scale3,
                                                             const __nv_bfloat16* __restrict__ h3,
                                                             __nv_bfloat16* __restrict__ d3, long long plane, int n) {
  pdl_trigger();
  pdl_wait();                                           // tapgemm.h: PDL
  __shared__ float sd[3 * 5 * 68];                       // [co][row 2a-2 .. 2a+2][col -2 .. 65]
  __shared__ __align__(16) float ws[25 * 3 * 128];       // dec_out weights of the valid kernel rows, [tap][co][ci] (in-reach rows only)
  const int k = blockIdx.x >> 5, a = blockIdx.x & 31;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // device-resident boxes cannot be validated on the host: clamp to the frame here (never read outside x_hat); an
  // empty box contributes nothing and brush_update_kernel turns its gradient into NaN (mean over an empty slice)
  const int c1 = max(boxes[k * 4 + 0], 0), r1 = max(boxes[k * 4 + 1], 0);
  const int c2 = min(boxes[k * 4 + 2], 64), r2 = min(boxes[k * 4 + 3], 64);
  const long long row_off = (long long)(k * 32 + a) * 32 * 128;   // this row of the map: 32 pixels x 128 channels
  // rows u = 2+2a-ki, ki in 0..4  ->  u in [2a-2, 2a+2]
  const bool row_reach = r1 < r2 && c1 < c2 && 2 * a + 2 >= r1 && 2 * a - 2 < r2;
  if (!row_reach) {                                      // 8 KB per plane = 512 uint4
    const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
    uint4* oh = reinterpret_cast<uint4*>(d3 + row_off);
    uint4* ol = reinterpret_cast<uint4*>(d3 + plane + row_off);
    oh[threadIdx.x] = z4; oh[threadIdx.x + 256] = z4;
    ol[threadIdx.x] = z4; ol[threadIdx.x + 256] = z4;
    return;
  }
  const float inv = 1.f / (3.f * (float)(r2 - r1) * (float)(c2 - c1));
  for (int i = threadIdx.x; i < 3 * 5 * 68; i += 256) {
    const int co = i / 340, rem = i % 340;
    const int u = 2 * a - 2 + rem / 68, v = rem % 68 - 2;
    float sdv = 0.f;
    if (u >= r1 && u < r2 && v >= c1 && v < c2) {
      const long long xi = ((long long)(k * 3 + co) * 64 + u) * 64 + v;
      const float xv = xhat[xi];
      if (target) {
        const float t = target_is_frame ? target[xi] : target[k * 3 + co];
        sdv = 2.f * inv * (xv - t);
      } else {
        sdv = inv;
      }
      sdv *= (1.f - xv * xv);
    }
    sd[i] = sdv;
  }
  // weights through shared memory: every in-reach pixel walks up to the whole 38 KB table, and from L1/L2 each tap was a
  // dependent round trip (the first block-per-row form spent 60 % of its samples there: 32 us for the launch)
  for (int i = threadIdx.x; i < 25 * 128; i += 256) {
    const int tap = i >> 7, ch = i & 127;
    const int u = 2 + 2 * a - tap / 5;
    if (u < r1 || u >= r2) continue;                      // (block-uniform per tap row)
    const float4 w4 = __ldg(reinterpret_cast<const float4*>(wt) + i);
    ws[(tap * 3 + 0) * 128 + ch] = w4.x;
    ws[(tap * 3 + 1) * 128 + ch] = w4.y;
    ws[(tap * 3 + 2) * 128 + ch] = w4.z;
  }
  __syncthreads();
  const float4 sc = *reinterpret_cast<const float4*>(scale3 + lane * 4);
  for (int j = warp; j < 16; j += 8) {
    const int b0 = 2 * j;
    const bool reach0 = 2 * b0 + 2 >= c1 && 2 * b0 - 2 < c2;
    const bool reach1 = 2 * b0 + 4 >= c1 && 2 * b0 < c2;
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    if (reach0 || reach1) {
      for (int ki = 0; ki < 5; ++ki) {
        const int u = 2 + 2 * a - ki;
        if (u < r1 || u >= r2) continue;
        const float* srow = sd + (4 - ki) * 68;
        for (int kj = 0; kj < 5; ++kj) {
          const int v0 = 2 + 2 * b0 - kj;                 // pixel b0 reads column v0, pixel b0+1 column v0+2
          if ((v0 < c1 || v0 >= c2) && (v0 + 2 < c1 || v0 + 2 >= c2)) continue;
          const float* wp = ws + (ki * 5 + kj) * 3 * 128 + lane * 4;
          const float4 w0 = *reinterpret_cast<const float4*>(wp);          // co = 0, channels 4l .. 4l+3
          const float4 w1 = *reinterpret_cast<const float4*>(wp + 128);    // co = 1
          const float4 w2 = *reinterpret_cast<const float4*>(wp + 256);    // co = 2
          const float wa[4] = {w0.x, w0.y, w0.z, w0.w}, wb[4] = {w1.x, w1.y, w1.z, w1.w}, wc[4] = {w2.x, w2.y, w2.z, w2.w};
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const float s0 = srow[v0 + 2 + 2 * q], s1 = srow[340 + v0 + 2 + 2 * q], s2 = srow[680 + v0 + 2 + 2 * q];
#pragma unroll
            for (int c = 0; c < 4; ++c) {                 // per channel: co = 0, 1, 2 in this order (as the first form)
              acc[q][c] = fmaf(s0, wa[c], acc[q][c]);
              acc[q][c] = fmaf(s1, wb[c], acc[q][c]);
              acc[q][c] = fmaf(s2, wc[c], acc[q][c]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const long long off = row_off + (long long)(b0 + q) * 128 + lane * 4;
      uint2 hv = make_uint2(0u, 0u), lv = make_uint2(0u, 0u);
      if (q ? reach1 : reach0) {
        const uint2 mraw = *reinterpret_cast<const uint2*>(h3 + off);
        const __nv_bfloat16* mk = reinterpret_cast<const __nv_bfloat16*>(&mraw);
        const float scv[4] = {sc.x, sc.y, sc.z, sc.w};
        __align__(8) __nv_bfloat16 hi4[4], lo4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float v = __bfloat162float(mk[c]) > 0.f ? acc[q][c] * scv[c] : 0.f;
          split_bf16(v, hi4[c], lo4[c]);
        }
        hv = *reinterpret_cast<uint2*>(hi4);
        lv = *reinterpret_cast<uint2*>(lo4);
      }
      *reinterpret_cast<uint2*>(d3 + off) = hv;
      *reinterpret_cast<uint2*>(d3 + plane + off) = lv;
    }
  }
}

// g fp32 (n,128 padded) -> user g (n,100) and/or z update  z <- z - weight*g*(1+c2-c1)  (NPE.py:206-209)
__global__ void brush_update_kernel(const float* __restrict__ gpad, const int32_t* __restrict__ boxes, float weight,
                                    float* __restrict__ g_out, float* __restrict__ z, __nv_bfloat16* __restrict__ zp,
                                    long long zplane, int n) {
  pdl_trigger();
  pdl_wait();                                           // tapgemm.h: PDL
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 128) return;
  const int k = i / 128, j = i % 128;
  float zv = 0.f;
  if (j < 100) {
    const int bc1 = max(boxes[k * 4 + 0], 0), br1 = max(boxes[k * 4 + 1], 0);
    const int bc2 = min(boxes[k * 4 + 2], 64), br2 = min(boxes[k * 4 + 3], 64);
    const float gv = (bc1 < bc2 && br1 < br2) ? gpad[i] : __int_as_float(0x7fc00000);   // empty box: NaN, as the reference
    if (g_out) g_out[k * 100 + j] = gv;
    if (z) {
      const float fac = 1.f + (float)(boxes[k * 4 + 2] - boxes[k * 4 + 0]);
      const float grad = gv * fac;                       // NPE.py:206  grad = temp*(1+(x2-x1))
      zv = z[k * 100 + j] - weight * grad;               // NPE.py:209  Z -= weight*grad
      z[k * 100 + j] = zv;
    }
  }
  if (z && zp) {
    __nv_bfloat16 hi, lo;
    split_bf16(zv, hi, lo);
    zp[i] = hi;
    zp[zplane + i] = lo;
  }
}

// ------------------------------------------------------------------------------------------------
// full IAN latent: z = (z0 - MADE_mu(z0)) / exp(MADE_ls(z0))     (reference IAN.py:126-128; layers.py:641-853)
//   MADE(z) = core(in(z)),  in(v) = relu(v (W0*M0) + b0),  core(u) = in(u) (W1*M1) + b1 + u (Wd*Md) + bd
//   (the input MaskedLayer runs twice: see below); the masks are pre-multiplied on the host
// mw: [2 nets][3 matrices: input, output_W, output_D][100][100] fp32 (in,out); mb: [2][3][100].
// one block per sample, 128 threads.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) made_iaf_kernel(const float* __restrict__ z0, const float* __restrict__ mw,
                                                       const float* __restrict__ mb, float* __restrict__ z,
                                                       __nv_bfloat16* __restrict__ zp, long long zplane, int n) {
  pdl_trigger();
  pdl_wait();                                           // tapgemm.h: PDL
  __shared__ float zs[100];
  __shared__ float us[2][100];
  __shared__ float hs[2][100];
  const int k = blockIdx.x, j = threadIdx.x;
  if (j < 100) zs[j] = z0[k * 100 + j];
  __syncthreads();
  // u = relu(z W0 + b0): the `<name>_input` MaskedLayer.  MADE.__init__ (layers.py:769) overwrites Layer.input_layer
  // with it, so inside the reference graph the MADE layer is fed u, not z, and applies its whole stack to u.
  if (j < 100) {
#pragma unroll
    for (int net = 0; net < 2; ++net) {
      const float* W0 = mw + (net * 3 + 0) * 10000;
      float a = mb[(net * 3 + 0) * 100 + j];
      for (int i = 0; i < 100; ++i) a = fmaf(zs[i], W0[i * 100 + j], a);
      us[net][j] = 0.5f * (a + fabsf(a));
    }
  }
  __syncthreads();
  if (j < 100) {
#pragma unroll
    for (int net = 0; net < 2; ++net) {
      const float* W0 = mw + (net * 3 + 0) * 10000;
      float a = mb[(net * 3 + 0) * 100 + j];
      for (int i = 0; i < 100; ++i) a = fmaf(us[net][i], W0[i * 100 + j], a);
      hs[net][j] = 0.5f * (a + fabsf(a));
    }
  }
  __syncthreads();
  float out = 0.f;
  if (j < 100) {
    float o[2];
#pragma unroll
    for (int net = 0; net < 2; ++net) {
      const float* W1 = mw + (net * 3 + 1) * 10000;
      const float* Wd = mw + (net * 3 + 2) * 10000;
      float a = mb[(net * 3 + 1) * 100 + j] + mb[(net * 3 + 2) * 100 + j];
      float a1 = 0.f, a2 = 0.f;
      for (int i = 0; i < 100; ++i) {
        a1 = fmaf(hs[net][i], W1[i * 100 + j], a1);
        a2 = fmaf(us[net][i], Wd[i * 100 + j], a2);
      }
      o[net] = a + a1 + a2;
    }
    out = (zs[j] - o[0]) / expf(o[1]);                   // IAFLayer (layers.py:649)
    if (z) z[k * 100 + j] = out;
  }
  if (zp) {
    __nv_bfloat16 hi, lo;
    split_bf16(j < 100 ? out : 0.f, hi, lo);
    zp[k * 128 + j] = hi;
    zp[zplane + k * 128 + j] = lo;
  }
}

// ------------------------------------------------------------------------------------------------
// full IAN RGB-Beta head (reference IAN.py:183-207; layers.py:397-408).  ha (n,64,64,16) fp32 holds the three
// 128->2 MDC convolutions of the feature map: [R | G_a | B_a | pad].  The autoregressive parts are 2->2 and
// 4->2 channel MDC convolutions over 33 dilated taps: a few hundred MACs per pixel, done per pixel here.
//   R = sig(ha[0:2]);  G = sig(ha[2:4] + MDC_Gb(R));  B = sig(ha[4:6] + MDC_Bb([R,G]));
//   out_c = 2 a/(a+b+1e-8) - 1
// taps: [33][2] int (dy,dx);  wgb: [33][2 out][2 in];  wbb: [33][2 out][4 in]   (composite MDC weights)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// tt: tap table of one dense GEMM (no shifts), tile-blocked: tt[(n*32 + p/2)][t*6+f][(p%2)*64 + q] =
//     sum_c h[n,p,q,c] * Wc[t][f][c]       (a tile = 2 image rows, see TapGemm::out_f32_t)
// ha[pix][f] = sum_t tt[..pix + (dy_t, dx_t)..][t*6+f]  -- the 33 dilated taps become 33 coalesced shifted reads.
template <typename T> __device__ __forceinline__ float tt_load(const T* p);
template <> __device__ __forceinline__ float tt_load<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float tt_load<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(__ushort_as_bfloat16(__ldg(reinterpret_cast<const unsigned short*>(p))));
}

template <typename T>
__global__ void __launch_bounds__(256) head_gather_kernel(const T* __restrict__ tt, const int* __restrict__ taps, int ntaps,
                                                          float* __restrict__ ha, int n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * 4096) return;
  const int q = (int)(i & 63), p = (int)((i >> 6) & 63);
  const long long img = i >> 12;
  const int ncol = ntaps * 6;
  float a[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int t = 0; t < ntaps; ++t) {
    const int pp = p + taps[2 * t], qq = q + taps[2 * t + 1];
    if (pp < 0 || pp > 63 || qq < 0 || qq > 63) continue;
    const T* src = tt + ((img * 32 + (pp >> 1)) * ncol + t * 6) * 128 + (pp & 1) * 64 + qq;
#pragma unroll
    for (int f = 0; f < 6; ++f) a[f] += tt_load<T>(src + f * 128);
  }
  float* o = ha + i * 16;
  *reinterpret_cast<float4*>(o) = make_float4(a[0], a[1], a[2], a[3]);
  *reinterpret_cast<float2*>(o + 4) = make_float2(a[4], a[5]);
}

// ha layouts: interleaved (n,64,64,16) from head_gather (verification path) or planar [n][6][4096] from head_tc_kernel
__device__ __forceinline__ float2 ha_pair(const float* __restrict__ ha, long long i, int c, int planar) {
  if (!planar) return *reinterpret_cast<const float2*>(ha + i * 16 + c);
  const float* p = ha + ((i >> 12) * 6 + c) * 4096 + (i & 4095);
  return make_float2(__ldg(p), __ldg(p + 4096));
}

__global__ void head_r_kernel(const float* __restrict__ ha, int planar, float* __restrict__ rg, long long npix) {
  pdl_trigger();
  pdl_wait();                                           // tapgemm.h: PDL
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const float2 a = ha_pair(ha, i, 0, planar);
  float4 o = make_float4(sigmoidf_(a.x), sigmoidf_(a.y), 0.f, 0.f);
  *reinterpret_cast<float4*>(rg + i * 4) = o;            // rg: (n,64,64,4) = [R0,R1,G0,G1]
}

// The tap offsets and the 2x2 / 4x2 weights of the autoregressive convolutions are the same for every pixel: staged in
// shared memory once per block (constants: before the PDL wait).  Read per tap from global memory they were 4-6 of the 7
// loads of an iteration and the L1 path was the bound (ncu: "Mem Busy 92 %", L1 hit rate 89 %, 121 us for head_b_out at
// batch 512); now an iteration is two broadcast LDS + the one neighbour load that really differs per pixel.
constexpr int kHeadMaxTaps = 48;

__global__ void head_g_kernel(const float* __restrict__ ha, int planar, float* __restrict__ rg, const int* __restrict__ taps,
                              const float* __restrict__ wgb, int ntaps, int n) {
  __shared__ int s_taps[2 * kHeadMaxTaps];
  __shared__ __align__(16) float s_w[4 * kHeadMaxTaps];
  pdl_trigger();
  for (int j = threadIdx.x; j < 2 * ntaps; j += blockDim.x) s_taps[j] = taps[j];
  for (int j = threadIdx.x; j < 4 * ntaps; j += blockDim.x) s_w[j] = wgb[j];
  __syncthreads();
  pdl_wait();                                           // tapgemm.h: PDL
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * 4096) return;
  const int q = (int)(i & 63), p = (int)((i >> 6) & 63);
  const long long img = i >> 12;
  const float2 gin = ha_pair(ha, i, 2, planar);
  float g0 = gin.x, g1 = gin.y;
  for (int t = 0; t < ntaps; ++t) {
    const int pp = p + s_taps[2 * t], qq = q + s_taps[2 * t + 1];
    if (pp < 0 || pp > 63 || qq < 0 || qq > 63) continue;
    const float2 r = *reinterpret_cast<const float2*>(rg + ((img * 64 + pp) * 64 + qq) * 4);
    const float4 w = *reinterpret_cast<const float4*>(s_w + t * 4);     // [out0: in0,in1 | out1: in0,in1]
    g0 = fmaf(r.x, w.x, fmaf(r.y, w.y, g0));
    g1 = fmaf(r.x, w.z, fmaf(r.y, w.w, g1));
  }
  *reinterpret_cast<float2*>(rg + i * 4 + 2) = make_float2(sigmoidf_(g0), sigmoidf_(g1));
}

__global__ void head_b_out_kernel(const float* __restrict__ ha, int planar, const float* __restrict__ rg, const int* __restrict__ taps,
                                  const float* __restrict__ wbb, int ntaps, const __grid_constant__ DecOutDst dst,
                                  float* __restrict__ bsave /*nullable: (n,64,64,2) = B, kept for the brush backward*/, int n) {
  __shared__ int s_taps[2 * kHeadMaxTaps];
  __shared__ __align__(16) float s_w[8 * kHeadMaxTaps];
  pdl_trigger();
  for (int j = threadIdx.x; j < 2 * ntaps; j += blockDim.x) s_taps[j] = taps[j];
  for (int j = threadIdx.x; j < 8 * ntaps; j += blockDim.x) s_w[j] = wbb[j];
  __syncthreads();
  pdl_wait();                                           // tapgemm.h: PDL
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * 4096) return;
  const int q = (int)(i & 63), p = (int)((i >> 6) & 63);
  const long long img = i >> 12;
  const float2 bin = ha_pair(ha, i, 4, planar);
  float b0 = bin.x, b1 = bin.y;
  for (int t = 0; t < ntaps; ++t) {
    const int pp = p + s_taps[2 * t], qq = q + s_taps[2 * t + 1];
    if (pp < 0 || pp > 63 || qq < 0 || qq > 63) continue;
    const float4 v = *reinterpret_cast<const float4*>(rg + ((img * 64 + pp) * 64 + qq) * 4);
    const float4 w0 = *reinterpret_cast<const float4*>(s_w + t * 8);
    const float4 w1 = *reinterpret_cast<const float4*>(s_w + t * 8 + 4);
    b0 = fmaf(v.x, w0.x, fmaf(v.y, w0.y, fmaf(v.z, w0.z, fmaf(v.w, w0.w, b0))));
    b1 = fmaf(v.x, w1.x, fmaf(v.y, w1.y, fmaf(v.z, w1.z, fmaf(v.w, w1.w, b1))));
  }
  const float4 me = *reinterpret_cast<const float4*>(rg + i * 4);
  const float B0 = sigmoidf_(b0), B1 = sigmoidf_(b1);
  if (bsave) *reinterpret_cast<float2*>(bsave + i * 2) = make_float2(B0, B1);
  const float y0 = 2.f * (me.x / (me.x + me.y + 1e-8f)) - 1.f;     // beta_layer (layers.py:408)
  const float y1 = 2.f * (me.z / (me.z + me.w + 1e-8f)) - 1.f;
  const float y2 = 2.f * (B0 / (B0 + B1 + 1e-8f)) - 1.f;
  const long long off = img * 3 * 4096 + p * 64 + q;
  for (int d = 0; d < dst.n; ++d) {                     // d > 0: peer GPUs' gather buffers (st.global over NVLink)
    float* o = dst.base[d] + off;
    o[0] = y0;
    o[4096] = y1;
    o[8192] = y2;
  }
}

// ------------------------------------------------------------------------------------------------
// NPE photo-mode blend after a paint stroke (reference NPE.py:218-231), one 64x64 image, one block:
//   DELTA = x_hat - to_tanh(RECON);  M = min(mean_c |DELTA|, 1);  MASK = gaussian_filter(M, sigma=0.7)
//   D = MASK*DELTA + (1-MASK)*ERROR;  IM = uint8(from_tanh(to_tanh(RECON) + D))
// gaussian_filter = scipy.ndimage: separable, radius int(4*0.7+0.5) = 3, weights exp(-k^2/(2 sigma^2)) normalised,
// boundary mode 'reflect' (d c b a | a b c d | d c b a), axis 0 then axis 1.
// Also writes the 4x nearest-neighbour upsampled display image (NPE.py:107-118) as HWC uint8 (256,256,3).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect64(int i) { return i < 0 ? -i - 1 : (i > 63 ? 127 - i : i); }

__global__ void __launch_bounds__(1024) npe_blend_kernel(const float* __restrict__ xhat, const uint8_t* __restrict__ recon,
                                                         const float* __restrict__ error, uint8_t* __restrict__ im,
                                                         uint8_t* __restrict__ display) {
  __shared__ float M[64][65], T[64][65];
  __shared__ float wk[4];
  const int tid = threadIdx.x;
  if (tid == 0) {
    float w[4], sum = 0.f;
    for (int k = 0; k < 4; ++k) { w[k] = expf(-0.5f * (float)(k * k) / (0.7f * 0.7f)); sum += (k == 0 ? w[k] : 2.f * w[k]); }
    for (int k = 0; k < 4; ++k) wk[k] = w[k] / sum;
  }
  for (int i = tid; i < 4096; i += 1024) {
    float m = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float rt = 2.0f * ((float)recon[c * 4096 + i] / 255.0f) - 1.0f;       // to_tanh (NPE.py:37-38)
      m += fabsf(xhat[c * 4096 + i] - rt);
    }
    M[i >> 6][i & 63] = fminf(m / 3.f, 1.f);
  }
  __syncthreads();
  for (int i = tid; i < 4096; i += 1024) {                // axis 0 (rows)
    const int r = i >> 6, c = i & 63;
    float a = wk[0] * M[r][c];
#pragma unroll
    for (int k = 1; k < 4; ++k) a += wk[k] * (M[reflect64(r - k)][c] + M[reflect64(r + k)][c]);
    T[r][c] = a;
  }
  __syncthreads();
  for (int i = tid; i < 4096; i += 1024) {                // axis 1 (columns) + blend
    const int r = i >> 6, c = i & 63;
    float mask = wk[0] * T[r][c];
#pragma unroll
    for (int k = 1; k < 4; ++k) mask += wk[k] * (T[r][reflect64(c - k)] + T[r][reflect64(c + k)]);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float rt = 2.0f * ((float)recon[ch * 4096 + i] / 255.0f) - 1.0f;
      const float delta = xhat[ch * 4096 + i] - rt;
      const float d = mask * delta + (1.f - mask) * error[ch * 4096 + i];
      float v = 255.0f * ((rt + d) + 1.f) / 2.0f;                                // from_tanh (NPE.py:40-41)
      v = fminf(fmaxf(v, 0.f), 255.f);
      const uint8_t u = (uint8_t)v;                                              // np.uint8 truncates
      im[ch * 4096 + i] = u;
#pragma unroll
      for (int dy = 0; dy < 4; ++dy)
#pragma unroll
        for (int dx = 0; dx < 4; ++dx) display[((4 * r + dy) * 256 + 4 * c + dx) * 3 + ch] = u;
    }
  }
}

}  // namespace

#define CHECK_LAUNCH() (cudaGetLastError() == cudaSuccess ? 1 : -1)

int launch_conv1(const float* x, const float* wt, const float* bias, __nv_bfloat16* out, long long plane, int n,
                 cudaStream_t st) {
  conv1_kernel<<<n * 16, 256, 0, st>>>(x, wt, bias, out, plane, n);
  return CHECK_LAUNCH();
}

int dec_out_smem_bytes() { return (DO_P * DO_P * DO_LD + 25 * 128 * 4) * (int)sizeof(float); }

int launch_dec_out(const __nv_bfloat16* h3, long long plane, const float* wt, float* xhat, int n, cudaStream_t st) {
  static DeviceOnce attr_set;
  const int dev = cur_device();
  if (!attr_set.is_done(dev)) {
    if (cudaFuncSetAttribute(dec_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dec_out_smem_bytes()) != cudaSuccess) return -1;
    attr_set.set_done(dev);
  }
  dec_out_kernel<<<n * 16, 256, dec_out_smem_bytes(), st>>>(h3, plane, wt, xhat, n);
  return CHECK_LAUNCH();
}

int launch_sample(const float* head, const float* eps, float* z, __nv_bfloat16* zp, long long zplane, int n,
                  cudaStream_t st) {
  if (launch_pdl(sample_kernel, dim3((n * 128 + 255) / 256), dim3(256), 0, st, head, eps, z, zp, zplane, n) != cudaSuccess) return -1;
  return CHECK_LAUNCH();
}

int launch_z_to_planes(const float* z, __nv_bfloat16* zp, long long zplane, int n, cudaStream_t st) {
  if (launch_pdl(z_to_planes_kernel, dim3((n * 128 + 255) / 256), dim3(256), 0, st, z, zp, zplane, n) != cudaSuccess) return -1;
  return CHECK_LAUNCH();
}

int launch_brush_seed_bwd(const float* xhat, const int32_t* boxes, const float* target, int target_is_frame,
                          const float* wt, const float* scale3, const __nv_bfloat16* h3, __nv_bfloat16* d3,
                          long long plane, int n, cudaStream_t st) {
  if (launch_pdl(brush_seed_bwd_kernel, dim3((unsigned)n * 32u), dim3(256), 0, st, xhat, boxes, target, target_is_frame, wt, scale3, h3, d3, plane, n) != cudaSuccess) return -1;
  return CHECK_LAUNCH();
}

int launch_brush_update(const float* gpad, const int32_t* boxes, float weight, float* g_out, float* z,
                        __nv_bfloat16* zp, long long zplane, int n, cudaStream_t st) {
  if (launch_pdl(brush_update_kernel, dim3((n * 128 + 255) / 256), dim3(256), 0, st, gpad, boxes, weight, g_out, z, zp, zplane, n) != cudaSuccess) return -1;
  return CHECK_LAUNCH();
}

}  // namespace ian

namespace ian {
int launch_npe_blend(const float* xhat, const uint8_t* recon, const float* error, uint8_t* im, uint8_t* display, cudaStream_t st) {
  npe_blend_kernel<<<1, 1024, 0, st>>>(xhat, recon, error, im, display);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_made_iaf(const float* z0, const float* mw, const float* mb, float* z, __nv_bfloat16* zp, long long zplane, int n,
                    cudaStream_t st) {
  if (launch_pdl(made_iaf_kernel, dim3(n), dim3(128), 0, st, z0, mw, mb, z, zp, zplane, n) != cudaSuccess) return -1;
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_head_gather(const float* tt, int tt_is_bf16, const int* taps, int ntaps, float* ha, int n, cudaStream_t st) {
  const long long npix = (long long)n * 4096;
  if (tt_is_bf16)
    head_gather_kernel<__nv_bfloat16><<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(tt), taps, ntaps, ha, n);
  else
    head_gather_kernel<float><<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(tt, taps, ntaps, ha, n);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_rgb_beta_head(const float* ha, int ha_planar, float* rg, const int* taps, const float* wgb, const float* wbb, int ntaps,
                         float* const* dsts, int ndst, float* bsave, int n, cudaStream_t st) {
  const long long npix = (long long)n * 4096;
  const unsigned blocks = (unsigned)((npix + 255) / 256);
  if (ntaps > kHeadMaxTaps) return -1;
  if (ndst < 1 || ndst > kMaxPeers) return -1;
  DecOutDst dst;
  dst.n = ndst;
  for (int d = 0; d < ndst; ++d) dst.base[d] = dsts[d];
  if (launch_pdl(head_r_kernel, dim3(blocks), dim3(256), 0, st, ha, ha_planar, rg, npix) != cudaSuccess) return -1;
  if (launch_pdl(head_g_kernel, dim3(blocks), dim3(256), 0, st, ha, ha_planar, rg, taps, wgb, ntaps, n) != cudaSuccess) return -1;
  if (launch_pdl(head_b_out_kernel, dim3(blocks), dim3(256), 0, st, ha, ha_planar, rg, taps, wbb, ntaps, dst, bsave, n) != cudaSuccess) return -1;
  return cudaGetLastError() == cudaSuccess ? 3 : -1;
}

// ------------------------------------------------------------------------------------------------
// Brush gradient through the RGB-Beta head (T.grad of API.py:59,64 on the IAN.py / IANv1.py graphs; forward:
// IAN.py:183-207, layers.py:397-408).  dpre (n,64,64,8) float32 ends up holding d loss / d [preR0 preR1 preG0 preG1 preB0
// preB1 . .] -- the gradient w.r.t. the three 128->2 MDC convolutions of the feature map -- in three passes that
// mirror the autoregressive forward in reverse (B, then G, then R):
//   seed : dL/dx_hat over the brush box (lighten: 1/(3 bh bw); RGB: 2 (x_hat - t)/(3 bh bw)), beta_layer backward
//          d out/d a = 2 (b + eps)/(a+b+eps)^2, d out/d b = -2 a/(a+b+eps)^2, and dpreB = dB * B (1-B)
//   g    : d[R,G] += MDC_Bb^T(dpreB)   (33 dilated taps, 2 -> 4 channels);  dpreG = dG * G (1-G)
//   r    : dR     += MDC_Gb^T(dpreG)   (2 -> 2 channels);                   dpreR = dR * R (1-R)
// and im2col lays dpre out as the K = 33 taps x 6 operand of the dense backward GEMM (dh = A2 * Wcomp).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) head_bwd_seed_kernel(const float* __restrict__ xhat, const float* __restrict__ rg,
                                                            const float* __restrict__ bsave, const int32_t* __restrict__ boxes,
                                                            const float* __restrict__ target, int target_is_frame,
                                                            float* __restrict__ dpre, int n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * 4096) return;
  const int q = (int)(i & 63), p = (int)((i >> 6) & 63);
  const int k = (int)(i >> 12);
  const int c1 = max(boxes[k * 4 + 0], 0), r1 = max(boxes[k * 4 + 1], 0);
  const int c2 = min(boxes[k * 4 + 2], 64), r2 = min(boxes[k * 4 + 3], 64);
  float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (p >= r1 && p < r2 && q >= c1 && q < c2) {
    const float inv = 1.f / (3.f * (float)(r2 - r1) * (float)(c2 - c1));
    const float4 rgv = *reinterpret_cast<const float4*>(rg + i * 4);
    const float2 bv = *reinterpret_cast<const float2*>(bsave + i * 2);
    const float a[3] = {rgv.x, rgv.z, bv.x}, b[3] = {rgv.y, rgv.w, bv.y};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float xv = xhat[((long long)(k * 3 + c) * 64 + p) * 64 + q];
      float sd = inv;
      if (target) {
        const float t = target_is_frame ? target[((long long)(k * 3 + c) * 64 + p) * 64 + q] : target[k * 3 + c];
        sd = 2.f * inv * (xv - t);
      }
      const float s = a[c] + b[c] + 1e-8f;
      o[2 * c] = sd * 2.f * (b[c] + 1e-8f) / (s * s);
      o[2 * c + 1] = -sd * 2.f * a[c] / (s * s);
    }
    o[4] *= bv.x * (1.f - bv.x);                         // dpreB
    o[5] *= bv.y * (1.f - bv.y);
  }
  float4* dp = reinterpret_cast<float4*>(dpre + i * 8);
  dp[0] = make_float4(o[0], o[1], o[2], o[3]);
  dp[1] = make_float4(o[4], o[5], 0.f, 0.f);
}

__global__ void __launch_bounds__(256) head_bwd_g_kernel(float* __restrict__ dpre, const float* __restrict__ rg,
                                                         const int* __restrict__ taps, const float* __restrict__ wbb, int ntaps, int n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * 4096) return;
  const int q = (int)(i & 63), p = (int)((i >> 6) & 63);
  const long long img = i >> 12;
  float d[4] = {0.f, 0.f, 0.f, 0.f};
  for (int t = 0; t < ntaps; ++t) {                      // forward read (p + off): the transpose reads (p - off)
    const int pp = p - taps[2 * t], qq = q - taps[2 * t + 1];
    if (pp < 0 || pp > 63 || qq < 0 || qq > 63) continue;
    const float2 g = *reinterpret_cast<const float2*>(dpre + ((img * 64 + pp) * 64 + qq) * 8 + 4);   // dpreB of the reader
    const float4 w0 = *reinterpret_cast<const float4*>(wbb + t * 8);       // out 0: in 0..3
    const float4 w1 = *reinterpret_cast<const float4*>(wbb + t * 8 + 4);   // out 1: in 0..3
    d[0] = fmaf(g.x, w0.x, fmaf(g.y, w1.x, d[0]));
    d[1] = fmaf(g.x, w0.y, fmaf(g.y, w1.y, d[1]));
    d[2] = fmaf(g.x, w0.z, fmaf(g.y, w1.z, d[2]));
    d[3] = fmaf(g.x, w0.w, fmaf(g.y, w1.w, d[3]));
  }
  float4 own = *reinterpret_cast<const float4*>(dpre + i * 8);
  const float4 rgv = *reinterpret_cast<const float4*>(rg + i * 4);
  own.x += d[0];
  own.y += d[1];
  own.z = (own.z + d[2]) * rgv.z * (1.f - rgv.z);        // dpreG
  own.w = (own.w + d[3]) * rgv.w * (1.f - rgv.w);
  *reinterpret_cast<float4*>(dpre + i * 8) = own;        // slots 0..3 only: the neighbours read slots 4,5
}

__global__ void __launch_bounds__(256) head_bwd_r_kernel(float* __restrict__ dpre, const float* __restrict__ rg,
                                                         const int* __restrict__ taps, const float* __restrict__ wgb, int ntaps, int n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * 4096) return;
  const int q = (int)(i & 63), p = (int)((i >> 6) & 63);
  const long long img = i >> 12;
  float d0 = 0.f, d1 = 0.f;
  for (int t = 0; t < ntaps; ++t) {
    const int pp = p - taps[2 * t], qq = q - taps[2 * t + 1];
    if (pp < 0 || pp > 63 || qq < 0 || qq > 63) continue;
    const float2 g = *reinterpret_cast<const float2*>(dpre + ((img * 64 + pp) * 64 + qq) * 8 + 2);   // dpreG of the reader
    const float4 w = *reinterpret_cast<const float4*>(wgb + t * 4);        // [out0: in0,in1 | out1: in0,in1]
    d0 = fmaf(g.x, w.x, fmaf(g.y, w.z, d0));
    d1 = fmaf(g.x, w.y, fmaf(g.y, w.w, d1));
  }
  float2 own = *reinterpret_cast<const float2*>(dpre + i * 8);
  const float2 r = *reinterpret_cast<const float2*>(rg + i * 4);
  own.x = (own.x + d0) * r.x * (1.f - r.x);              // dpreR
  own.y = (own.y + d1) * r.y * (1.f - r.y);
  *reinterpret_cast<float2*>(dpre + i * 8) = own;        // slots 0,1 only: the neighbours read slots 2,3
}

// A2[pix][t*6 + f] = dpre[pix - off_t][f] as bf16 hi|lo planes (n,64,64,256); columns 198..255 stay zero (allocation memset)
__global__ void __launch_bounds__(256) head_bwd_im2col_kernel(const float* __restrict__ dpre, const int* __restrict__ taps, int ntaps,
                                                              __nv_bfloat16* __restrict__ a2, long long plane, int n) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * 4096 * ntaps) return;
  const int t = (int)(idx % ntaps);
  const long long pix = idx / ntaps;
  const int q = (int)(pix & 63), p = (int)((pix >> 6) & 63);
  const long long img = pix >> 12;
  const int pp = p - taps[2 * t], qq = q - taps[2 * t + 1];
  float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (pp >= 0 && pp <= 63 && qq >= 0 && qq <= 63) {
    const float* src = dpre + ((img * 64 + pp) * 64 + qq) * 8;
    const float4 a = *reinterpret_cast<const float4*>(src);
    const float2 b = *reinterpret_cast<const float2*>(src + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y;
  }
  __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(a2 + pix * 256 + t * 6);
  __nv_bfloat162* ol = reinterpret_cast<__nv_bfloat162*>(a2 + plane + pix * 256 + t * 6);
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const __nv_bfloat162 hi = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    const float2 hf = __bfloat1622float2(hi);
    oh[j] = hi;
    ol[j] = __floats2bfloat162_rn(v[2 * j] - hf.x, v[2 * j + 1] - hf.y);
  }
}

int launch_head_bwd(const float* xhat, const float* rg, const float* bsave, const int32_t* boxes, const float* target,
                    int target_is_frame, const int* taps, const float* wgb, const float* wbb, int ntaps, float* dpre,
                    __nv_bfloat16* a2, long long a2_plane, int n, cudaStream_t st) {
  const long long npix = (long long)n * 4096;
  const unsigned blocks = (unsigned)((npix + 255) / 256);
  head_bwd_seed_kernel<<<blocks, 256, 0, st>>>(xhat, rg, bsave, boxes, target, target_is_frame, dpre, n);
  head_bwd_g_kernel<<<blocks, 256, 0, st>>>(dpre, rg, taps, wbb, ntaps, n);
  head_bwd_r_kernel<<<blocks, 256, 0, st>>>(dpre, rg, taps, wgb, ntaps, n);
  head_bwd_im2col_kernel<<<(unsigned)((npix * ntaps + 255) / 256), 256, 0, st>>>(dpre, taps, ntaps, a2, a2_plane, n);
  return cudaGetLastError() == cudaSuccess ? 4 : -1;
}
}  // namespace ian
