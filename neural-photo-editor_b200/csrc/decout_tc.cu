// decout_tc.cu -- dec_out (reference IAN_simple.py:171-181: DeconvLayer 128 -> 3 ch, 5x5, stride 2, tanh;
// layers.py:436-483) as ONE dense tcgen05 GEMM plus an on-chip col2im, reading its input once.
//
// The output has only 3 channels, so the layer is bandwidth work: h3 is 512 KB/image, x_hat 48 KB.
// Running it as a shifted-tap GEMM would re-stage every input pixel once per tap (25x).  Instead:
//     T[pixel][tap*3+co] = sum_ci h3[pixel][ci] * W[ci][co][tap]          (M = pixels, K = 128, N = 75 -> 80)
// has no shifts at all -- the A operand is the plain NHWC activation, one TMA box per 128 pixels -- and
//     y[co, 2p+r, 2q+s] = sum_{d,e} T[(p+d, q+e)][tap(2+2d-r, 2+2e-s)*3 + co]       (<= 9 terms)
// is a gather over a 3x3 pixel neighbourhood done from shared memory, followed by tanh and a coalesced
// float32 NCHW store.  A work item is 4 input rows x 32 columns (= the 128-row MMA tile, rows p0-1..p0+2,
// TMA zero-fills rows outside the image) and finishes the 4 output rows that depend only on it
// (input rows p0, p0+1): 2x redundant GEMM work, which is free next to the saved traffic.
//
// Roles (persistent CTA, one per SM): warp 0 TMA producer (weights once, then an A ring), warp 1 MMA
// issuer (3-pass bf16 split, main|cross accumulators, two TMEM buffers), warps 2-9 epilogue
// (TMEM -> smem T tile -> col2im -> tanh -> store).
#include <cstdio>
#include <cstring>

#include "edge.h"
#include "tc_ptx.cuh"

namespace ian {

struct DecOutMaps {
  CUtensorMap a;   // h3 planes (C=128, W=32, H=32, N, 2)
  CUtensorMap b;   // weights  (C=128, 80 rows, 2)
};

namespace {

using namespace tc;

constexpr int kThreads = 320;
constexpr int kEpiThreads = 256;
constexpr int BN = 80;                       // 25 taps x 3 channels = 75, padded to a legal UMMA N
constexpr int kAStage = 128 * 64 * 2 * 2;    // one K chunk of the A tile, hi+lo: 32 KB
constexpr int kAStages = 4;                  // 2 work items of look-ahead (an item is two K chunks): hides the TMA round trip
constexpr int kBChunk = BN * 64 * 2 * 2;     // one K chunk of the weights, hi+lo: 20 KB
constexpr int kTLd = 77;                     // T tile row pitch in floats (odd: conflict-free column access)
constexpr int kTBytes = 128 * kTLd * 4;
constexpr int kSmemBytes = 1024 + kAStages * kAStage + 2 * kBChunk + kTBytes + 256;
constexpr int kItemsPerImage = 16;           // 32 input rows / 2 interior rows per item

__global__ void __launch_bounds__(kThreads, 1)
decout_tc_kernel(const __grid_constant__ DecOutMaps maps, const __grid_constant__ DecOutDst dst, const int n_img) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_base = smem_base;
  const uint32_t b_base = a_base + kAStages * kAStage;
  const uint32_t t_base = b_base + 2 * kBChunk;
  const uint32_t bar_base = t_base + kTBytes;
  float* Ts = reinterpret_cast<float*>(smem_al + (t_base - smem_base));
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kAStages + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * kAStages + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * kAStages + 2 + b); };
  const uint32_t b_bar = bar_base + 8u * (2 * kAStages + 4);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kAStages + 5);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_al + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = n_img * kItemsPerImage;

  if (threadIdx.x == 0) {
    pdl_trigger();                                      // tapgemm.h: PDL
    for (int s = 0; s < kAStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), kEpiThreads / 32); }
    mbar_init(b_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_expect_tx(b_bar, 2 * kBChunk);
      tma_load_3d(&maps.b, b_bar, b_base, 0, 0, 0);
      tma_load_3d(&maps.b, b_bar, b_base + kBChunk, 64, 0, 0);
      pdl_wait();                                       // the weights above are constants; h3 below is dec_conv3's output
      uint32_t i = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int n = w / kItemsPerImage, p0 = (w % kItemsPerImage) * 2;
        for (int c = 0; c < 2; ++c, ++i) {
          const int s = i % kAStages;
          mbar_wait(empty_bar(s), ((i / kAStages) & 1u) ^ 1u);
          mbar_expect_tx(full_bar(s), kAStage);
          tma_load_5d(&maps.a, full_bar(s), a_base + s * kAStage, c * 64, 0, p0 - 1, n, 0);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp in uniform control flow; one elected lane issues) =====================
    {
      constexpr uint32_t idesc = make_idesc_bf16_m128(BN);
      mbar_wait(b_bar, 0);
      uint32_t i = 0, t = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x, ++t) {
        const uint32_t buf = t & 1u, use = t >> 1;
        const uint32_t acc_main = tmem_base + buf * 256, acc_cross = acc_main + 128;
        mbar_wait(tempty_bar(buf), (use & 1u) ^ 1u);
        tc_fence_after();
        for (int c = 0; c < 2; ++c, ++i) {
          const int s = i % kAStages;
          mbar_wait(full_bar(s), (i / kAStages) & 1u);
          tc_fence_after();
          const uint32_t sa = a_base + s * kAStage, sb = b_base + c * kBChunk;
          const uint64_t a_hi = make_sw128_desc(sa), a_lo = make_sw128_desc(sa + 128 * 64 * 2);
          const uint64_t b_hi = make_sw128_desc(sb), b_lo = make_sw128_desc(sb + BN * 64 * 2);
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ko = (uint64_t)(k * 2);
              const uint32_t acc = (c > 0 || k > 0) ? 1u : 0u;
              umma_bf16(acc_main, a_hi + ko, b_hi + ko, idesc, acc);
              umma_bf16(acc_cross, a_lo + ko, b_hi + ko, idesc, acc);
              umma_bf16(acc_cross, a_hi + ko, b_lo + ko, idesc, 1u);
            }
            umma_commit(empty_bar(s));
          }
          __syncwarp();
        }
        if (elect_one_sync()) umma_commit(tfull_bar(buf));
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue: TMEM -> smem T tile -> col2im -> tanh -> NCHW store =====================
    pdl_wait();                                         // the destinations may still be read by an earlier kernel of the stream
    const int et = threadIdx.x - 64;                    // 0..255
    const int ew = warp - 2;
    const int lg = warp & 3;                            // TMEM lane group
    const int half = ew >> 2;                           // columns [0,48) or [48,80)
    const int row = lg * 32 + lane;                     // T tile row = pixel (pr*32 + q), pr = 0..3 <-> input row p0-1+pr
    // output element handled in the col2im: out row ur (0..3) of the item, out col v (0..63)
    const int ur = et >> 6, v = et & 63;
    const int q = v >> 1, sx = v & 1, pr = 1 + (ur >> 1), ry = ur & 1;
    uint32_t t = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x, ++t) {
      const int n = w / kItemsPerImage, p0 = (w % kItemsPerImage) * 2;
      const uint32_t buf = t & 1u, use = t >> 1;
      const uint32_t lane_addr = tmem_base + buf * 256 + ((uint32_t)(lg * 32) << 16);
      mbar_wait(tfull_bar(buf), use & 1u);
      tc_fence_after();
      // this warp's columns: half 0 -> [0,48), half 1 -> [48,80)
      const int c_begin = half ? 48 : 0, c_end = half ? 80 : 48;
#pragma unroll 1
      for (int cb = c_begin; cb < c_end; cb += 16) {
        uint32_t vm[16], vc[16];
        __syncwarp();
        tmem_ld16(lane_addr + cb, vm);
        tmem_ld16(lane_addr + 128 + cb, vc);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (cb + j < 75) Ts[row * kTLd + cb + j] = __uint_as_float(vm[j]) + __uint_as_float(vc[j]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(buf));       // TMEM buffer free: next item's MMAs may start
      asm volatile("bar.sync 1, 256;" ::: "memory");     // T tile complete (epilogue warps only)

      // y[co, 2p+ry, 2q+sx] = sum_{d,e} T[(p+d, q+e)][(ki*5+kj)*3+co], ki = 2+2d-ry, kj = 2+2e-sx
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
      for (int d = -1; d <= 1; ++d) {
        if (ry && d < 0) continue;
        const int ki = 2 + 2 * d - ry;
#pragma unroll
        for (int e = -1; e <= 1; ++e) {
          if (sx && e < 0) continue;
          const int qq = q + e;
          if (qq < 0 || qq > 31) continue;               // image border (rows are handled by TMA zero fill)
          const int kj = 2 + 2 * e - sx;
          const float* tp = Ts + ((pr + d) * 32 + qq) * kTLd + (ki * 5 + kj) * 3;
          a0 += tp[0]; a1 += tp[1]; a2 += tp[2];
        }
      }
      const long long off = ((long long)n * 3 * 64 + (2 * p0 + ur)) * 64 + v;
      const float y0 = tanhf(a0), y1 = tanhf(a1), y2 = tanhf(a2);
      for (int d = 0; d < dst.n; ++d) {                  // d > 0: peer GPUs' gather buffers (st.global over NVLink)
        float* o = dst.base[d] + off;
        o[0] = y0;
        o[4096] = y1;
        o[8192] = y2;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");     // T tile consumed: may be overwritten
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ---- cross-GPU barrier over peer memory: every rank owns flags[kMaxPeers]; rank r writes its epoch into slot r of
// every peer's array (release, system scope) and waits until all slots of its own array reached the epoch.
__global__ void peer_signal_kernel(DecOutDst flags, int rank, int epoch) {
  const int p = threadIdx.x;
  if (p >= flags.n) return;
  __threadfence_system();                                // order this GPU's earlier peer stores before the flag
  int* slot = reinterpret_cast<int*>(flags.base[p]) + rank;
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(slot), "r"(epoch) : "memory");
}

__global__ void peer_wait_kernel(const int* my_flags, int world, int epoch) {
  const int p = threadIdx.x;
  if (p >= world) return;
  const long long t0 = clock64();
  int v;
  do {
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(my_flags + p) : "memory");
    if (clock64() - t0 > 20000000000LL) __trap();       // ~10 s: a peer died
  } while (v < epoch);
}

// ---- pipelined all-gather: the decoded shard of step t is pushed to the peers by this small copy kernel on a side
// stream WHILE the tensor kernels of step t+1 run on the main stream (8 GPUs: 7 x 12.6 MB leave each GPU per step; at
// the measured ~770 GB/s per direction that is 0.11 ms of link time, which the 40 us dec_out kernel cannot hide but a
// 1.6 ms step can).  Flags (int, in every rank's own allocation, written by the peers with release.sys stores):
//   free[r]   = t : rank r is done with the gather buffer half that step t writes (its consumer of step t-2 has run)
//   pushed[r] = t : rank r's shard of step t has landed in this rank's buffer
// Block 0 publishes this rank's free[t]; every block waits for peer p's free[t] before its first store to p; the last
// block to finish publishes pushed[t] to everybody.
struct PushArgs {
  const float* src;                 // this rank's shard inside its own gather buffer
  float* dst[kMaxPeers];            // the same slot inside every rank's buffer (dst[rank] unused)
  int* flags[kMaxPeers];            // every rank's flag block: [0,8) barrier, [8,16) free, [16,24) pushed, [24] counter
  long long n_vec;                  // uint4 elements of the shard
  int world, rank, step;
};

__device__ __forceinline__ void st_release_sys(int* p, int v) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int* p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Footprint: the push runs NEXT TO the persistent tensor kernels of the following step (1 CTA per SM, 168 registers x 320
// threads, or 72 x 832 for enc_conv1), so a push CTA must fit in what they leave free -- 128 threads, <= 40 registers, no
// shared memory -- or it would hold an SM back from a statically scheduled persistent kernel (measured: +57 us on
// enc_conv2 with 256-thread / 60-register push CTAs).
__global__ void __launch_bounds__(128, 12) peer_push_kernel(const PushArgs a) {
  int* my_flags = a.flags[a.rank];
  if (blockIdx.x == 0 && threadIdx.x < a.world && (int)threadIdx.x != a.rank) {
    __threadfence_system();
    st_release_sys(a.flags[threadIdx.x] + 8 + a.rank, a.step);          // my half for step t is free
  }
  const uint4* src = reinterpret_cast<const uint4*>(a.src);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (int k = 1; k < a.world; ++k) {
    const int p = (a.rank + k) % a.world;                                // ring order: spreads the switch ports
    if (threadIdx.x == 0) {
      const long long t0 = clock64();
      while (ld_acquire_sys(my_flags + 8 + p) < a.step)
        if (clock64() - t0 > 20000000000LL) __trap();                    // ~10 s: a peer died
    }
    __syncthreads();
    uint4* dst = reinterpret_cast<uint4*>(a.dst[p]);
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < a.n_vec; i += 4 * stride) {                  // 4 independent 16-byte loads in flight per thread
      const uint4 v0 = __ldg(src + i), v1 = __ldg(src + i + stride), v2 = __ldg(src + i + 2 * stride), v3 = __ldg(src + i + 3 * stride);
      dst[i] = v0; dst[i + stride] = v1; dst[i + 2 * stride] = v2; dst[i + 3 * stride] = v3;
    }
    for (; i < a.n_vec; i += stride) dst[i] = __ldg(src + i);
  }
  __threadfence_system();                                                // my peer stores before the flag
  __syncthreads();
  if (threadIdx.x == 0) {
    const int done = atomicAdd(my_flags + 24, 1);
    if (done == (int)gridDim.x - 1) {
      my_flags[24] = 0;                                                  // re-arm for the next launch (stream-ordered)
      __threadfence_system();
      for (int p = 0; p < a.world; ++p) st_release_sys(a.flags[p] + 16 + a.rank, a.step);
    }
  }
}

__global__ void peer_wait_pushed_kernel(const int* my_flags, int world, int step) {
  const int p = threadIdx.x;
  if (p >= world) return;
  const long long t0 = clock64();
  while (ld_acquire_sys(my_flags + 16 + p) < step)
    if (clock64() - t0 > 20000000000LL) __trap();
}

}  // namespace

int launch_peer_push(const float* src, float* const* dsts, float* const* flag_ptrs, long long n_floats, int world, int rank,
                     int step, int ctas, cudaStream_t st) {
  if (world < 1 || world > kMaxPeers || (n_floats & 3)) return -1;
  PushArgs a;
  a.src = src; a.n_vec = n_floats / 4; a.world = world; a.rank = rank; a.step = step;
  for (int d = 0; d < world; ++d) { a.dst[d] = dsts[d]; a.flags[d] = reinterpret_cast<int*>(flag_ptrs[d]); }
  peer_push_kernel<<<ctas, 128, 0, st>>>(a);
  peer_wait_pushed_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const int*>(flag_ptrs[rank]), world, step);
  return cudaGetLastError() == cudaSuccess ? 2 : -1;
}

int launch_peer_barrier(float* const* flag_ptrs, int world, int rank, int epoch, cudaStream_t st) {
  if (world < 1 || world > kMaxPeers) return -1;
  DecOutDst f;
  f.n = world;
  for (int d = 0; d < world; ++d) f.base[d] = flag_ptrs[d];
  peer_signal_kernel<<<1, 32, 0, st>>>(f, rank, epoch);
  peer_wait_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const int*>(flag_ptrs[rank]), world, epoch);
  return cudaGetLastError() == cudaSuccess ? 2 : -1;
}

DecOutMaps* decout_build_maps(const __nv_bfloat16* h3, long long h3_plane, int n_img, const __nv_bfloat16* wt,
                              long long wt_plane, char* err, int errlen) {
  tc::EncodeTiledFn enc = tc::get_encode_fn();
  if (!enc) { snprintf(err, errlen, "cuTensorMapEncodeTiled entry point not available"); return nullptr; }
  DecOutMaps* m = new DecOutMaps();
  memset(m, 0, sizeof(*m));
  {
    cuuint64_t dims[5] = {128, 32, 32, (cuuint64_t)n_img, 2};
    cuuint64_t strides[4] = {128 * 2, 32 * 128 * 2, 32 * 32 * 128 * 2, (cuuint64_t)h3_plane * 2};
    cuuint32_t box[5] = {64, 32, 4, 1, 2};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(&m->a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)h3, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { snprintf(err, errlen, "cuTensorMapEncodeTiled(dec_out A) failed: %d", (int)r); delete m; return nullptr; }
  }
  {
    cuuint64_t dims[3] = {128, BN, 2};
    cuuint64_t strides[2] = {128 * 2, (cuuint64_t)wt_plane * 2};
    cuuint32_t box[3] = {64, BN, 2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(&m->b, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void*)wt, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { snprintf(err, errlen, "cuTensorMapEncodeTiled(dec_out B) failed: %d", (int)r); delete m; return nullptr; }
  }
  return m;
}

void decout_free_maps(DecOutMaps* m) { delete m; }

int launch_dec_out_tc(const DecOutMaps* maps, float* const* dsts, int ndst, int n, cudaStream_t st) {
  static DeviceOnce attr_set;
  const int dev = cur_device();
  if (!attr_set.is_done(dev)) {
    if (cudaFuncSetAttribute(decout_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) != cudaSuccess) return -1;
    attr_set.set_done(dev);
  }
  const int num_sms = tc_num_sms();
  const int total = n * kItemsPerImage;
  const int grid = total < num_sms ? total : num_sms;
  if (ndst < 1 || ndst > kMaxPeers) return -1;
  DecOutDst dst;
  dst.n = ndst;
  for (int d = 0; d < ndst; ++d) dst.base[d] = dsts[d];
  if (launch_pdl(decout_tc_kernel, dim3(grid), dim3(kThreads), kSmemBytes, st, *maps, dst, n) != cudaSuccess) return -1;
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace ian
