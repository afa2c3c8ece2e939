// The 3-D ResNet encoder of BASELINE configs[3] (SURVEY.md 8f-3): /root/reference/models/resnet.py -- BasicStem
// (Conv3d(1 -> 64, k (1,7,7), s (1,2,2), p (1,3,3)) + BN + ReLU, :5-13), BasicBlock (two Conv3DSimple 3x3x3 + BN, residual
// add, ReLU, :61-95) with the 1x1x1 strided down-sample branch (:172-179), planes 8 / 16 / 8 / 16 (:134-137), element-wise
// Dropout after every stage (:156-163), AdaptiveAvgPool3d(1) + Linear + sigmoid (:165-170) -- forward and backward.
//
// Every layer behind the stem has 8 or 16 channels (80 706 parameters in total): there is no dense contraction worth a
// tcgen05 tile (a 128 x 8 MMA would be bound by re-reading A, see DESIGN.md 3.1), the activations are what costs: the
// stem output alone is 8 x 258 x 128 x 32 x 64 x 2 B = 1.08 GB at configs[3].  So these are direct convolutions on
// channels-last (NDHWC) 16-bit tensors (activations fp16, gradients bf16): one thread per output voxel x CT output channels with the weight slice of the
// block resident in shared memory (fp32, broadcast float4 reads), fp32 accumulate, fused per-channel batch statistics
// of the STORED (rounded) output for the BatchNorm that follows; the data gradient is the same kernel run as the
// transposed gather; the weight gradient keeps 8 accumulators per (tap, c_in, c_out-group) work item in registers
// across a run of voxels and finishes with fp32 atomics.  BatchNorm / residual / ReLU / Dropout are fused element-wise
// passes (128-bit accesses, HBM-bound).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "prof.h"

namespace mmnn {
namespace rn {

struct RnConvGeom {
  int N, Di, Hi, Wi, Cin, Do, Ho, Wo, Cout;
  int kd, kh, kw, sd, sh, sw, pd, ph, pw;
};

constexpr int THREADS = 256;
// Deterministic shared-memory accumulation of per-warp partial sums: the warps of the block add their partials one after the other
// (warp 0 first) with plain read-modify-writes instead of shared-memory atomics, whose arrival order -- and, fp32 addition not being
// associative, whose result -- changes from run to run.  The BatchNorm statistics of the forward pass decide every ReLU mask: with
// atomics two runs of the same input differed in the last bit of a statistic, a rounding flipped, and the gradients below moved by
// 10-25 % (round 1).  `body` must touch each address from at most one lane per warp; all threads of the block must reach the macro.
#define RN_WARP_ORDERED(nwarps, body)                         \
  for (int w_ = 0; w_ < (nwarps); ++w_) {                     \
    if ((int)(threadIdx.x >> 5) == w_) { body }               \
    __syncthreads();                                          \
  }

__device__ __forceinline__ float bf_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ void unpack8(const uint4 q, float* f) {
  f[0] = bf_lo(q.x); f[1] = bf_hi(q.x); f[2] = bf_lo(q.y); f[3] = bf_hi(q.y);
  f[4] = bf_lo(q.z); f[5] = bf_hi(q.z); f[6] = bf_lo(q.w); f[7] = bf_hi(q.w);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
__device__ __forceinline__ float round_bf(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
// forward activations are IEEE fp16 (3 more mantissa bits than bf16; every tensor here is O(1..100)), gradients bf16
__device__ __forceinline__ void unpack8h(const uint4 q, float* f) {
  const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 t = __half22float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}
__device__ __forceinline__ uint4 pack8h(const float* f) {
  uint4 q;
  __half2* h = reinterpret_cast<__half2*>(&q);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
  return q;
}
__device__ __forceinline__ float round_h(float v) { return __half2float(__float2half_rn(v)); }
template <bool BF>
__device__ __forceinline__ void unpack8t(const uint4 q, float* f) { if (BF) unpack8(q, f); else unpack8h(q, f); }
template <bool BF>
__device__ __forceinline__ uint4 pack8t(const float* f) { return BF ? pack8(f) : pack8h(f); }

// ------------------------------------------------------------------------------------------------ direct convolution
// DGRAD == false: dst[n,od,oh,ow,co] = sum_{tap,ci} src[n, o*s - p + tap, ci] * w[co][ci][tap]      (nn.Conv3d forward)
// DGRAD == true : dst[n,id,ih,iw,ci] = sum_{tap,co} src[n, (i + p - tap)/s, co] * w[co][ci][tap]    (its data gradient)
// KC = channels of `src` (the reduction), CT = channels of `dst` one thread owns; blockIdx.y = channel group of dst.
template <typename TIN, int KC, int CT, bool DGRAD>
__global__ void __launch_bounds__(THREADS) rn_conv_kernel(const RnConvGeom g, const TIN* __restrict__ src,
                                                          const float* __restrict__ w, uint16_t* __restrict__ dst,
                                                          const uint16_t* add, double* __restrict__ stats) {
  extern __shared__ float ws[];                       // [taps][KC][CT] then [2][CT] block statistics
  const int taps = g.kd * g.kh * g.kw;
  const int cg = blockIdx.y;
  const int tid = threadIdx.x;
  float* sstat = ws + taps * KC * CT;
  for (int i = tid; i < taps * KC * CT; i += THREADS) {
    const int c = i % CT, k = (i / CT) % KC, t = i / (CT * KC);
    const int co = DGRAD ? k : cg * CT + c;
    const int ci = DGRAD ? cg * CT + c : k;
    ws[i] = w[((long long)co * g.Cin + ci) * taps + t];
  }
  if (tid < 2 * CT) sstat[tid] = 0.f;
  __syncthreads();

  const int OD = DGRAD ? g.Di : g.Do, OH = DGRAD ? g.Hi : g.Ho, OW = DGRAD ? g.Wi : g.Wo;   // dst extent
  const int ID = DGRAD ? g.Do : g.Di, IH = DGRAD ? g.Ho : g.Hi, IW = DGRAD ? g.Wo : g.Wi;   // src extent
  const int OC = DGRAD ? g.Cin : g.Cout;
  const long long total = (long long)g.N * OD * OH * OW;
  float ssum[CT], ssq[CT];
#pragma unroll
  for (int c = 0; c < CT; ++c) { ssum[c] = 0.f; ssq[c] = 0.f; }

  for (long long v = (long long)blockIdx.x * THREADS + tid; v < total; v += (long long)gridDim.x * THREADS) {
    const int ow = (int)(v % OW);
    long long t = v / OW;
    const int oh = (int)(t % OH);
    t /= OH;
    const int od = (int)(t % OD);
    const int n = (int)(t / OD);
    float acc[CT];
#pragma unroll
    for (int c = 0; c < CT; ++c) acc[c] = 0.f;
    // data gradient: only the taps congruent to (o + p) modulo the stride reach an integer source coordinate, so the tap loops
    // start there and step by the stride (a stride-2 3x3x3 gather visits ~3.4 taps instead of testing 27)
    for (int a = DGRAD ? (od + g.pd) % g.sd : 0; a < g.kd; a += DGRAD ? g.sd : 1) {
      int zd;
      if (!DGRAD) { zd = od * g.sd - g.pd + a; if ((unsigned)zd >= (unsigned)ID) continue; }
      else { const int q = od + g.pd - a; if (q < 0) continue; zd = q / g.sd; if (zd >= ID) continue; }
      for (int b = DGRAD ? (oh + g.ph) % g.sh : 0; b < g.kh; b += DGRAD ? g.sh : 1) {
        int zh;
        if (!DGRAD) { zh = oh * g.sh - g.ph + b; if ((unsigned)zh >= (unsigned)IH) continue; }
        else { const int q = oh + g.ph - b; if (q < 0) continue; zh = q / g.sh; if (zh >= IH) continue; }
        for (int c = DGRAD ? (ow + g.pw) % g.sw : 0; c < g.kw; c += DGRAD ? g.sw : 1) {
          int zw;
          if (!DGRAD) { zw = ow * g.sw - g.pw + c; if ((unsigned)zw >= (unsigned)IW) continue; }
          else { const int q = ow + g.pw - c; if (q < 0) continue; zw = q / g.sw; if (zw >= IW) continue; }
          const TIN* px = src + ((((long long)n * ID + zd) * IH + zh) * IW + zw) * KC;
          const float* pw = ws + ((a * g.kh + b) * g.kw + c) * (KC * CT);
          if constexpr (std::is_same<TIN, float>::value) {
#pragma unroll
            for (int k = 0; k < KC; ++k) {
              const float xv = __ldg(px + k);
#pragma unroll
              for (int j = 0; j < CT; j += 4) {
                const float4 wv = *reinterpret_cast<const float4*>(pw + k * CT + j);
                acc[j] = fmaf(xv, wv.x, acc[j]); acc[j + 1] = fmaf(xv, wv.y, acc[j + 1]);
                acc[j + 2] = fmaf(xv, wv.z, acc[j + 2]); acc[j + 3] = fmaf(xv, wv.w, acc[j + 3]);
              }
            }
          } else {
#pragma unroll
            for (int k0 = 0; k0 < KC; k0 += 8) {
              float xf[8];
              unpack8t<DGRAD>(__ldg(reinterpret_cast<const uint4*>(px + k0)), xf);
#pragma unroll
              for (int k = 0; k < 8; ++k) {
#pragma unroll
                for (int j = 0; j < CT; j += 4) {
                  const float4 wv = *reinterpret_cast<const float4*>(pw + (k0 + k) * CT + j);
                  acc[j] = fmaf(xf[k], wv.x, acc[j]); acc[j + 1] = fmaf(xf[k], wv.y, acc[j + 1]);
                  acc[j + 2] = fmaf(xf[k], wv.z, acc[j + 2]); acc[j + 3] = fmaf(xf[k], wv.w, acc[j + 3]);
                }
              }
            }
          }
        }
      }
    }
    const long long o = v * OC + cg * CT;
    if (add != nullptr) {
#pragma unroll
      for (int j = 0; j < CT; j += 8) {
        float af[8];
        unpack8t<DGRAD>(*reinterpret_cast<const uint4*>(add + o + j), af);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[j + k] += af[k];
      }
    }
#pragma unroll
    for (int j = 0; j < CT; j += 8) *reinterpret_cast<uint4*>(dst + o + j) = pack8t<DGRAD>(acc + j);
    if (stats != nullptr) {
#pragma unroll
      for (int c = 0; c < CT; ++c) { const float r = DGRAD ? round_bf(acc[c]) : round_h(acc[c]); ssum[c] += r; ssq[c] = fmaf(r, r, ssq[c]); }
    }
  }
  if (stats != nullptr) {
#pragma unroll
    for (int c = 0; c < CT; ++c) {
      float s = ssum[c], q = ssq[c];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        q += __shfl_xor_sync(0xffffffffu, q, off);
      }
      ssum[c] = s; ssq[c] = q;
    }
    RN_WARP_ORDERED(THREADS / 32, if ((tid & 31) == 0) {
      _Pragma("unroll") for (int c = 0; c < CT; ++c) { sstat[c] += ssum[c]; sstat[CT + c] += ssq[c]; }
    })
    if (tid < CT) atomicAdd(&stats[cg * CT + tid], (double)sstat[tid]);
    else if (tid < 2 * CT) atomicAdd(&stats[OC + cg * CT + (tid - CT)], (double)sstat[tid]);
  }
}

template <typename TIN, int KC, int CT, bool DGRAD>
static int launch_conv(const RnConvGeom& g, const void* src, const float* w, void* dst, const void* add, double* stats,
                       cudaStream_t st) {
  const int taps = g.kd * g.kh * g.kw;
  const size_t smem = ((size_t)taps * KC * CT + 2 * CT) * sizeof(float);
  auto kern = rn_conv_kernel<TIN, KC, CT, DGRAD>;
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    smem_set = smem;
  }
  const long long total = DGRAD ? (long long)g.N * g.Di * g.Hi * g.Wi : (long long)g.N * g.Do * g.Ho * g.Wo;
  const int OC = DGRAD ? g.Cin : g.Cout;
  long long bx = (total + THREADS - 1) / THREADS;
  const long long cap = 148LL * 8;
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  kern<<<dim3((unsigned)bx, (unsigned)(OC / CT)), THREADS, smem, st>>>(g, (const TIN*)src, w, (uint16_t*)dst,
                                                                      (const uint16_t*)add, stats);
  return (int)cudaGetLastError();
}

template <bool DGRAD>
static int dispatch_conv(const RnConvGeom& g, int src_f32, const void* src, const float* w, void* dst, const void* add,
                         double* stats, cudaStream_t st) {
  const int KC = DGRAD ? g.Cout : g.Cin, OC = DGRAD ? g.Cin : g.Cout;
  if (OC % 8 != 0) return -2;
  const bool c16 = (OC % 16 == 0);
  if (src_f32) {
    if (KC != 1 || DGRAD) return -3;
    if (c16) return launch_conv<float, 1, 16, false>(g, src, w, dst, add, stats, st);
    return launch_conv<float, 1, 8, false>(g, src, w, dst, add, stats, st);
  }
#define RN_CASE(kc)                                                                                          \
  if (KC == kc) {                                                                                            \
    if (c16) return launch_conv<uint16_t, kc, 16, DGRAD>(g, src, w, dst, add, stats, st);               \
    return launch_conv<uint16_t, kc, 8, DGRAD>(g, src, w, dst, add, stats, st);                         \
  }
  RN_CASE(8)
  RN_CASE(16)
  RN_CASE(64)
#undef RN_CASE
  return -4;
}

// ------------------------------------------------------------------------------------------------ weight gradient
// dw[co][ci][tap] += sum_voxels dy[n,o,co] * x[n, o*s - p + tap, ci].  Tile = TW consecutive output voxels of one output row
// (n, od, oh): the kd x kh input rows the tile touches ((TW-1) sw + kw voxels each, zero-filled outside the volume) and the
// tile's dy are staged in shared memory, so the inner loop has no bounds checks and only fixed-latency operands.  The
// input rows of tile t+1 arrive by cp.async (zero-fill form) into the other half of a double buffer and its dy through
// registers while tile t is being accumulated: one __syncthreads per tile, no exposed global latency.  Work item =
// (tap, ci, group of 8 co); a thread owns up to MAXI items (8 fp32 accumulators each) across all tiles of its block
// (grid-stride), and finishes with fp32 atomics.
constexpr int WG_TW = 32;

template <typename TX>
__device__ __forceinline__ float wg_ld(const TX* p) {
  if constexpr (std::is_same<TX, float>::value) return *p;
  else return __half2float(*p);
}

template <int BYTES>
__device__ __forceinline__ void cp_async_zfill(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int n = valid ? BYTES : 0;
  if (BYTES == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}

// ---- 64 -> 8 forward on HMMA (placed here: uses cp_async_zfill)
// The one convolution of the network with a reduction deep enough for the tensor pipe: layer1.0.conv1, Conv3d(64 -> 8, 3x3x3,
// stride 1, pad 1) over the 1.08 GB stem activation (234 GFLOP per batch of 8 at configs[3], 12.5 ms on the FMA pipe).
// N = 8 output channels is far below a tcgen05 tile (a 128 x 8 UMMA would be bound by re-reading A from shared memory,
// DESIGN.md 3.1), but it is exactly the n8 of the warp-level mma.sync.m16n8k16: M = 16 voxels along W, K = 16 of the 64
// input channels, 27 taps x 4 k-chunks per m-tile.  Tile = 2 output rows x 32 voxels of one (n, od): the 3 x 4 halo rows
// (34 voxels each, zero-filled outside the volume) arrive by cp.async into shared memory with a 144-byte voxel stride
// (conflict-free ldmatrix), the B fragments of all 108 (tap, k-chunk) pairs are packed once per block; 8 warps = 4 m-tiles
// x 2 halves of the tap range, summed through shared memory; fp16 store + the BatchNorm statistics of the stored values.
constexpr int MF_R = 2, MF_XW = 34, MF_VS = 72, MF_HR = MF_R + 2, MF_ROWS = 3 * MF_HR;
constexpr int MF_XS_BYTES = MF_ROWS * MF_XW * MF_VS * 2;            // 58 752
constexpr int MF_WB_BYTES = 27 * 4 * 32 * 8;                        // 27 648
constexpr int MF_SMEM = MF_XS_BYTES + MF_WB_BYTES + 4 * 32 * 16 + 64 + 4 * 32 * 8 + 64;

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

__global__ void __launch_bounds__(THREADS, 2) rn_conv3_mma_fwd_kernel(const RnConvGeom g, const __half* __restrict__ x,
                                                                      const float* __restrict__ w, __half* __restrict__ y,
                                                                      double* __restrict__ stats, const float* __restrict__ w_ds,
                                                                      __half* __restrict__ y_ds, double* __restrict__ stats_ds) {
  // w_ds / y_ds / stats_ds: the block's 1x1x1 stride-1 down-sample convolution (64 -> 8) reads the same input tile: it is the
  // centre tap with its own weights and accumulator (4 more MMAs per m-tile), so the 1.08 GB input is read once for both
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __half* xs = reinterpret_cast<__half*>(smem_raw);
  uint2* wb = reinterpret_cast<uint2*>(smem_raw + MF_XS_BYTES);
  float4* red = reinterpret_cast<float4*>(smem_raw + MF_XS_BYTES + MF_WB_BYTES);
  float* sstat = reinterpret_cast<float*>(smem_raw + MF_XS_BYTES + MF_WB_BYTES + 4 * 32 * 16);
  uint2* wbd = reinterpret_cast<uint2*>(smem_raw + MF_XS_BYTES + MF_WB_BYTES + 4 * 32 * 16 + 64);   // [4 k-chunks][32]
  float* sstat2 = reinterpret_cast<float*>(wbd + 4 * 32);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool ds = w_ds != nullptr;
  if (ds && tid < 128) {
    const int l = tid & 31, kc = tid >> 5;
    const int n = l >> 2, k0 = kc * 16 + (l & 3) * 2;
    const float* pw = w_ds + (long long)n * 64 + k0;          // w_ds[n][ci]
    wbd[tid] = make_uint2(pack_h2(pw[0], pw[1]), pack_h2(pw[8], pw[9]));
  }
  if (tid < 16) sstat2[tid] = 0.f;
  float dsum0 = 0.f, dsum1 = 0.f, dsq0 = 0.f, dsq1 = 0.f;
  for (int i = tid; i < 108 * 32; i += THREADS) {
    const int l = i & 31, t = i >> 5, tap = t >> 2, kc = t & 3;
    const int n = l >> 2, k0 = kc * 16 + (l & 3) * 2;
    const float* pw = w + ((long long)n * 64 + k0) * 27 + tap;      // w[n][ci][tap], ci stride 27
    wb[i] = make_uint2(pack_h2(pw[0], pw[27]), pack_h2(pw[8 * 27], pw[9 * 27]));
  }
  if (tid < 16) sstat[tid] = 0.f;
  float ssum0 = 0.f, ssum1 = 0.f, ssq0 = 0.f, ssq1 = 0.f;
  const int tiles_w = (g.Wo + 31) / 32, tiles_h = (g.Ho + MF_R - 1) / MF_R;
  const int ntiles = g.N * g.Do * tiles_h * tiles_w;
  const int mt = warp & 3, half_ = warp >> 2, rr = mt >> 1, wbase = (mt & 1) * 16;
  const int row_l = (lane & 7) + ((lane >> 3) & 1) * 8, koff = (lane >> 4) * 8;
  const int tap_lo = half_ ? 14 : 0, tap_hi = half_ ? 27 : 14;
  const uint32_t xs_addr = (uint32_t)__cvta_generic_to_shared(xs);
  uint32_t toff[14];                                        // this lane's ldmatrix row address (bytes) for each of its taps
#pragma unroll
  for (int ti = 0; ti < 14; ++ti) {
    const int tap = (tap_lo + ti < 27) ? tap_lo + ti : 26;
    const int a = tap / 9, b = (tap / 3) % 3, c = tap % 3;
    toff[ti] = (uint32_t)((((a * MF_HR + rr + b) * MF_XW + wbase + c + row_l) * MF_VS + koff) * 2);
  }

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int th = r_ % tiles_h;
    r_ /= tiles_h;
    const int od = r_ % g.Do, n = r_ / g.Do;
    const int oh0 = th * MF_R, ow0 = tw * 32;
    __syncthreads();                                        // everyone is done with xs / red of the previous tile
    for (int i = tid; i < MF_ROWS * MF_XW * 8; i += THREADS) {
      const int c = i & 7, vp = i >> 3;
      const int p = vp % MF_XW, r = vp / MF_XW;
      const int a = r / MF_HR, hb = r % MF_HR;
      const int zd = od - 1 + a, zh = oh0 - 1 + hb, zw = ow0 - 1 + p;
      const bool ok = (unsigned)zd < (unsigned)g.Di && (unsigned)zh < (unsigned)g.Hi && (unsigned)zw < (unsigned)g.Wi;
      const __half* src = ok ? x + ((((long long)n * g.Di + zd) * g.Hi + zh) * g.Wi + zw) * 64 + c * 8 : x;
      cp_async_zfill<16>(xs + (r * MF_XW + p) * MF_VS + c * 8, src, ok);
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();
    float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
    float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
    for (int ti = 0; ti < 14; ++ti) {
      const int tap = tap_lo + ti;
      if (tap >= tap_hi) break;
      const uint32_t abase = xs_addr + toff[ti];
      const bool centre = ds && tap == 13;
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        uint32_t a0, a1, a2, a3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(abase + kc * 32));
        const uint2 bf = wb[(tap * 4 + kc) * 32 + lane];
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                     : "+f"(c0), "+f"(c1), "+f"(c2), "+f"(c3) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.x), "r"(bf.y));
        if (centre) {                                       // warp-uniform (tap 13 belongs to the first half of the tap range)
          const uint2 bd = wbd[kc * 32 + lane];
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                       : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bd.x), "r"(bd.y));
        }
      }
    }
    if (half_ == 1) red[mt * 32 + lane] = make_float4(c0, c1, c2, c3);
    __syncthreads();
    if (half_ == 0) {
      const float4 o = red[mt * 32 + lane];
      c0 += o.x; c1 += o.y; c2 += o.z; c3 += o.w;
      const int oh = oh0 + rr, gq = lane >> 2, co = (lane & 3) * 2;
      if (oh < g.Ho) {
        const long long rowbase = (((long long)n * g.Do + od) * g.Ho + oh) * g.Wo;
        const int owa = ow0 + wbase + gq, owb = owa + 8;
        if (owa < g.Wo) {
          const __half2 h = __floats2half2_rn(c0, c1);
          *reinterpret_cast<__half2*>(y + (rowbase + owa) * 8 + co) = h;
          const float2 f = __half22float2(h);
          ssum0 += f.x; ssum1 += f.y; ssq0 = fmaf(f.x, f.x, ssq0); ssq1 = fmaf(f.y, f.y, ssq1);
        }
        if (owb < g.Wo) {
          const __half2 h = __floats2half2_rn(c2, c3);
          *reinterpret_cast<__half2*>(y + (rowbase + owb) * 8 + co) = h;
          const float2 f = __half22float2(h);
          ssum0 += f.x; ssum1 += f.y; ssq0 = fmaf(f.x, f.x, ssq0); ssq1 = fmaf(f.y, f.y, ssq1);
        }
        if (ds) {
          if (owa < g.Wo) {
            const __half2 h = __floats2half2_rn(d0, d1);
            *reinterpret_cast<__half2*>(y_ds + (rowbase + owa) * 8 + co) = h;
            const float2 f = __half22float2(h);
            dsum0 += f.x; dsum1 += f.y; dsq0 = fmaf(f.x, f.x, dsq0); dsq1 = fmaf(f.y, f.y, dsq1);
          }
          if (owb < g.Wo) {
            const __half2 h = __floats2half2_rn(d2, d3);
            *reinterpret_cast<__half2*>(y_ds + (rowbase + owb) * 8 + co) = h;
            const float2 f = __half22float2(h);
            dsum0 += f.x; dsum1 += f.y; dsq0 = fmaf(f.x, f.x, dsq0); dsq1 = fmaf(f.y, f.y, dsq1);
          }
        }
      }
    }
  }
  if (ds && stats_ds != nullptr) {
#pragma unroll
    for (int off = 4; off < 32; off <<= 1) {
      dsum0 += __shfl_xor_sync(0xffffffffu, dsum0, off); dsum1 += __shfl_xor_sync(0xffffffffu, dsum1, off);
      dsq0 += __shfl_xor_sync(0xffffffffu, dsq0, off); dsq1 += __shfl_xor_sync(0xffffffffu, dsq1, off);
    }
    RN_WARP_ORDERED(THREADS / 32, if (lane < 4) {
      sstat2[lane * 2] += dsum0; sstat2[lane * 2 + 1] += dsum1;
      sstat2[8 + lane * 2] += dsq0; sstat2[8 + lane * 2 + 1] += dsq1;
    })
    if (tid < 16) atomicAdd(&stats_ds[tid], (double)sstat2[tid]);
  }
  if (stats != nullptr) {
#pragma unroll
    for (int off = 4; off < 32; off <<= 1) {
      ssum0 += __shfl_xor_sync(0xffffffffu, ssum0, off); ssum1 += __shfl_xor_sync(0xffffffffu, ssum1, off);
      ssq0 += __shfl_xor_sync(0xffffffffu, ssq0, off); ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, off);
    }
    RN_WARP_ORDERED(THREADS / 32, if (lane < 4) {
      sstat[lane * 2] += ssum0; sstat[lane * 2 + 1] += ssum1;
      sstat[8 + lane * 2] += ssq0; sstat[8 + lane * 2 + 1] += ssq1;
    })
    if (tid < 16) atomicAdd(&stats[tid], (double)sstat[tid]);
  }
}

// ---- 8-channel source, 3x3x3 stride 1 pad 1, on HMMA with TAP PAIRS as the k16: the forward of the 8 -> 8 convolutions
// (fp16), their data gradient (bf16) and the data gradient 8 -> 64 of layer1.0.conv1 (NT = 8 n-tiles).  One voxel of the
// source is 8 channels = one 16-byte ldmatrix row, so the four 8x8 matrices of an ldmatrix.x4 can come from two different
// taps (lanes 16-31 point into the second tap's window): k = (tap pair, 8 channels), 14 pairs cover the 27 taps (the 28th
// has zero weights).  NT = 1: tile = 4 rows x 32 voxels, one m-tile per warp, direct 128-byte-per-instruction stores;
// NT = 8: tile = 2 rows x 32, warps = 4 m-tiles x 2 halves of the 64 output channels, stores staged through shared memory
// so every voxel's 64 bytes leave as full sectors.
template <int NT, bool DGRAD>
__global__ void __launch_bounds__(THREADS, 2) rn_conv3_k8_mma_kernel(const RnConvGeom g, const uint16_t* __restrict__ src,
                                                                     const float* __restrict__ w, uint16_t* __restrict__ dst,
                                                                     const uint16_t* __restrict__ add, double* __restrict__ stats,
                                                                     const uint16_t* __restrict__ src2, const float* __restrict__ w2) {
  // src2 / w2 (DGRAD only): the output gradient and [8][OC] weight of the block's 1x1x1 stride-1 down-sample convolution; its
  // data gradient is one more "tap" (the 28th, at the centre) of the same gather, so dx = dgrad(conv1) + dgrad(downsample)
  // leaves in ONE pass instead of a second kernel that re-reads and re-writes dx (1.08 GB at layer1)
  constexpr int R = (NT == 1) ? 4 : 2, HR = R + 2, NH = (NT == 1) ? 1 : 4, OC = 8 * NT;
  constexpr int XS_BYTES = 3 * HR * MF_XW * 16, WB_BYTES = 14 * NT * 32 * 8;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int XS2_BYTES = R * 32 * 16;
  uint16_t* xs = reinterpret_cast<uint16_t*>(smem_raw);                               // [2][3 HR][34][8]: double buffer
  uint2* wb = reinterpret_cast<uint2*>(smem_raw + 2 * XS_BYTES);
  uint16_t* stg = reinterpret_cast<uint16_t*>(smem_raw + 2 * XS_BYTES + WB_BYTES);  // NT == 8: [8 warps][16][40]
  float* sstat = reinterpret_cast<float*>(smem_raw + 2 * XS_BYTES + WB_BYTES + 8 * 16 * 40 * 2);
  uint16_t* xs2 = reinterpret_cast<uint16_t*>(smem_raw + 2 * XS_BYTES + WB_BYTES + 8 * 16 * 40 * 2 + 64);   // [2][R][32][8]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wCin = g.Cin;                                   // weight tensor is [Cout][Cin][27]
  for (int i = tid; i < 14 * NT * 32; i += THREADS) {
    const int l = i & 31, j = (i >> 5) % NT, pair = (i >> 5) / NT;
    const int n = 8 * j + (l >> 2), k = (l & 3) * 2;
    float v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int tap = 2 * pair + (q >> 1), kk = k + (q & 1);
      const int co = DGRAD ? kk : n, ci = DGRAD ? n : kk;
      v[q] = (tap < 27) ? w[((long long)co * wCin + ci) * 27 + tap] : ((DGRAD && w2 != nullptr) ? w2[(long long)co * wCin + ci] : 0.f);
    }
    wb[i] = DGRAD ? make_uint2(pack2(v[0], v[1]), pack2(v[2], v[3])) : make_uint2(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]));
  }
  if (tid < 16) sstat[tid] = 0.f;
  float ssum0 = 0.f, ssum1 = 0.f, ssq0 = 0.f, ssq1 = 0.f;
  const int tiles_w = (g.Wo + 31) / 32, tiles_h = (g.Ho + R - 1) / R;
  const int ntiles = g.N * g.Do * tiles_h * tiles_w;
  const int mt = (NT == 1) ? warp : (warp & 3), nh = (NT == 1) ? 0 : (warp >> 2);
  const int rr = mt >> 1, wbase = (mt & 1) * 16;
  const int row_l = (lane & 7) + ((lane >> 3) & 1) * 8, second = lane >> 4;
  const uint32_t xs_addr = (uint32_t)__cvta_generic_to_shared(xs);
  uint32_t poff[14];                                        // this lane's ldmatrix row address (bytes) for every tap pair
#pragma unroll
  for (int pair = 0; pair < 14; ++pair) {
    int tap = 2 * pair + second;
    if (tap > 26) tap = 26;                                 // zero weights: any finite window will do
    int a = tap / 9, b = (tap / 3) % 3, c = tap % 3;
    if (DGRAD) { a = 2 - a; b = 2 - b; c = 2 - c; }
    poff[pair] = (uint32_t)((((a * HR + rr + b) * MF_XW + wbase + c + row_l) * 8) * 2);
  }
  const bool special = DGRAD && src2 != nullptr && second == 1;       // pair 13, lanes 16-31: the down-sample "tap" in xs2
  const uint32_t xs2_addr = (uint32_t)__cvta_generic_to_shared(xs2);
  const uint32_t poff2 = (uint32_t)(((rr * 32 + wbase + row_l) * 8) * 2);

  auto stage = [&](int tile, int buf) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int th = r_ % tiles_h;
    r_ /= tiles_h;
    const int od = r_ % g.Do, n = r_ / g.Do;
    const int oh0 = th * R, ow0 = tw * 32;
    uint16_t* xb = xs + (size_t)buf * (XS_BYTES / 2);
    for (int i = tid; i < 3 * HR * MF_XW; i += THREADS) {
      const int p = i % MF_XW, r = i / MF_XW;
      const int a = r / HR, hb = r % HR;
      const int zd = od - 1 + a, zh = oh0 - 1 + hb, zw = ow0 - 1 + p;
      const bool ok = (unsigned)zd < (unsigned)g.Do && (unsigned)zh < (unsigned)g.Ho && (unsigned)zw < (unsigned)g.Wo;
      const uint16_t* sp = ok ? src + ((((long long)n * g.Do + zd) * g.Ho + zh) * g.Wo + zw) * 8 : src;
      cp_async_zfill<16>(xb + i * 8, sp, ok);
    }
    if (DGRAD && src2 != nullptr && tid < R * 32) {
      const int oh = oh0 + tid / 32, ow = ow0 + (tid & 31);
      const bool ok = oh < g.Ho && ow < g.Wo;
      const uint16_t* sp = ok ? src2 + ((((long long)n * g.Do + od) * g.Ho + oh) * g.Wo + ow) * 8 : src2;
      cp_async_zfill<16>(xs2 + (size_t)buf * (XS2_BYTES / 2) + tid * 8, sp, ok);
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };

  int buf = 0;
  if ((int)blockIdx.x < ntiles) stage(blockIdx.x, 0);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, buf ^= 1) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int th = r_ % tiles_h;
    r_ /= tiles_h;
    const int od = r_ % g.Do, n = r_ / g.Do;
    const int oh0 = th * R, ow0 = tw * 32;
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();                                        // tile `buf` has landed; everyone is done reading buffer buf ^ 1
    if (tile + (int)gridDim.x < ntiles) stage(tile + gridDim.x, buf ^ 1);   // next tile streams in behind the MMAs
    const uint32_t xbase = xs_addr + (uint32_t)(buf * XS_BYTES);
    const uint32_t x2base = xs2_addr + (uint32_t)(buf * XS2_BYTES) + poff2;
    float acc[NH][4];
#pragma unroll
    for (int j = 0; j < NH; ++j) { acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f; }
#pragma unroll
    for (int pair = 0; pair < 14; ++pair) {
      const uint32_t aaddr = (pair == 13 && special) ? x2base : xbase + poff[pair];
      uint32_t a0, a1, a2, a3;
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                   : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(aaddr));
#pragma unroll
      for (int j = 0; j < NH; ++j) {
        const uint2 bf = wb[(pair * NT + nh * NH + j) * 32 + lane];
        if (DGRAD)
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                       : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                       : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.x), "r"(bf.y));
        else
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                       : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                       : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.x), "r"(bf.y));
      }
    }
    const int oh = oh0 + rr;
    const long long rowbase = (((long long)n * g.Do + od) * g.Ho + oh) * g.Wo;
    if (NT == 1) {
      const int gq = lane >> 2, co = (lane & 3) * 2;
      if (oh < g.Ho) {
#pragma unroll
        for (int hsel = 0; hsel < 2; ++hsel) {
          const int ow = ow0 + wbase + gq + hsel * 8;
          if (ow < g.Wo) {
            float v0 = acc[0][hsel * 2], v1 = acc[0][hsel * 2 + 1];
            const long long o = (rowbase + ow) * 8 + co;
            if (add != nullptr) {
              const uint32_t u = *reinterpret_cast<const uint32_t*>(add + o);
              if (DGRAD) { v0 += bf_lo(u); v1 += bf_hi(u); }
              else { const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u)); v0 += f.x; v1 += f.y; }
            }
            if (DGRAD) {
              *reinterpret_cast<uint32_t*>(dst + o) = pack2(v0, v1);
            } else {
              const __half2 h = __floats2half2_rn(v0, v1);
              *reinterpret_cast<__half2*>(dst + o) = h;
              const float2 f = __half22float2(h);
              ssum0 += f.x; ssum1 += f.y; ssq0 = fmaf(f.x, f.x, ssq0); ssq1 = fmaf(f.y, f.y, ssq1);
            }
          }
        }
      }
    } else {
      uint16_t* st_ = stg + warp * (16 * 40);
      const int gq = lane >> 2, t2 = (lane & 3) * 2;
#pragma unroll
      for (int j = 0; j < NH; ++j) {
        *reinterpret_cast<uint32_t*>(st_ + gq * 40 + 8 * j + t2) = DGRAD ? pack2(acc[j][0], acc[j][1]) : pack_h2(acc[j][0], acc[j][1]);
        *reinterpret_cast<uint32_t*>(st_ + (gq + 8) * 40 + 8 * j + t2) = DGRAD ? pack2(acc[j][2], acc[j][3]) : pack_h2(acc[j][2], acc[j][3]);
      }
      __syncwarp();
#pragma unroll
      for (int it = 0; it < 2; ++it) {
        const int row = (lane >> 2) + it * 8, chunk = lane & 3;
        const int ow = ow0 + wbase + row;
        if (oh < g.Ho && ow < g.Wo)
          *reinterpret_cast<uint4*>(dst + (rowbase + ow) * OC + nh * 32 + chunk * 8) = *reinterpret_cast<const uint4*>(st_ + row * 40 + chunk * 8);
      }
      __syncwarp();
    }
  }
  if (stats != nullptr) {
#pragma unroll
    for (int off = 4; off < 32; off <<= 1) {
      ssum0 += __shfl_xor_sync(0xffffffffu, ssum0, off); ssum1 += __shfl_xor_sync(0xffffffffu, ssum1, off);
      ssq0 += __shfl_xor_sync(0xffffffffu, ssq0, off); ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, off);
    }
    RN_WARP_ORDERED(THREADS / 32, if (lane < 4) {
      sstat[lane * 2] += ssum0; sstat[lane * 2 + 1] += ssum1;
      sstat[8 + lane * 2] += ssq0; sstat[8 + lane * 2 + 1] += ssq1;
    })
    if (tid < 16) atomicAdd(&stats[tid], (double)sstat[tid]);
  }
}

template <int NT, bool DGRAD>
static int launch_conv3_k8_mma(const RnConvGeom& g, const void* src, const float* w, void* dst, const void* add, double* stats,
                               cudaStream_t st, const void* src2 = nullptr, const float* w2 = nullptr) {
  constexpr int R = (NT == 1) ? 4 : 2, HR = R + 2;
  constexpr int SMEM = 2 * 3 * HR * MF_XW * 16 + 14 * NT * 32 * 8 + 8 * 16 * 40 * 2 + 64 + 2 * R * 32 * 16;
  auto kern = rn_conv3_k8_mma_kernel<NT, DGRAD>;
  static bool attr = false;
  if (!attr && SMEM > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  const long long ntiles = (long long)g.N * g.Do * ((g.Ho + R - 1) / R) * ((g.Wo + 31) / 32);
  if (ntiles > 0x7fffffffLL) return -6;
  const int blocks = (int)(ntiles < 148 * 4 ? ntiles : 148 * 4);
  kern<<<blocks, THREADS, SMEM, st>>>(g, (const uint16_t*)src, w, (uint16_t*)dst, (const uint16_t*)add, stats,
                                      (const uint16_t*)src2, w2);
  return (int)cudaGetLastError();
}

// ---- weight gradient on HMMA: dw^T[ci][co] (per tap) = sum_v x[v + tap][ci] * dy[v][co] with the VOXELS as the k16.  Both
// operands are stored voxel-major (channels contiguous), which is the transposed form of what mma.sync wants, so both
// fragments come from ldmatrix.trans: A = 16 ci x 16 voxels from the staged input rows (for C_in = 8 the two halves of the
// m16 are two different taps), B = 16 voxels x 8 co from the staged dy.  dy is bf16, so the fp16 input rows are converted
// to bf16 while they are staged (the weight gradient averages over ~10^6 voxels; 8 mantissa bits of x are plenty).
// A warp owns up to MAXU (tap, ci-chunk) units x NTN co-tiles of accumulators across all tiles of its block; fp32 atomics
// at the end.  Any kernel size / stride / padding (each lane supplies its own ldmatrix row address).
template <int CIN, int NTN, int MAXU>
__global__ void __launch_bounds__(THREADS, 2) rn_wgrad_mma_kernel(const RnConvGeom g, const __half* __restrict__ x,
                                                                  const uint16_t* __restrict__ dy, float* __restrict__ dw, int R) {
  constexpr int VS = (CIN == 64) ? 72 : ((CIN == 16) ? 24 : 8);   // voxel stride in shared memory (conflict-free ldmatrix)
  constexpr int COUT = 8 * NTN, CH8 = CIN / 8, C16 = (CIN >= 16) ? CIN / 16 : 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int taps = g.kd * g.kh * g.kw;
  const int HRs = (R - 1) * g.sh + g.kh, XW = 31 * g.sw + g.kw, nrows = g.kd * HRs;
  uint16_t* xs = reinterpret_cast<uint16_t*>(smem_raw);
  uint16_t* dys = xs + (size_t)nrows * XW * VS;               // [R][32][COUT]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q = lane >> 3, vl = (lane & 7) + (q >> 1) * 8;
  const int nunits = (CIN >= 16) ? taps * C16 : (taps + 1) / 2;
  int ubase[MAXU];
  float acc[MAXU][NTN][4];
#pragma unroll
  for (int i = 0; i < MAXU; ++i) {
    const int u = warp + 8 * i;
    const int uu = (u < nunits) ? u : 0;
    int tap, choff;
    if (CIN >= 16) { tap = uu / C16; choff = (uu % C16) * 16 + (q & 1) * 8; }
    else { tap = 2 * uu + (q & 1); if (tap >= taps) tap = 2 * uu; choff = 0; }
    const int a = tap / (g.kh * g.kw), b = (tap / g.kw) % g.kh, c = tap % g.kw;
    ubase[i] = ((a * HRs + b) * XW + c + vl * g.sw) * VS + choff;
#pragma unroll
    for (int j = 0; j < NTN; ++j) { acc[i][j][0] = 0.f; acc[i][j][1] = 0.f; acc[i][j][2] = 0.f; acc[i][j][3] = 0.f; }
  }
  const int tiles_w = (g.Wo + 31) / 32, tiles_h = (g.Ho + R - 1) / R;
  const int ntiles = g.N * g.Do * tiles_h * tiles_w;
  const uint32_t xs_addr = (uint32_t)__cvta_generic_to_shared(xs), dys_addr = (uint32_t)__cvta_generic_to_shared(dys);
  const float inv_xw = 1.0f / (float)XW, inv_hrs = 1.0f / (float)HRs;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int th = r_ % tiles_h;
    r_ /= tiles_h;
    const int od = r_ % g.Do, n = r_ / g.Do;
    const int oh0 = th * R, ow0 = tw * 32;
    __syncthreads();
    // input rows, fp16 -> bf16 on the way; one flat loop (a row-by-row loop measured 1.5-3x slower), runtime divisors replaced
    // by an exact float reciprocal (operands < 2^16), loads batched U at a time so their latencies overlap
    {
      constexpr int U = 4;                                  // loads of U chunks in flight before the first conversion
      const int total = nrows * XW * CH8;
      for (int base = 0; base < total; base += THREADS * U) {
        uint4 qv[U];
        int dsto[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int i = base + u * THREADS + tid;
          const int ch = i % CH8, vp = i / CH8;
          const int r = __float2int_rd(((float)vp + 0.5f) * inv_xw), p = vp - r * XW;
          const int a = __float2int_rd(((float)r + 0.5f) * inv_hrs), hb = r - a * HRs;
          const int zd = od * g.sd - g.pd + a, zh = oh0 * g.sh - g.ph + hb, zw = ow0 * g.sw - g.pw + p;
          dsto[u] = (i < total) ? vp * VS + ch * 8 : -1;
          qv[u] = make_uint4(0u, 0u, 0u, 0u);
          if (i < total && (unsigned)zd < (unsigned)g.Di && (unsigned)zh < (unsigned)g.Hi && (unsigned)zw < (unsigned)g.Wi)
            qv[u] = __ldg(reinterpret_cast<const uint4*>(x + ((((long long)n * g.Di + zd) * g.Hi + zh) * g.Wi + zw) * CIN + ch * 8));
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (dsto[u] >= 0) {
            float f[8];
            unpack8h(qv[u], f);                             // fp16 zero -> bf16 zero
            *reinterpret_cast<uint4*>(xs + dsto[u]) = pack8(f);
          }
        }
      }
    }
    for (int i = tid; i < R * 32 * NTN; i += THREADS) {
      const int c8 = i % NTN, v = (i / NTN) % 32, rr = i / NTN / 32;
      uint4 o = make_uint4(0u, 0u, 0u, 0u);
      if (oh0 + rr < g.Ho && ow0 + v < g.Wo)
        o = __ldg(reinterpret_cast<const uint4*>(dy + ((((long long)n * g.Do + od) * g.Ho + oh0 + rr) * g.Wo + ow0 + v) * COUT + c8 * 8));
      *reinterpret_cast<uint4*>(dys + (size_t)i * 8) = o;
    }
    __syncthreads();
    for (int kc = 0; kc < R * 2; ++kc) {
      const int rr = kc >> 1, wh = kc & 1;
      const int koff = (rr * g.sh * XW + wh * 16 * g.sw) * VS;
      uint32_t b0[NTN], b1[NTN];
#pragma unroll
      for (int j = 0; j < NTN; ++j) {
        const uint32_t baddr = dys_addr + (uint32_t)(((rr * 32 + wh * 16 + (lane & 15)) * COUT + j * 8) * 2);
        asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];\n" : "=r"(b0[j]), "=r"(b1[j]) : "r"(baddr));
      }
#pragma unroll
      for (int i = 0; i < MAXU; ++i) {
        uint32_t a0, a1, a2, a3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(xs_addr + (uint32_t)((ubase[i] + koff) * 2)));
#pragma unroll
        for (int j = 0; j < NTN; ++j)
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                       : "+f"(acc[i][j][0]), "+f"(acc[i][j][1]), "+f"(acc[i][j][2]), "+f"(acc[i][j][3])
                       : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0[j]), "r"(b1[j]));
      }
    }
  }
  const int gq = lane >> 2, t2 = (lane & 3) * 2;
#pragma unroll
  for (int i = 0; i < MAXU; ++i) {
    const int u = warp + 8 * i;
    if (u >= nunits) continue;
#pragma unroll
    for (int hsel = 0; hsel < 2; ++hsel) {                  // accumulator rows g (hsel 0) and g + 8 (hsel 1)
      int tap, ci;
      if (CIN >= 16) { tap = u / C16; ci = (u % C16) * 16 + gq + hsel * 8; }
      else { tap = 2 * u + hsel; ci = gq; }
      if (tap >= taps) continue;
#pragma unroll
      for (int j = 0; j < NTN; ++j) {
        const int co = j * 8 + t2;
        atomicAdd(&dw[((long long)co * CIN + ci) * taps + tap], acc[i][j][hsel * 2]);
        atomicAdd(&dw[((long long)(co + 1) * CIN + ci) * taps + tap], acc[i][j][hsel * 2 + 1]);
      }
    }
  }
}

template <int CIN, int NTN, int MAXU>
static int launch_wgrad_mma(const RnConvGeom& g, const void* x, const void* dy, float* dw, cudaStream_t st) {
  constexpr int VS = (CIN == 64) ? 72 : ((CIN == 16) ? 24 : 8);
  const int XW = 31 * g.sw + g.kw;
  int R = 4;
  size_t smem = 0;
  for (;; R >>= 1) {
    const int HRs = (R - 1) * g.sh + g.kh;
    smem = ((size_t)g.kd * HRs * XW * VS + (size_t)R * 32 * 8 * NTN) * 2;
    if (smem <= 60 * 1024 || R == 1) break;
  }
  if (smem > 200 * 1024) return -7;
  auto kern = rn_wgrad_mma_kernel<CIN, NTN, MAXU>;
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    smem_set = smem;
  }
  const long long ntiles = (long long)g.N * g.Do * ((g.Ho + R - 1) / R) * ((g.Wo + 31) / 32);
  if (ntiles > 0x7fffffffLL) return -6;
  const int blocks = (int)(ntiles < 148 * 3 ? ntiles : 148 * 3);
  kern<<<blocks, THREADS, smem, st>>>(g, (const __half*)x, (const uint16_t*)dy, dw, R);
  return (int)cudaGetLastError();
}

// ---- the same weight gradient with fp16 operands: dy (bf16) is rescaled by a power of two S = 2^floor(log2(8192 / max|dy|))
// while its small tile passes through registers, so the fp16 input rows need NO conversion and arrive by zero-filling
// cp.async into the other half of a double buffer while the current tile is in the tensor pipe (the bf16 variant above
// spends its time converting 59 KB per tile through registers, ncu: long-scoreboard 6.5 of 12.5 cycles per issue).
// max|dy| comes from rn_absmax_kernel (one pass over dy, < 2 % of the weight gradient's own traffic at layer1); fp16
// keeps 11 significant bits of every dy within 2^-14 of the maximum, more than the 8 of its bf16 storage.
__global__ void __launch_bounds__(THREADS) rn_absmax_kernel(const uint4* __restrict__ dy, long long n8, unsigned* __restrict__ out) {
  unsigned m = 0;
  for (long long i = (long long)blockIdx.x * THREADS + threadIdx.x; i < n8; i += (long long)gridDim.x * THREADS) {
    const uint4 q = __ldg(dy + i);
    const unsigned w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) { m = max(m, w4[k] & 0x7fffu); m = max(m, (w4[k] >> 16) & 0x7fffu); }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0 && m != 0) atomicMax(out, m << 16);       // bf16 magnitude bits -> fp32 bits
}

template <int CIN, int NTN, int MAXU, int NW>
__global__ void __launch_bounds__(NW * 32, (NW > 8 ? 1 : (MAXU * NTN <= 4 ? 4 : 2))) rn_wgrad_mma16_kernel(const RnConvGeom g, const __half* __restrict__ x,
                                                                    const uint16_t* __restrict__ dy, float* __restrict__ dw, int R,
                                                                    const unsigned* __restrict__ amax_bits) {
  // NW warps per block: 16 for the 14-units-per-warp shape (64 -> 8: 7 units per warp, one 512-thread block per SM)
  constexpr int VS = (CIN == 64) ? 72 : ((CIN == 16) ? 24 : 8);
  constexpr int COUT = 8 * NTN, CH8 = CIN / 8, C16 = (CIN >= 16) ? CIN / 16 : 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int taps = g.kd * g.kh * g.kw;
  const int HRs = (R - 1) * g.sh + g.kh, XW = 31 * g.sw + g.kw, nrows = g.kd * HRs;
  const int xbuf = nrows * XW * VS, dbuf = R * 32 * COUT;          // elements per buffer
  uint16_t* xs = reinterpret_cast<uint16_t*>(smem_raw);            // [2][xbuf]
  uint16_t* dys = xs + 2 * (size_t)xbuf;                           // [2][dbuf]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q = lane >> 3, vl = (lane & 7) + (q >> 1) * 8;
  const int nunits = (CIN >= 16) ? taps * C16 : (taps + 1) / 2;
  const float amax = __uint_as_float(*amax_bits);
  float S = 1.f;
  if (amax > 0.f && amax < 3.0e38f) S = exp2f(floorf(log2f(8192.f / amax)));
  int ubase[MAXU];
  float acc[MAXU][NTN][4];
#pragma unroll
  for (int i = 0; i < MAXU; ++i) {
    const int u = warp + NW * i;
    const int uu = (u < nunits) ? u : 0;
    int tap, choff;
    if (CIN >= 16) { tap = uu / C16; choff = (uu % C16) * 16 + (q & 1) * 8; }
    else { tap = 2 * uu + (q & 1); if (tap >= taps) tap = 2 * uu; choff = 0; }
    const int a = tap / (g.kh * g.kw), b = (tap / g.kw) % g.kh, c = tap % g.kw;
    ubase[i] = ((a * HRs + b) * XW + c + vl * g.sw) * VS + choff;
#pragma unroll
    for (int j = 0; j < NTN; ++j) { acc[i][j][0] = 0.f; acc[i][j][1] = 0.f; acc[i][j][2] = 0.f; acc[i][j][3] = 0.f; }
  }
  const int tiles_w = (g.Wo + 31) / 32, tiles_h = (g.Ho + R - 1) / R;
  const int ntiles = g.N * g.Do * tiles_h * tiles_w;
  const uint32_t xs_addr = (uint32_t)__cvta_generic_to_shared(xs), dys_addr = (uint32_t)__cvta_generic_to_shared(dys);
  const float inv_xw = 1.0f / (float)XW, inv_hrs = 1.0f / (float)HRs;
  const int dyvecs = R * 32 * NTN;                                  // <= 256: one uint4 of dy per thread

  auto decode = [&](int tile, int& n, int& od, int& oh0, int& ow0) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int th = r_ % tiles_h;
    r_ /= tiles_h;
    od = r_ % g.Do; n = r_ / g.Do; oh0 = th * R; ow0 = tw * 32;
  };
  auto stage_x = [&](int tile, int buf) {
    int n, od, oh0, ow0;
    decode(tile, n, od, oh0, ow0);
    uint16_t* xb = xs + (size_t)buf * xbuf;
    const int total = nrows * XW * CH8;
    for (int i = tid; i < total; i += NW * 32) {
      const int ch = i % CH8, vp = i / CH8;
      const int r = __float2int_rd(((float)vp + 0.5f) * inv_xw), p = vp - r * XW;
      const int a = __float2int_rd(((float)r + 0.5f) * inv_hrs), hb = r - a * HRs;
      const int zd = od * g.sd - g.pd + a, zh = oh0 * g.sh - g.ph + hb, zw = ow0 * g.sw - g.pw + p;
      const bool ok = (unsigned)zd < (unsigned)g.Di && (unsigned)zh < (unsigned)g.Hi && (unsigned)zw < (unsigned)g.Wi;
      const __half* sp = ok ? x + ((((long long)n * g.Di + zd) * g.Hi + zh) * g.Wi + zw) * CIN + ch * 8 : x;
      cp_async_zfill<16>(xb + vp * VS + ch * 8, sp, ok);
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };
  auto load_dy = [&](int tile) -> uint4 {
    int n, od, oh0, ow0;
    decode(tile, n, od, oh0, ow0);
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (tid < dyvecs) {
      const int c8 = tid % NTN, v = (tid / NTN) % 32, rr = tid / NTN / 32;
      if (oh0 + rr < g.Ho && ow0 + v < g.Wo)
        o = __ldg(reinterpret_cast<const uint4*>(dy + ((((long long)n * g.Do + od) * g.Ho + oh0 + rr) * g.Wo + ow0 + v) * COUT + c8 * 8));
    }
    return o;
  };
  auto store_dy = [&](const uint4 o, int buf) {
    if (tid < dyvecs) {
      float f[8];
      unpack8(o, f);
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] *= S;
      *reinterpret_cast<uint4*>(dys + (size_t)buf * dbuf + (size_t)tid * 8) = pack8h(f);
    }
  };

  int tile = blockIdx.x, buf = 0;
  if (tile < ntiles) { stage_x(tile, 0); store_dy(load_dy(tile), 0); }
  for (; tile < ntiles; tile += gridDim.x, buf ^= 1) {
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();                                        // tile `buf` staged; everyone is done with buffer buf ^ 1
    const int nxt = tile + gridDim.x;
    uint4 dq = make_uint4(0u, 0u, 0u, 0u);
    if (nxt < ntiles) { stage_x(nxt, buf ^ 1); dq = load_dy(nxt); }
    const uint32_t xa = xs_addr + (uint32_t)(buf * xbuf * 2), da = dys_addr + (uint32_t)(buf * dbuf * 2);
    for (int kc = 0; kc < R * 2; ++kc) {
      const int rr = kc >> 1, wh = kc & 1;
      const int koff = (rr * g.sh * XW + wh * 16 * g.sw) * VS;
      uint32_t b0[NTN], b1[NTN];
#pragma unroll
      for (int j = 0; j < NTN; ++j) {
        const uint32_t baddr = da + (uint32_t)(((rr * 32 + wh * 16 + (lane & 15)) * COUT + j * 8) * 2);
        asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];\n" : "=r"(b0[j]), "=r"(b1[j]) : "r"(baddr));
      }
#pragma unroll
      for (int i = 0; i < MAXU; ++i) {
        uint32_t a0, a1, a2, a3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(xa + (uint32_t)((ubase[i] + koff) * 2)));
#pragma unroll
        for (int j = 0; j < NTN; ++j)
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                       : "+f"(acc[i][j][0]), "+f"(acc[i][j][1]), "+f"(acc[i][j][2]), "+f"(acc[i][j][3])
                       : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0[j]), "r"(b1[j]));
      }
    }
    if (nxt < ntiles) store_dy(dq, buf ^ 1);
  }
  const float invS = 1.f / S;
  const int gq = lane >> 2, t2 = (lane & 3) * 2;
#pragma unroll
  for (int i = 0; i < MAXU; ++i) {
    const int u = warp + NW * i;
    if (u >= nunits) continue;
#pragma unroll
    for (int hsel = 0; hsel < 2; ++hsel) {
      int tap, ci;
      if (CIN >= 16) { tap = u / C16; ci = (u % C16) * 16 + gq + hsel * 8; }
      else { tap = 2 * u + hsel; ci = gq; }
      if (tap >= taps) continue;
#pragma unroll
      for (int j = 0; j < NTN; ++j) {
        const int co = j * 8 + t2;
        atomicAdd(&dw[((long long)co * CIN + ci) * taps + tap], acc[i][j][hsel * 2] * invS);
        atomicAdd(&dw[((long long)(co + 1) * CIN + ci) * taps + tap], acc[i][j][hsel * 2 + 1] * invS);
      }
    }
  }
}

__device__ unsigned g_rn_amax_slot[1];

static bool rn_wgrad16_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("MMNN_RN_WGRAD16"); v = (e != nullptr && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

template <int CIN, int NTN, int MAXU, int NW = 8>
static int launch_wgrad_mma16(const RnConvGeom& g, const void* x, const void* dy, float* dw, cudaStream_t st) {
  constexpr int VS = (CIN == 64) ? 72 : ((CIN == 16) ? 24 : 8);
  const int XW = 31 * g.sw + g.kw;
  int R = 4;
  size_t smem = 0;
  for (;; R >>= 1) {
    const int HRs = (R - 1) * g.sh + g.kh;
    smem = 2 * ((size_t)g.kd * HRs * XW * VS + (size_t)R * 32 * 8 * NTN) * 2;
    if (smem <= 120 * 1024 || R == 1) break;
  }
  if (smem > 220 * 1024) return -8;                         // caller falls back to the converting variant
  auto kern = rn_wgrad_mma16_kernel<CIN, NTN, MAXU, NW>;
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    smem_set = smem;
  }
  unsigned* slot = nullptr;
  cudaError_t e = cudaGetSymbolAddress((void**)&slot, g_rn_amax_slot);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemsetAsync(slot, 0, sizeof(unsigned), st);
  if (e != cudaSuccess) return (int)e;
  const long long n8 = (long long)g.N * g.Do * g.Ho * g.Wo * g.Cout / 8;
  long long ab = (n8 + THREADS - 1) / THREADS;
  if (ab > 148 * 8) ab = 148 * 8;
  rn_absmax_kernel<<<(unsigned)ab, THREADS, 0, st>>>((const uint4*)dy, n8, slot);
  const long long ntiles = (long long)g.N * g.Do * ((g.Ho + R - 1) / R) * ((g.Wo + 31) / 32);
  if (ntiles > 0x7fffffffLL) return -6;
  int bps = (int)((200 * 1024) / (smem + 1024));
  const int bmax = (MAXU * NTN <= 4) ? 4 : 2;               // matches __launch_bounds__
  if (bps > bmax) bps = bmax;
  if (bps < 1 || NW > 8) bps = 1;
  const int blocks = (int)(ntiles < 148LL * bps ? ntiles : 148LL * bps);
  kern<<<blocks, NW * 32, smem, st>>>(g, (const __half*)x, (const uint16_t*)dy, dw, R, slot);
  return (int)cudaGetLastError();
}

template <int CIN, int NTN>
static int dispatch_wgrad_mma(const RnConvGeom& g, const void* x, const void* dy, float* dw, cudaStream_t st) {
  const int taps = g.kd * g.kh * g.kw;
  const int nunits = (CIN >= 16) ? taps * (CIN / 16) : (taps + 1) / 2;
  const int per = (nunits + 7) / 8;
  if (rn_wgrad16_enabled()) {
    int rc = -8;
    if (per <= 1) rc = launch_wgrad_mma16<CIN, NTN, 1>(g, x, dy, dw, st);
    else if (per <= 2) rc = launch_wgrad_mma16<CIN, NTN, 2>(g, x, dy, dw, st);
    else if (per <= 4) rc = launch_wgrad_mma16<CIN, NTN, 4>(g, x, dy, dw, st);
    else if (per <= 14 && NTN == 1) rc = launch_wgrad_mma16<CIN, NTN, (NTN == 1 ? 7 : 4), 16>(g, x, dy, dw, st);
    if (rc != -8) return rc;
  }
  if (per <= 1) return launch_wgrad_mma<CIN, NTN, 1>(g, x, dy, dw, st);
  if (per <= 2) return launch_wgrad_mma<CIN, NTN, 2>(g, x, dy, dw, st);
  if (per <= 4) return launch_wgrad_mma<CIN, NTN, 4>(g, x, dy, dw, st);
  if (per <= 14 && NTN == 1) return launch_wgrad_mma<CIN, NTN, (NTN == 1 ? 14 : 4)>(g, x, dy, dw, st);
  return -8;
}

// ---- the stem, Conv3d(1 -> 64, k (1,7,7), s (1,2,2), p (pd,3,3)) on a single-channel fp32 image, on HMMA through an
// explicit im2col in shared memory: tile = 32 voxels of one output row; its 7 input rows (69 voxels) are read once
// (coalesced fp32), converted to 16 bit, expanded to A_s[32 voxels][49 -> 64 taps]; forward: M = 16 voxels, N = 64 channels
// (8 warps = 2 m-tiles x 4 channel quarters), K = 4 k16 chunks of taps; the 32 x 64 output tile is staged in shared memory
// so each voxel's 128 bytes leave as one line, statistics from the staged (rounded) values.  Weight gradient: M = 64
// channels (dy^T by ldmatrix.trans), N = 56 taps (im2col by ldmatrix.trans), K = the tile's 32 voxels; bf16 operands.
constexpr int ST_XW = 72, ST_AS = 72;

template <bool BF>
__device__ __forceinline__ uint16_t st_cvt(float v) {
  if (BF) { const __nv_bfloat16 h = __float2bfloat16_rn(v); return *reinterpret_cast<const uint16_t*>(&h); }
  const __half h = __float2half_rn(v);
  return *reinterpret_cast<const uint16_t*>(&h);
}

template <bool BF>
__device__ __forceinline__ void stem_stage(const RnConvGeom& g, const float* __restrict__ x, int n, int od, int oh, int ow0,
                                           uint16_t* in_s, uint16_t* A_s, int tid) {
  const int zd = od * g.sd - g.pd;
  const bool d_ok = (unsigned)zd < (unsigned)g.Di;
  for (int i = tid; i < 7 * ST_XW; i += THREADS) {
    const int b = i / ST_XW, p = i % ST_XW;
    const int zh = oh * 2 - 3 + b, zw = ow0 * 2 - 3 + p;
    float v = 0.f;
    if (d_ok && p < 69 && (unsigned)zh < (unsigned)g.Hi && (unsigned)zw < (unsigned)g.Wi)
      v = __ldg(x + (((long long)n * g.Di + zd) * g.Hi + zh) * g.Wi + zw);
    in_s[i] = st_cvt<BF>(v);
  }
  __syncthreads();
  for (int i = tid; i < 32 * 64; i += THREADS) {
    const int v = i >> 6, tap = i & 63;
    uint16_t val = 0;
    if (tap < 49) { const int b = tap / 7, c = tap % 7; val = in_s[b * ST_XW + 2 * v + c]; }
    A_s[v * ST_AS + tap] = val;
  }
}

__global__ void __launch_bounds__(THREADS, 4) rn_stem_mma_fwd_kernel(const RnConvGeom g, const float* __restrict__ x,
                                                                     const float* __restrict__ w, __half* __restrict__ y,
                                                                     double* __restrict__ stats) {
  __shared__ __align__(16) uint16_t in_s[7 * ST_XW];
  __shared__ __align__(16) uint16_t A_s[32 * ST_AS];
  __shared__ __align__(16) uint16_t out_s[32 * ST_AS];
  __shared__ __align__(16) uint2 wb[4 * 8 * 32];
  __shared__ float sstat[128];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 4 * 8 * 32; i += THREADS) {
    const int l = i & 31, nt = (i >> 5) & 7, kc = i >> 8;
    const int n = nt * 8 + (l >> 2), k0 = kc * 16 + (l & 3) * 2;
    const float* pw = w + (long long)n * 49;
    const float w0 = k0 < 49 ? pw[k0] : 0.f, w1 = k0 + 1 < 49 ? pw[k0 + 1] : 0.f;
    const float w8 = k0 + 8 < 49 ? pw[k0 + 8] : 0.f, w9 = k0 + 9 < 49 ? pw[k0 + 9] : 0.f;
    wb[i] = make_uint2(pack_h2(w0, w1), pack_h2(w8, w9));
  }
  if (tid < 128) sstat[tid] = 0.f;
  float ssum = 0.f, ssq = 0.f;
  const int tiles_w = (g.Wo + 31) / 32;
  const int ntiles = g.N * g.Do * g.Ho * tiles_w;
  const int mt = warp & 1, nq = warp >> 1;
  const int row_l = (lane & 7) + ((lane >> 3) & 1) * 8, koff = (lane >> 4) * 8;
  const uint32_t a_addr = (uint32_t)__cvta_generic_to_shared(A_s + (mt * 16 + row_l) * ST_AS + koff);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int oh = r_ % g.Ho;
    r_ /= g.Ho;
    const int od = r_ % g.Do, n = r_ / g.Do;
    const int ow0 = tw * 32;
    stem_stage<false>(g, x, n, od, oh, ow0, in_s, A_s, tid);
    __syncthreads();
    float acc[2][4];
#pragma unroll
    for (int j = 0; j < 2; ++j) { acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f; }
#pragma unroll
    for (int kc = 0; kc < 4; ++kc) {
      uint32_t a0, a1, a2, a3;
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                   : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(a_addr + kc * 32));
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const uint2 bf = wb[(kc * 8 + nq * 2 + j) * 32 + lane];
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                     : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.x), "r"(bf.y));
      }
    }
    const int gq = lane >> 2, t2 = (lane & 3) * 2;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      *reinterpret_cast<uint32_t*>(out_s + (mt * 16 + gq) * ST_AS + (nq * 2 + j) * 8 + t2) = pack_h2(acc[j][0], acc[j][1]);
      *reinterpret_cast<uint32_t*>(out_s + (mt * 16 + gq + 8) * ST_AS + (nq * 2 + j) * 8 + t2) = pack_h2(acc[j][2], acc[j][3]);
    }
    __syncthreads();
    {
      const int v = tid >> 3, chunk = tid & 7;
      if (ow0 + v < g.Wo)
        *reinterpret_cast<uint4*>(y + ((((long long)n * g.Do + od) * g.Ho + oh) * g.Wo + ow0 + v) * 64 + chunk * 8) =
            *reinterpret_cast<const uint4*>(out_s + v * ST_AS + chunk * 8);
      const int c = tid & 63, vg = tid >> 6;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int vv = vg * 8 + k;
        if (ow0 + vv < g.Wo) {
          const float f = __half2float(*reinterpret_cast<const __half*>(out_s + vv * ST_AS + c));
          ssum += f; ssq = fmaf(f, f, ssq);
        }
      }
    }
  }
  if (stats != nullptr) {
    RN_WARP_ORDERED(THREADS / 32, { sstat[tid & 63] += ssum; sstat[64 + (tid & 63)] += ssq; })
    if (tid < 128) atomicAdd(&stats[tid], (double)sstat[tid]);
  }
}

__global__ void __launch_bounds__(THREADS, 4) rn_stem_mma_wgrad_kernel(const RnConvGeom g, const float* __restrict__ x,
                                                                       const uint16_t* __restrict__ dy, float* __restrict__ dw) {
  __shared__ __align__(16) uint16_t in_s[7 * ST_XW];
  __shared__ __align__(16) uint16_t A_s[32 * ST_AS];
  __shared__ __align__(16) uint16_t dy_s[32 * ST_AS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tiles_w = (g.Wo + 31) / 32;
  const int ntiles = g.N * g.Do * g.Ho * tiles_w;
  const int mt = warp & 3, nh = warp >> 2;
  const int q = lane >> 3;
  const uint32_t a_addr = (uint32_t)__cvta_generic_to_shared(dy_s + ((lane & 7) + (q >> 1) * 8) * ST_AS + mt * 16 + (q & 1) * 8);
  const uint32_t b_addr = (uint32_t)__cvta_generic_to_shared(A_s + (lane & 15) * ST_AS + nh * 32);
  float acc[4][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f; }
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int oh = r_ % g.Ho;
    r_ /= g.Ho;
    const int od = r_ % g.Do, n = r_ / g.Do;
    const int ow0 = tw * 32;
    __syncthreads();                                        // previous tile's fragments are loaded
    {
      const int v = tid >> 3, chunk = tid & 7;
      const bool ok = ow0 + v < g.Wo;
      const uint16_t* sp = ok ? dy + ((((long long)n * g.Do + od) * g.Ho + oh) * g.Wo + ow0 + v) * 64 + chunk * 8 : dy;
      cp_async_zfill<16>(dy_s + v * ST_AS + chunk * 8, sp, ok);
      asm volatile("cp.async.commit_group;\n" ::: "memory");
    }
    stem_stage<true>(g, x, n, od, oh, ow0, in_s, A_s, tid);
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();
#pragma unroll
    for (int kc = 0; kc < 2; ++kc) {
      uint32_t a0, a1, a2, a3;
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                   : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(a_addr + kc * 16 * ST_AS * 2));
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t b0, b1;
        asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];\n"
                     : "=r"(b0), "=r"(b1) : "r"(b_addr + (kc * 16 * ST_AS + j * 8) * 2));
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                     : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
      }
    }
  }
  const int gq = lane >> 2, t2 = (lane & 3) * 2;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int tap = (nh * 4 + j) * 8 + t2;
    const int co = mt * 16 + gq;
    if (tap < 49) { atomicAdd(&dw[co * 49 + tap], acc[j][0]); atomicAdd(&dw[(co + 8) * 49 + tap], acc[j][2]); }
    if (tap + 1 < 49) { atomicAdd(&dw[co * 49 + tap + 1], acc[j][1]); atomicAdd(&dw[(co + 8) * 49 + tap + 1], acc[j][3]); }
  }
}

static bool rn_is_stem(const RnConvGeom& g) {
  return g.Cin == 1 && g.Cout == 64 && g.kd == 1 && g.kh == 7 && g.kw == 7 && g.sd == 1 && g.sh == 2 && g.sw == 2 && g.ph == 3 &&
         g.pw == 3;
}

// ---- 16-channel source, 16 outputs, 3x3x3 stride 1 pad 1 (layer2 / layer4): one tap = one k16.  The rows of these stages
// are 16 (or fewer) voxels wide, so the tile shape adapts: TWm m-tiles along W (1 when Wo <= 16) x 8 / TWm rows.
template <bool DGRAD>
__global__ void __launch_bounds__(THREADS, 2) rn_conv3_k16_mma_kernel(const RnConvGeom g, const uint16_t* __restrict__ src,
                                                                      const float* __restrict__ w, uint16_t* __restrict__ dst,
                                                                      const uint16_t* __restrict__ add, double* __restrict__ stats,
                                                                      int TWm) {
  constexpr int VS = 24;
  const int R = 8 / TWm, HR = R + 2, XW = 16 * TWm + 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint16_t* xs = reinterpret_cast<uint16_t*>(smem_raw);
  uint2* wb = reinterpret_cast<uint2*>(smem_raw + (size_t)3 * HR * XW * VS * 2);
  float* sstat = reinterpret_cast<float*>(wb + 27 * 2 * 32);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 27 * 2 * 32; i += THREADS) {
    const int l = i & 31, j = (i >> 5) & 1, tap = i >> 6;
    const int n = 8 * j + (l >> 2), k = (l & 3) * 2;
    float v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int kk = k + (q & 1) + (q >> 1) * 8;
      const int co = DGRAD ? kk : n, ci = DGRAD ? n : kk;
      v[q] = w[((long long)co * 16 + ci) * 27 + tap];
    }
    wb[i] = DGRAD ? make_uint2(pack2(v[0], v[1]), pack2(v[2], v[3])) : make_uint2(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]));
  }
  if (tid < 32) sstat[tid] = 0.f;
  float ssum[4] = {0.f, 0.f, 0.f, 0.f}, ssq[4] = {0.f, 0.f, 0.f, 0.f};
  const int tiles_w = (g.Wo + 16 * TWm - 1) / (16 * TWm), tiles_h = (g.Ho + R - 1) / R;
  const int ntiles = g.N * g.Do * tiles_h * tiles_w;
  const int rr = warp / TWm, wbase = (warp % TWm) * 16;
  const int row_l = (lane & 7) + ((lane >> 3) & 1) * 8, koff = (lane >> 4) * 8;
  const uint32_t xs_addr = (uint32_t)__cvta_generic_to_shared(xs);
  uint32_t toff[27];
#pragma unroll
  for (int tap = 0; tap < 27; ++tap) {
    int a = tap / 9, b = (tap / 3) % 3, c = tap % 3;
    if (DGRAD) { a = 2 - a; b = 2 - b; c = 2 - c; }
    toff[tap] = (uint32_t)((((a * HR + rr + b) * XW + wbase + c + row_l) * VS + koff) * 2);
  }
  const float inv_xw = 1.0f / (float)XW, inv_hr = 1.0f / (float)HR;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tw = tile % tiles_w;
    int r_ = tile / tiles_w;
    const int th = r_ % tiles_h;
    r_ /= tiles_h;
    const int od = r_ % g.Do, n = r_ / g.Do;
    const int oh0 = th * R, ow0 = tw * 16 * TWm;
    __syncthreads();
    for (int i = tid; i < 3 * HR * XW * 2; i += THREADS) {
      const int ch = i & 1, vp = i >> 1;
      const int r = __float2int_rd(((float)vp + 0.5f) * inv_xw), p = vp - r * XW;
      const int a = __float2int_rd(((float)r + 0.5f) * inv_hr), hb = r - a * HR;
      const int zd = od - 1 + a, zh = oh0 - 1 + hb, zw = ow0 - 1 + p;
      const bool ok = (unsigned)zd < (unsigned)g.Do && (unsigned)zh < (unsigned)g.Ho && (unsigned)zw < (unsigned)g.Wo;
      const uint16_t* sp = ok ? src + ((((long long)n * g.Do + zd) * g.Ho + zh) * g.Wo + zw) * 16 + ch * 8 : src;
      cp_async_zfill<16>(xs + vp * VS + ch * 8, sp, ok);
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();
    float acc[2][4];
#pragma unroll
    for (int j = 0; j < 2; ++j) { acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f; }
#pragma unroll
    for (int tap = 0; tap < 27; ++tap) {
      uint32_t a0, a1, a2, a3;
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                   : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(xs_addr + toff[tap]));
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const uint2 bf = wb[(tap * 2 + j) * 32 + lane];
        if (DGRAD)
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                       : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                       : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.x), "r"(bf.y));
        else
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                       : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                       : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.x), "r"(bf.y));
      }
    }
    const int oh = oh0 + rr, gq = lane >> 2, t2 = (lane & 3) * 2;
    if (oh < g.Ho) {
      const long long rowbase = (((long long)n * g.Do + od) * g.Ho + oh) * g.Wo;
#pragma unroll
      for (int hsel = 0; hsel < 2; ++hsel) {
        const int ow = ow0 + wbase + gq + hsel * 8;
        if (ow < g.Wo) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            float v0 = acc[j][hsel * 2], v1 = acc[j][hsel * 2 + 1];
            const long long o = (rowbase + ow) * 16 + j * 8 + t2;
            if (add != nullptr) {
              const uint32_t u = *reinterpret_cast<const uint32_t*>(add + o);
              if (DGRAD) { v0 += bf_lo(u); v1 += bf_hi(u); }
              else { const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u)); v0 += f.x; v1 += f.y; }
            }
            if (DGRAD) {
              *reinterpret_cast<uint32_t*>(dst + o) = pack2(v0, v1);
            } else {
              const __half2 h = __floats2half2_rn(v0, v1);
              *reinterpret_cast<__half2*>(dst + o) = h;
              const float2 f = __half22float2(h);
              ssum[j * 2] += f.x; ssum[j * 2 + 1] += f.y;
              ssq[j * 2] = fmaf(f.x, f.x, ssq[j * 2]); ssq[j * 2 + 1] = fmaf(f.y, f.y, ssq[j * 2 + 1]);
            }
          }
        }
      }
    }
  }
  if (stats != nullptr) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
      for (int off = 4; off < 32; off <<= 1) {
        ssum[k] += __shfl_xor_sync(0xffffffffu, ssum[k], off);
        ssq[k] += __shfl_xor_sync(0xffffffffu, ssq[k], off);
      }
    }
    RN_WARP_ORDERED(THREADS / 32, if (lane < 4) {
      _Pragma("unroll") for (int k = 0; k < 4; ++k) {
        const int co = (k >> 1) * 8 + lane * 2 + (k & 1);
        sstat[co] += ssum[k];
        sstat[16 + co] += ssq[k];
      }
    })
    if (tid < 32) atomicAdd(&stats[tid], (double)sstat[tid]);
  }
}

template <bool DGRAD>
static int launch_conv3_k16_mma(const RnConvGeom& g, const void* src, const float* w, void* dst, const void* add, double* stats,
                                cudaStream_t st) {
  const int TWm = g.Wo > 16 ? 2 : 1;
  const int R = 8 / TWm, HR = R + 2, XW = 16 * TWm + 2;
  const size_t smem = (size_t)3 * HR * XW * 24 * 2 + 27 * 2 * 32 * 8 + 32 * 4;
  auto kern = rn_conv3_k16_mma_kernel<DGRAD>;
  static bool attr = false;
  if (!attr) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  const long long ntiles = (long long)g.N * g.Do * ((g.Ho + R - 1) / R) * ((g.Wo + 16 * TWm - 1) / (16 * TWm));
  if (ntiles > 0x7fffffffLL || smem > 64 * 1024) return -6;
  const int blocks = (int)(ntiles < 148 * 3 ? ntiles : 148 * 3);
  kern<<<blocks, THREADS, smem, st>>>(g, (const uint16_t*)src, w, (uint16_t*)dst, (const uint16_t*)add, stats, TWm);
  return (int)cudaGetLastError();
}

static bool rn_mma_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("MMNN_RN_MMA"); v = (e != nullptr && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

static int launch_conv3_mma_fwd(const RnConvGeom& g, const void* x, const float* w, void* y, double* stats, cudaStream_t st,
                                const float* w_ds = nullptr, void* y_ds = nullptr, double* stats_ds = nullptr) {
  static bool attr = false;
  if (!attr) {
    const cudaError_t e = cudaFuncSetAttribute(rn_conv3_mma_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MF_SMEM);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  const long long ntiles = (long long)g.N * g.Do * ((g.Ho + MF_R - 1) / MF_R) * ((g.Wo + 31) / 32);
  if (ntiles > 0x7fffffffLL) return -6;
  const int blocks = (int)(ntiles < 296 ? ntiles : 296);
  rn_conv3_mma_fwd_kernel<<<blocks, THREADS, MF_SMEM, st>>>(g, (const __half*)x, w, (__half*)y, stats, w_ds, (__half*)y_ds, stats_ds);
  return (int)cudaGetLastError();
}

struct WgTile { int n, od, oh, ow0; };
__device__ __forceinline__ WgTile wg_decode(long long tile, int tiles_w, const RnConvGeom& g) {
  WgTile t;
  t.ow0 = (int)(tile % tiles_w) * WG_TW;
  long long r = tile / tiles_w;
  t.oh = (int)(r % g.Ho);
  r /= g.Ho;
  t.od = (int)(r % g.Do);
  t.n = (int)(r / g.Do);
  return t;
}

template <typename TX, int CIN, int MAXI>
__global__ void __launch_bounds__(THREADS, (MAXI > 2 ? 2 : 3)) rn_wgrad_kernel(const RnConvGeom g, const TX* __restrict__ x,
                                                                              const uint16_t* __restrict__ dy,
                                                                              float* __restrict__ dw, int tiles_w,
                                                                              long long ntiles) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int taps = g.kd * g.kh * g.kw;
  const int items = taps * CIN * (g.Cout / 8);
  const int tid = threadIdx.x;
  const int XW = (WG_TW - 1) * g.sw + g.kw;               // staged voxels per input row
  const int rowlen = XW * CIN;                            // elements per staged input row
  const int nrows = g.kd * g.kh;
  const int xbuf = nrows * rowlen;                        // elements per x buffer (a multiple of 8 when CIN >= 8)
  const int xbuf_al = (xbuf + 7) & ~7;
  float* dy_s = reinterpret_cast<float*>(smem_raw);       // [2][WG_TW][Cout] fp32
  TX* x_s = reinterpret_cast<TX*>(smem_raw + (size_t)2 * WG_TW * g.Cout * sizeof(float));   // [2][kd*kh][XW][CIN]
  int xo[MAXI], icog[MAXI], dyo[MAXI];
  float acc[MAXI][8];
#pragma unroll
  for (int j = 0; j < MAXI; ++j) {
    const int it = tid + j * THREADS;
    const int ci = it % CIN, rest = it / CIN;
    const int tap = rest % taps;
    icog[j] = (it < items) ? rest / taps : -1;
    const int a = tap / (g.kh * g.kw), b = (tap / g.kw) % g.kh, c = tap % g.kw;
    xo[j] = (it < items) ? ((a * g.kh + b) * XW + c) * CIN + ci : 0;      // idle items read element 0 (branch-free inner loop)
    dyo[j] = (it < items) ? (rest / taps) * 8 : 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[j][k] = 0.f;
  }
  const bool one = (g.Cout == 8);
  const int step = g.sw * CIN;
  constexpr int VEC = (CIN * (int)sizeof(TX) >= 16) ? 16 / (int)sizeof(TX) : 1;     // elements per cp.async
  constexpr int CPB = VEC * (int)sizeof(TX);                                          // 16 or 4 bytes
  static_assert(CPB == 16 || CPB == 4, "cp.async size");
  const int dyvecs = WG_TW * g.Cout / 8;                  // <= 64: one uint4 of dy per thread

  auto stage_x = [&](const WgTile& t, int buf) {
    TX* xs = x_s + (size_t)buf * xbuf_al;
    const int iw0 = t.ow0 * g.sw - g.pw;
    const int per_row = rowlen / VEC;
    for (int a = 0; a < g.kd; ++a) {
      const int zd = t.od * g.sd - g.pd + a;
      for (int b = 0; b < g.kh; ++b) {
        const int zh = t.oh * g.sh - g.ph + b;
        const bool row_ok = (unsigned)zd < (unsigned)g.Di && (unsigned)zh < (unsigned)g.Hi;
        const long long rowbase = (((long long)t.n * g.Di + zd) * g.Hi + zh) * g.Wi;
        TX* xr = xs + (a * g.kh + b) * rowlen;
        for (int j = tid; j < per_row; j += THREADS) {
          const int e = j * VEC;
          const int zw = iw0 + e / CIN;
          const bool ok = row_ok && (unsigned)zw < (unsigned)g.Wi;
          const TX* src = ok ? x + (rowbase + zw) * CIN + e % CIN : x;
          cp_async_zfill<CPB>(xr + e, src, ok);
        }
      }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };
  auto load_dy = [&](const WgTile& t) -> uint4 {
    uint4 q = make_uint4(0u, 0u, 0u, 0u);
    if (tid < dyvecs) {
      const int v = tid / (g.Cout / 8), c8 = tid % (g.Cout / 8);
      if (t.ow0 + v < g.Wo)
        q = __ldg(reinterpret_cast<const uint4*>(dy + ((((long long)t.n * g.Do + t.od) * g.Ho + t.oh) * g.Wo + t.ow0 + v) * g.Cout + c8 * 8));
    }
    return q;
  };
  auto store_dy = [&](const uint4 q, int buf) {
    if (tid < dyvecs) {
      float d[8];
      unpack8(q, d);
      float4* dst = reinterpret_cast<float4*>(dy_s + (size_t)buf * WG_TW * g.Cout + tid * 8);
      dst[0] = make_float4(d[0], d[1], d[2], d[3]);
      dst[1] = make_float4(d[4], d[5], d[6], d[7]);
    }
  };

  long long tile = blockIdx.x;
  if (tile < ntiles) {
    const WgTile t0 = wg_decode(tile, tiles_w, g);
    stage_x(t0, 0);
    store_dy(load_dy(t0), 0);
  }
  int buf = 0;
  for (; tile < ntiles; tile += gridDim.x, buf ^= 1) {
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();                                      // tile `buf` staged; everyone is done with buffer buf^1
    const long long nxt = tile + gridDim.x;
    uint4 dq = make_uint4(0u, 0u, 0u, 0u);
    if (nxt < ntiles) {
      const WgTile tn = wg_decode(nxt, tiles_w, g);
      stage_x(tn, buf ^ 1);
      dq = load_dy(tn);
    }
    const TX* xs = x_s + (size_t)buf * xbuf_al;
    const float* ds = dy_s + (size_t)buf * WG_TW * g.Cout;
#pragma unroll 4
    for (int v = 0; v < WG_TW; ++v) {
      float d[8];
      if (one) {
        const float4 d0 = *reinterpret_cast<const float4*>(ds + v * 8), d1 = *reinterpret_cast<const float4*>(ds + v * 8 + 4);
        d[0] = d0.x; d[1] = d0.y; d[2] = d0.z; d[3] = d0.w; d[4] = d1.x; d[5] = d1.y; d[6] = d1.z; d[7] = d1.w;
      }
#pragma unroll
      for (int j = 0; j < MAXI; ++j) {
        const float xv = wg_ld(xs + xo[j] + v * step);
        if (!one) {
          const float* pd = ds + v * g.Cout + dyo[j];
          const float4 d0 = *reinterpret_cast<const float4*>(pd), d1 = *reinterpret_cast<const float4*>(pd + 4);
          d[0] = d0.x; d[1] = d0.y; d[2] = d0.z; d[3] = d0.w; d[4] = d1.x; d[5] = d1.y; d[6] = d1.z; d[7] = d1.w;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[j][k] = fmaf(xv, d[k], acc[j][k]);
      }
    }
    if (nxt < ntiles) store_dy(dq, buf ^ 1);
  }
#pragma unroll
  for (int j = 0; j < MAXI; ++j) {
    if (icog[j] < 0) continue;
    const int it = tid + j * THREADS;
    const int ci = it % CIN, tap = (it / CIN) % taps;
#pragma unroll
    for (int k = 0; k < 8; ++k)
      atomicAdd(&dw[((long long)(icog[j] * 8 + k) * CIN + ci) * taps + tap], acc[j][k]);
  }
}

template <typename TX, int CIN, int MAXI>
static int launch_wgrad(const RnConvGeom& g, const void* x, const void* dy, float* dw, cudaStream_t st) {
  const int tiles_w = (g.Wo + WG_TW - 1) / WG_TW;
  const long long ntiles = (long long)g.N * g.Do * g.Ho * tiles_w;
  const int XW = (WG_TW - 1) * g.sw + g.kw;
  const size_t xbuf_al = ((size_t)g.kd * g.kh * XW * CIN + 7) & ~(size_t)7;
  const size_t smem = (size_t)2 * WG_TW * g.Cout * sizeof(float) + 2 * xbuf_al * sizeof(TX);
  if (WG_TW * g.Cout / 8 > THREADS) return -5;
  auto kern = rn_wgrad_kernel<TX, CIN, MAXI>;
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    smem_set = smem;
  }
  long long blocks = ntiles;
  const long long cap = 148LL * (MAXI > 2 ? 2 : 3);
  if (blocks > cap) blocks = cap;
  kern<<<(unsigned)blocks, THREADS, smem, st>>>(g, (const TX*)x, (const uint16_t*)dy, dw, tiles_w, ntiles);
  return (int)cudaGetLastError();
}

template <int CIN>
static int dispatch_wgrad_h(const RnConvGeom& g, int per, const void* x, const void* dy, float* dw, cudaStream_t st) {
  if (per <= 1) return launch_wgrad<__half, CIN, 1>(g, x, dy, dw, st);
  if (per <= 2) return launch_wgrad<__half, CIN, 2>(g, x, dy, dw, st);
  if (per <= 4) return launch_wgrad<__half, CIN, 4>(g, x, dy, dw, st);
  if (per <= 7) return launch_wgrad<__half, CIN, 7>(g, x, dy, dw, st);
  return -4;
}

// ------------------------------------------------------------------------------------------------ BatchNorm coefficients
// coef [4][C]: scale = gamma * rstd, shift = beta - mean * scale, mean, rstd.  Training: batch statistics (biased variance
// for the normalisation, unbiased for the running update, momentum 0.1 -- torch defaults, SURVEY.md row a-17).
__global__ void rn_bn_coeffs_kernel(const double* __restrict__ stats, double count, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, float* rmean, float* rvar, long long* nbt, float eps,
                                    float momentum, int training, int C, float* __restrict__ coef) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0 && training && nbt != nullptr) *nbt += 1;
  if (c >= C) return;
  double mean, var;
  if (training) {
    mean = stats[c] / count;
    var = stats[C + c] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const double unb = count > 1.0 ? var * count / (count - 1.0) : var;
    rmean[c] = (float)((1.0 - (double)momentum) * (double)rmean[c] + (double)momentum * mean);
    rvar[c] = (float)((1.0 - (double)momentum) * (double)rvar[c] + (double)momentum * unb);
  } else {
    mean = (double)rmean[c];
    var = (double)rvar[c];
  }
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float sc = gamma[c] * rstd;
  coef[c] = sc;
  coef[C + c] = beta[c] - (float)mean * sc;
  coef[2 * C + c] = (float)mean;
  coef[3 * C + c] = rstd;
}

// ------------------------------------------------------------------------------------------------ element-wise passes
__device__ __forceinline__ float hash_uniform(unsigned long long seed, unsigned long long e) {
  unsigned long long z = seed + e * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (float)(z >> 40) * (1.0f / 16777216.0f);
}

// y = [relu]( raw * scale + shift  [+ res | + raw2 * scale2 + shift2] )  [ * keep / (1 - p) ]
// RES 0: none, 1: identity tensor, 2: second BatchNorm'ed raw tensor (the down-sample branch).
template <int RES>
__global__ void __launch_bounds__(THREADS) rn_bn_act_kernel(const uint4* __restrict__ raw, const float* __restrict__ coef,
                                                            const uint4* __restrict__ res, const float* __restrict__ coef2,
                                                            uint4* __restrict__ y, long long n8, int C, int relu,
                                                            float drop_p, unsigned long long seed,
                                                            const unsigned char* __restrict__ mask) {
  const int c0 = (threadIdx.x * 8) % C;
  float sc[8], sh[8], sc2[8], sh2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    sc[k] = coef[c0 + k]; sh[k] = coef[C + c0 + k];
    if (RES == 2) { sc2[k] = coef2[c0 + k]; sh2[k] = coef2[C + c0 + k]; }
  }
  const bool drop = drop_p > 0.f || mask != nullptr;
  const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  for (long long i = (long long)blockIdx.x * THREADS + threadIdx.x; i < n8; i += (long long)gridDim.x * THREADS) {
    float v[8], r[8];
    unpack8h(__ldg(raw + i), v);
    if (RES != 0) unpack8h(__ldg(res + i), r);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float o = fmaf(v[k], sc[k], sh[k]);
      if (RES == 1) o += r[k];
      if (RES == 2) o += fmaf(r[k], sc2[k], sh2[k]);
      if (relu) o = fmaxf(o, 0.f);
      if (drop) {
        const unsigned long long e = (unsigned long long)i * 8ull + k;
        const bool keep = mask != nullptr ? (mask[e] != 0) : (hash_uniform(seed, e) >= drop_p);
        o = keep ? o * keep_scale : 0.f;
      }
      v[k] = o;
    }
    y[i] = pack8h(v);
  }
}

// dz = dy * [y > 0] * post_scale.  sums [3][C] (fp64): sum dz, sum dz * xhat(raw), sum dz * xhat(raw2) (TWO only).
template <bool TWO>
__global__ void __launch_bounds__(THREADS) rn_act_bwd_reduce_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ y,
                                                                    float post_scale, const uint4* __restrict__ raw,
                                                                    const float* __restrict__ coef,
                                                                    const uint4* __restrict__ raw2,
                                                                    const float* __restrict__ coef2, double* __restrict__ sums,
                                                                    long long n8, int C) {
  __shared__ float sm[3 * 64];
  for (int i = threadIdx.x; i < 3 * C; i += THREADS) sm[i] = 0.f;
  __syncthreads();
  const int c0 = (threadIdx.x * 8) % C;
  float mean[8], rstd[8], mean2[8], rstd2[8], s0[8], s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    mean[k] = coef[2 * C + c0 + k]; rstd[k] = coef[3 * C + c0 + k];
    if (TWO) { mean2[k] = coef2[2 * C + c0 + k]; rstd2[k] = coef2[3 * C + c0 + k]; }
    s0[k] = 0.f; s1[k] = 0.f; s2[k] = 0.f;
  }
  for (long long i = (long long)blockIdx.x * THREADS + threadIdx.x; i < n8; i += (long long)gridDim.x * THREADS) {
    float g[8], yy[8], x[8], x2[8];
    unpack8(__ldg(dy + i), g);
    unpack8h(__ldg(y + i), yy);
    unpack8h(__ldg(raw + i), x);
    if (TWO) unpack8h(__ldg(raw2 + i), x2);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float dz = yy[k] > 0.f ? g[k] * post_scale : 0.f;
      s0[k] += dz;
      s1[k] = fmaf(dz, (x[k] - mean[k]) * rstd[k], s1[k]);
      if (TWO) s2[k] = fmaf(dz, (x2[k] - mean2[k]) * rstd2[k], s2[k]);
    }
  }
  // lanes l and l ^ off own the same 8 channels when 8 * off is a multiple of C: reduce those in registers first, so that
  // only C / 8 lanes per warp touch shared memory (ncu: the 6 144 same-address shared atomics of the first version showed
  // as short-scoreboard 11 / barrier 3.8 stall cycles per issue)
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    if ((off * 8) % C == 0) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        s0[k] += __shfl_xor_sync(0xffffffffu, s0[k], off);
        s1[k] += __shfl_xor_sync(0xffffffffu, s1[k], off);
        if (TWO) s2[k] += __shfl_xor_sync(0xffffffffu, s2[k], off);
      }
    }
  }
  RN_WARP_ORDERED(THREADS / 32, if ((int)(threadIdx.x & 31) < C / 8) {
    _Pragma("unroll") for (int k = 0; k < 8; ++k) {
      sm[c0 + k] += s0[k];
      sm[C + c0 + k] += s1[k];
      if (TWO) sm[2 * C + c0 + k] += s2[k];
    }
  })
  for (int i = threadIdx.x; i < (TWO ? 3 : 2) * C; i += THREADS) atomicAdd(&sums[i], (double)sm[i]);
}

// draw = gamma * rstd * (dz - mean(dz) - xhat * mean(dz * xhat))  (BatchNorm backward, training mode); eval_mode: draw =
// gamma * rstd * dz.  Optional second branch (down-sample BatchNorm) and optional dz output (identity residual).
template <bool TWO>
__global__ void __launch_bounds__(THREADS) rn_bn_bwd_apply_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ y,
                                                                  float post_scale, const uint4* __restrict__ raw,
                                                                  const float* __restrict__ coef, const uint4* __restrict__ raw2,
                                                                  const float* __restrict__ coef2,
                                                                  const double* __restrict__ sums, double inv_count,
                                                                  int eval_mode, uint4* __restrict__ draw,
                                                                  uint4* __restrict__ draw2, uint4* __restrict__ dzout,
                                                                  float* dgamma, float* dbeta, float* dgamma2, float* dbeta2,
                                                                  long long n8, int C) {
  if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < C; c += THREADS) {
      dbeta[c] = (float)sums[c];
      dgamma[c] = (float)sums[C + c];
      if (TWO) { dbeta2[c] = (float)sums[c]; dgamma2[c] = (float)sums[2 * C + c]; }
    }
  }
  const int c0 = (threadIdx.x * 8) % C;
  float mean[8], rstd[8], sc[8], m1[8], m2[8], mean2[8], rstd2[8], sc2[8], m22[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    sc[k] = coef[c0 + k]; mean[k] = coef[2 * C + c0 + k]; rstd[k] = coef[3 * C + c0 + k];
    m1[k] = eval_mode ? 0.f : (float)(sums[c0 + k] * inv_count);
    m2[k] = eval_mode ? 0.f : (float)(sums[C + c0 + k] * inv_count);
    if (TWO) {
      sc2[k] = coef2[c0 + k]; mean2[k] = coef2[2 * C + c0 + k]; rstd2[k] = coef2[3 * C + c0 + k];
      m22[k] = eval_mode ? 0.f : (float)(sums[2 * C + c0 + k] * inv_count);
    }
  }
  for (long long i = (long long)blockIdx.x * THREADS + threadIdx.x; i < n8; i += (long long)gridDim.x * THREADS) {
    float g[8], yy[8], x[8], x2[8], o[8], o2[8];
    unpack8(__ldg(dy + i), g);
    unpack8h(__ldg(y + i), yy);
    unpack8h(__ldg(raw + i), x);
    if (TWO) unpack8h(__ldg(raw2 + i), x2);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float dz = yy[k] > 0.f ? g[k] * post_scale : 0.f;
      g[k] = dz;
      o[k] = sc[k] * (dz - m1[k] - (x[k] - mean[k]) * rstd[k] * m2[k]);
      if (TWO) o2[k] = sc2[k] * (dz - m1[k] - (x2[k] - mean2[k]) * rstd2[k] * m22[k]);
    }
    draw[i] = pack8(o);
    if (TWO) draw2[i] = pack8(o2);
    if (dzout != nullptr) dzout[i] = pack8(g);
  }
}

// ------------------------------------------------------------------------------------------------ head
// AdaptiveAvgPool3d(1) -> flatten -> Linear(C -> K) -> sigmoid (/root/reference/models/resnet.py:165-170); one block per sample.
__global__ void __launch_bounds__(128) rn_head_fwd_kernel(const __half* __restrict__ y, int V, int C,
                                                          const float* __restrict__ W, const float* __restrict__ bias, int K,
                                                          float* __restrict__ pooled, float* __restrict__ out) {
  __shared__ float sp[64];
  __shared__ float sthr[128];
  const int b = blockIdx.x;
  const __half* py = y + (long long)b * V * C;
  // thread owns channel (tid % C) when 128 % C == 0 (C = 8 / 16 / 64); the 128 / C partial sums of a channel are added in thread order
  float s = 0.f;
  for (long long i = threadIdx.x; i < (long long)V * C; i += 128) s += __half2float(py[i]);
  sthr[threadIdx.x] = s;
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += 128) {
    float a = 0.f;
    for (int t = i; t < 128; t += C) a += sthr[t];
    sp[i] = a;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += 128) { sp[i] *= 1.f / (float)V; pooled[b * C + i] = sp[i]; }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += 128) {
    float z = bias[k];
    for (int i = 0; i < C; ++i) z = fmaf(W[k * C + i], sp[i], z);
    out[b * K + k] = 1.f / (1.f + expf(-z));
  }
}

// dlogit = dout * out * (1 - out); dW += dlogit^T pooled; db += sum dlogit; dy[b][v][c] = (dlogit W)[b][c] / V
__global__ void __launch_bounds__(128) rn_head_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ out,
                                                          const float* __restrict__ pooled, const float* __restrict__ W, int V,
                                                          int C, int K, __nv_bfloat16* __restrict__ dy, float* dW, float* db) {
  __shared__ float sdl[64];
  __shared__ float sdp[64];
  const int b = blockIdx.x;
  for (int k = threadIdx.x; k < K; k += 128) {
    const float o = out[b * K + k];
    sdl[k] = dout[b * K + k] * o * (1.f - o);
  }
  __syncthreads();
  if (b == 0) {
    // fc gradients: block 0 sums over the samples in index order (B x K x C terms: nothing) -- the per-sample blocks used to add
    // their terms with global atomics in arrival order.  dW / db are accumulated INTO (the caller passes zeroed or running totals).
    const int B = gridDim.x;
    for (int i = threadIdx.x; i < K * C + K; i += 128) {
      float acc = 0.f;
      for (int bb = 0; bb < B; ++bb) {
        const int k = i < K * C ? i / C : i - K * C;
        const float o = out[bb * K + k];
        const float dl = dout[bb * K + k] * o * (1.f - o);
        acc += i < K * C ? dl * pooled[bb * C + (i % C)] : dl;
      }
      if (i < K * C) dW[i] += acc; else db[i - K * C] += acc;
    }
  }
  for (int c = threadIdx.x; c < C; c += 128) {
    float s = 0.f;
    for (int k = 0; k < K; ++k) s = fmaf(sdl[k], W[k * C + c], s);
    sdp[c] = s / (float)V;
  }
  __syncthreads();
  __nv_bfloat16* pdy = dy + (long long)b * V * C;
  const __nv_bfloat16 val = __float2bfloat16_rn(sdp[threadIdx.x % C]);
  for (long long i = threadIdx.x; i < (long long)V * C; i += 128) pdy[i] = val;
}

static inline unsigned elt_grid(long long n8) {
  long long b = (n8 + THREADS - 1) / THREADS;
  const long long cap = 148LL * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

}  // namespace rn
}  // namespace mmnn

using namespace mmnn;
using namespace mmnn::rn;

extern "C" {

int mmnn_sizeof_rn_conv_geom(void) { return (int)sizeof(RnConvGeom); }

int mmnn_rn_conv(const RnConvGeom* g, int dgrad, int src_is_f32, const void* src, const float* w, void* dst, const void* add,
                 double* stats, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(dgrad ? PC_RN_DGRAD : PC_RN_FPROP, st);
  if (!dgrad && !src_is_f32 && add == nullptr && g->Cin == 64 && g->Cout == 8 && g->kd == 3 && g->kh == 3 && g->kw == 3 &&
      g->sd == 1 && g->sh == 1 && g->sw == 1 && g->pd == 1 && g->ph == 1 && g->pw == 1 && rn_mma_enabled())
    return launch_conv3_mma_fwd(*g, src, w, dst, stats, st);
  if (!dgrad && src_is_f32 && add == nullptr && rn_is_stem(*g) && rn_mma_enabled()) {
    const long long nt = (long long)g->N * g->Do * g->Ho * ((g->Wo + 31) / 32);
    if (nt <= 0x7fffffffLL) {
      rn_stem_mma_fwd_kernel<<<(unsigned)(nt < 148 * 4 ? nt : 148 * 4), THREADS, 0, st>>>(*g, (const float*)src, w, (__half*)dst, stats);
      return (int)cudaGetLastError();
    }
  }
  const bool k333 = g->kd == 3 && g->kh == 3 && g->kw == 3 && g->sd == 1 && g->sh == 1 && g->sw == 1 && g->pd == 1 && g->ph == 1 &&
                    g->pw == 1 && !src_is_f32 && rn_mma_enabled();
  if (k333 && !dgrad && g->Cin == 8 && g->Cout == 8) return launch_conv3_k8_mma<1, false>(*g, src, w, dst, add, stats, st);
  if (k333 && dgrad && g->Cout == 8 && g->Cin == 8) return launch_conv3_k8_mma<1, true>(*g, src, w, dst, add, nullptr, st);
  if (k333 && g->Cin == 16 && g->Cout == 16) {
    if (dgrad) return launch_conv3_k16_mma<true>(*g, src, w, dst, add, nullptr, st);
    if (add == nullptr) return launch_conv3_k16_mma<false>(*g, src, w, dst, nullptr, stats, st);
  }
  if (k333 && dgrad && g->Cout == 8 && g->Cin == 64 && add == nullptr) return launch_conv3_k8_mma<8, true>(*g, src, w, dst, nullptr, nullptr, st);
  if (dgrad) return dispatch_conv<true>(*g, src_is_f32, src, w, dst, add, stats, st);
  return dispatch_conv<false>(*g, src_is_f32, src, w, dst, add, stats, st);
}

static bool rn_is_l1_block(const RnConvGeom& g) {
  return g.Cin == 64 && g.Cout == 8 && g.kd == 3 && g.kh == 3 && g.kw == 3 && g.sd == 1 && g.sh == 1 && g.sw == 1 && g.pd == 1 &&
         g.ph == 1 && g.pw == 1;
}

// BasicBlock.conv1 (64 -> 8, 3x3x3) and the block's 1x1x1 stride-1 down-sample convolution on the same input in ONE launch;
// returns -9 when the geometry is not that pair (the caller then issues two mmnn_rn_conv calls).
int mmnn_rn_conv_fwd_ds(const RnConvGeom* g, const void* x, const float* w, const float* w_ds, void* y, void* y_ds, double* stats,
                        double* stats_ds, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!rn_is_l1_block(*g) || !rn_mma_enabled()) return -9;
  ProfScope ps(PC_RN_FPROP, st);
  return launch_conv3_mma_fwd(*g, x, w, y, stats, st, w_ds, y_ds, stats_ds);
}

// dx = dgrad(conv1; dy) + dgrad(down-sample; dy_ds) of the same pair in ONE launch (-9: not that pair).
int mmnn_rn_conv_dgrad_ds(const RnConvGeom* g, const void* dy, const float* w, const void* dy_ds, const float* w_ds, void* dx,
                          void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!rn_is_l1_block(*g) || !rn_mma_enabled()) return -9;
  ProfScope ps(PC_RN_DGRAD, st);
  return launch_conv3_k8_mma<8, true>(*g, dy, w, dx, nullptr, nullptr, st, dy_ds, w_ds);
}

int mmnn_rn_conv_wgrad(const RnConvGeom* g, int x_is_f32, const void* x, const void* dy, float* dw, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(PC_RN_WGRAD, st);
  if (g->Cout % 8 != 0) return -2;
  const int items = g->kd * g->kh * g->kw * g->Cin * (g->Cout / 8);
  const int per = (items + THREADS - 1) / THREADS;
  if (x_is_f32 && rn_is_stem(*g) && rn_mma_enabled()) {
    const long long nt = (long long)g->N * g->Do * g->Ho * ((g->Wo + 31) / 32);
    if (nt <= 0x7fffffffLL) {
      rn_stem_mma_wgrad_kernel<<<(unsigned)(nt < 148 * 4 ? nt : 148 * 4), THREADS, 0, st>>>(*g, (const float*)x, (const uint16_t*)dy, dw);
      return (int)cudaGetLastError();
    }
  }
  if (x_is_f32) {
    if (g->Cin != 1) return -3;
    if (per <= 2) return launch_wgrad<float, 1, 2>(*g, x, dy, dw, st);
    if (per <= 4) return launch_wgrad<float, 1, 4>(*g, x, dy, dw, st);
    return -3;
  }
  if (rn_mma_enabled() && (g->Cout == 8 || g->Cout == 16)) {
    int rc = -8;
    if (g->Cin == 8) rc = g->Cout == 8 ? dispatch_wgrad_mma<8, 1>(*g, x, dy, dw, st) : dispatch_wgrad_mma<8, 2>(*g, x, dy, dw, st);
    else if (g->Cin == 16) rc = g->Cout == 8 ? dispatch_wgrad_mma<16, 1>(*g, x, dy, dw, st) : dispatch_wgrad_mma<16, 2>(*g, x, dy, dw, st);
    else if (g->Cin == 64 && g->Cout == 8) rc = dispatch_wgrad_mma<64, 1>(*g, x, dy, dw, st);
    if (rc != -8) return rc;
  }
  if (g->Cin == 8) return dispatch_wgrad_h<8>(*g, per, x, dy, dw, st);
  if (g->Cin == 16) return dispatch_wgrad_h<16>(*g, per, x, dy, dw, st);
  if (g->Cin == 64) return dispatch_wgrad_h<64>(*g, per, x, dy, dw, st);
  return -4;
}

int mmnn_rn_bn_coeffs(const double* stats, double count, const float* gamma, const float* beta, float* rmean, float* rvar,
                      long long* nbt, float eps, float momentum, int training, int C, float* coef, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  // reject before the launch: the kernel's single 64-thread block would otherwise update the running statistics of the
  // first 64 channels and num_batches_tracked before the caller learns the call failed
  if (C < 1 || C > 64) return -2;
  ProfScope ps(PC_RN_ELTWISE, st);
  rn_bn_coeffs_kernel<<<1, 64, 0, st>>>(stats, count, gamma, beta, rmean, rvar, nbt, eps, momentum, training, C, coef);
  return (int)cudaGetLastError();
}

int mmnn_rn_bn_act(const void* raw, const float* coef, int res_mode, const void* res, const float* coef2, void* y,
                   long long elems, int C, int relu, float drop_p, unsigned long long seed, const unsigned char* mask,
                   void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (elems % 8 != 0 || (C != 8 && C != 16 && C != 64)) return -2;
  ProfScope ps(PC_RN_ELTWISE, st);
  const long long n8 = elems / 8;
  const unsigned grid = elt_grid(n8);
  if (res_mode == 0)
    rn_bn_act_kernel<0><<<grid, THREADS, 0, st>>>((const uint4*)raw, coef, nullptr, nullptr, (uint4*)y, n8, C, relu, drop_p, seed, mask);
  else if (res_mode == 1)
    rn_bn_act_kernel<1><<<grid, THREADS, 0, st>>>((const uint4*)raw, coef, (const uint4*)res, nullptr, (uint4*)y, n8, C, relu, drop_p, seed, mask);
  else
    rn_bn_act_kernel<2><<<grid, THREADS, 0, st>>>((const uint4*)raw, coef, (const uint4*)res, coef2, (uint4*)y, n8, C, relu, drop_p, seed, mask);
  return (int)cudaGetLastError();
}

int mmnn_rn_act_bwd_reduce(const void* dy, const void* y, float post_scale, const void* raw, const float* coef,
                           const void* raw2, const float* coef2, double* sums, long long elems, int C, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (elems % 8 != 0 || (C != 8 && C != 16 && C != 64)) return -2;
  ProfScope ps(PC_RN_ELTWISE, st);
  const long long n8 = elems / 8;
  const unsigned grid = elt_grid(n8);
  if (raw2 != nullptr)
    rn_act_bwd_reduce_kernel<true><<<grid, THREADS, 0, st>>>((const uint4*)dy, (const uint4*)y, post_scale, (const uint4*)raw, coef, (const uint4*)raw2, coef2, sums, n8, C);
  else
    rn_act_bwd_reduce_kernel<false><<<grid, THREADS, 0, st>>>((const uint4*)dy, (const uint4*)y, post_scale, (const uint4*)raw, coef, nullptr, nullptr, sums, n8, C);
  return (int)cudaGetLastError();
}

int mmnn_rn_bn_bwd_apply(const void* dy, const void* y, float post_scale, const void* raw, const float* coef, const void* raw2,
                         const float* coef2, const double* sums, double inv_count, int eval_mode, void* draw, void* draw2,
                         void* dz, float* dgamma, float* dbeta, float* dgamma2, float* dbeta2, long long elems, int C,
                         void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (elems % 8 != 0 || (C != 8 && C != 16 && C != 64)) return -2;
  ProfScope ps(PC_RN_ELTWISE, st);
  const long long n8 = elems / 8;
  const unsigned grid = elt_grid(n8);
  if (raw2 != nullptr)
    rn_bn_bwd_apply_kernel<true><<<grid, THREADS, 0, st>>>((const uint4*)dy, (const uint4*)y, post_scale, (const uint4*)raw, coef, (const uint4*)raw2, coef2, sums, inv_count, eval_mode, (uint4*)draw, (uint4*)draw2, (uint4*)dz, dgamma, dbeta, dgamma2, dbeta2, n8, C);
  else
    rn_bn_bwd_apply_kernel<false><<<grid, THREADS, 0, st>>>((const uint4*)dy, (const uint4*)y, post_scale, (const uint4*)raw, coef, nullptr, nullptr, sums, inv_count, eval_mode, (uint4*)draw, nullptr, (uint4*)dz, dgamma, dbeta, nullptr, nullptr, n8, C);
  return (int)cudaGetLastError();
}

int mmnn_rn_head_fwd(const void* y, int B, int V, int C, const float* W, const float* bias, int K, float* pooled, float* out,
                     void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (C > 64 || 128 % C != 0 || K > 64) return -2;
  ProfScope ps(PC_RN_HEAD, st);
  rn_head_fwd_kernel<<<B, 128, 0, st>>>((const __half*)y, V, C, W, bias, K, pooled, out);
  return (int)cudaGetLastError();
}

int mmnn_rn_head_bwd(const float* dout, const float* out, const float* pooled, const float* W, int B, int V, int C, int K,
                     void* dy, float* dW, float* db, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (C > 64 || 128 % C != 0 || K > 64) return -2;
  ProfScope ps(PC_RN_HEAD, st);
  rn_head_bwd_kernel<<<B, 128, 0, st>>>(dout, out, pooled, W, V, C, K, (__nv_bfloat16*)dy, dW, db);
  return (int)cudaGetLastError();
}

}  // extern "C"
