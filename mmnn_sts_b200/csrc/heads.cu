// Small latency-bound kernels after the trunk: image feature head (ReLU -> global average pool -> Linear -> Dropout),
// clinical MLP + fusion heads, Cox partial-likelihood loss, bootstrap concordance index, batched GradCAM maps.
// References: /root/reference/models/densenet.py:234-247, /root/reference/models/mlp.py:19-51,
// /root/reference/models/multimodal.py:51-80, /root/reference/losses/losses.py:6-9 (pycox CoxPHLoss),
// /root/reference/main.py:106-123 (lifelines concordance_index), /root/reference/utils/utils.py:253-344 (GradCAM).
#include <algorithm>
#include <climits>
#include <mutex>

#include "common.cuh"
#include "prof.h"

using namespace mmnn;

#define LAUNCH_RET()                          \
  do {                                        \
    cudaError_t e_ = cudaGetLastError();      \
    if (e_ != cudaSuccess) return (int)e_;    \
  } while (0)

namespace mmnn_heads {

// ---------------------------------------------------------------------------------------------- feature head
// y: fp32 [B][V][C] (norm5 output, NDHWC);  pooled[b][c] = mean_v relu(y);  out[b][f] = (W[f]·pooled[b] + bias[f]) * mask[b][f]
__global__ void __launch_bounds__(256) gap_linear_fwd_kernel(const float* __restrict__ y, int V, int C, const float* __restrict__ W,
                                                             const float* __restrict__ bias, const float* __restrict__ mask,
                                                             int F, float* __restrict__ pooled, float* __restrict__ out) {
  extern __shared__ float sp[];  // [C]
  const int b = blockIdx.x;
  const float* yb = y + (size_t)b * V * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc = 0.f;
    for (int v = 0; v < V; ++v) acc += fmaxf(yb[(size_t)v * C + c], 0.f);
    acc /= (float)V;
    sp[c] = acc;
    pooled[(size_t)b * C + c] = acc;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int f = warp; f < F; f += blockDim.x >> 5) {
    float acc = 0.f;
    for (int c = lane; c < C; c += 32) acc = fmaf(W[(size_t)f * C + c], sp[c], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      float r = acc + bias[f];
      if (mask != nullptr) r *= mask[(size_t)b * F + f];
      out[(size_t)b * F + f] = r;
    }
  }
}

// dy[b][v][c] = relu'(y) * (1/V) * sum_f g[b][f] W[f][c],   g = dout * mask
__global__ void __launch_bounds__(256) gap_linear_bwd_dy_kernel(const float* __restrict__ y, int V, int C, const float* __restrict__ W,
                                                                const float* __restrict__ dout, const float* __restrict__ mask,
                                                                int F, float* __restrict__ dy) {
  extern __shared__ float sg[];  // [F]
  const int b = blockIdx.x;
  for (int f = threadIdx.x; f < F; f += blockDim.x)
    sg[f] = dout[(size_t)b * F + f] * (mask != nullptr ? mask[(size_t)b * F + f] : 1.f);
  __syncthreads();
  const float* yb = y + (size_t)b * V * C;
  float* dyb = dy + (size_t)b * V * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc = 0.f;
    for (int f = 0; f < F; ++f) acc = fmaf(sg[f], W[(size_t)f * C + c], acc);
    acc /= (float)V;
    for (int v = 0; v < V; ++v) dyb[(size_t)v * C + c] = yb[(size_t)v * C + c] > 0.f ? acc : 0.f;
  }
}

// dW[f][c] = sum_b g[b][f] pooled[b][c];  db[f] = sum_b g[b][f]
__global__ void __launch_bounds__(256) gap_linear_bwd_w_kernel(const float* __restrict__ pooled, const float* __restrict__ dout,
                                                               const float* __restrict__ mask, int B, int C, int F,
                                                               float* __restrict__ dW, float* __restrict__ db) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < F * C) {
    const int f = idx / C, c = idx - f * C;
    float acc = 0.f;
    for (int b = 0; b < B; ++b) {
      const float g = dout[(size_t)b * F + f] * (mask != nullptr ? mask[(size_t)b * F + f] : 1.f);
      acc = fmaf(g, pooled[(size_t)b * C + c], acc);
    }
    dW[idx] = acc;
  }
  if (idx < F) {
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += dout[(size_t)b * F + idx] * (mask != nullptr ? mask[(size_t)b * F + idx] : 1.f);
    db[idx] = acc;
  }
}


// ---------------------------------------------------------------------------------------------- clinical MLP + heads
// One CTA runs the whole clinical branch (6 x Linear -> BatchNorm1d -> ReLU/Dropout1d) and the fusion heads.
// Dropout1d on a 2-D [B,F] input drops whole SAMPLES (reference quirk Q3): mask[i][b] is 0 or 1/(1-p) >= 0, so
// relu(m*x) == m*relu(x) and the two layer orders of /root/reference/models/mlp.py:21-50 coincide.
constexpr int MLP_LAYERS = 6;
struct MlpArgs {
  const float* W[MLP_LAYERS];
  const float* b[MLP_LAYERS];
  const float* gamma[MLP_LAYERS];
  const float* beta[MLP_LAYERS];
  float* rmean[MLP_LAYERS];
  float* rvar[MLP_LAYERS];
  long long* nbt[MLP_LAYERS];
  const float* Wo; const float* bo;   // output_head            [C][2F]
  const float* Wi; const float* bi;   // image_output_head      [C][F]
  const float* Wc; const float* bc;   // clinical_output_head   [C][F]
  int width[MLP_LAYERS + 1];          // width[0] = clinical inputs, width[6] = features F
  int B, C, blend, training;
  const float* x;        // [B][width[0]]
  const float* img_f;    // [B][F]
  const float* mask;     // [6][B] or null
  float* z;              // saved pre-BN  [sum width[1..6]][B]-ish: layer i at zoff[i], row-major [B][width[i+1]]
  float* a;              // saved post-activation, same layout
  float* stat;           // saved mean/rstd: [6][2][32]
  float* preds;          // [H][B][C]
  // backward
  const float* dpreds;   // [H][B][C]
  float* dW[MLP_LAYERS]; float* db[MLP_LAYERS]; float* dgamma[MLP_LAYERS]; float* dbeta[MLP_LAYERS];
  float* dWo; float* dbo; float* dWi; float* dbi; float* dWc; float* dbc;
  float* d_img_f;        // [B][F]
  float* scratch;        // [2][B][32] ping-pong activation gradients
};

__device__ int mlp_off(const MlpArgs& p, int layer) {
  int o = 0;
  for (int i = 0; i < layer; ++i) o += p.B * p.width[i + 1];
  return o;
}

__global__ void __launch_bounds__(256) mlp_heads_fwd_kernel(const __grid_constant__ MlpArgs p) {
  __shared__ float s_mean[32], s_rstd[32];
  const int tid = threadIdx.x, B = p.B;
  const float* in = p.x;
  for (int i = 0; i < MLP_LAYERS; ++i) {
    const int K = p.width[i], O = p.width[i + 1];
    float* z = p.z + mlp_off(p, i);
    float* a = p.a + mlp_off(p, i);
    for (int idx = tid; idx < B * O; idx += blockDim.x) {
      const int b = idx / O, o = idx - b * O;
      float acc = p.b[i][o];
      for (int k = 0; k < K; ++k) acc = fmaf(in[b * K + k], p.W[i][o * K + k], acc);
      z[idx] = acc;
    }
    __syncthreads();
    for (int o = tid; o < O; o += blockDim.x) {
      float mean, var;
      if (p.training) {
        float s = 0.f;
        for (int b = 0; b < B; ++b) s += z[b * O + o];
        mean = s / (float)B;
        float q = 0.f;
        for (int b = 0; b < B; ++b) { const float d = z[b * O + o] - mean; q = fmaf(d, d, q); }
        var = q / (float)B;
        const float unbiased = B > 1 ? q / (float)(B - 1) : var;
        p.rmean[i][o] = 0.9f * p.rmean[i][o] + 0.1f * mean;
        p.rvar[i][o] = 0.9f * p.rvar[i][o] + 0.1f * unbiased;
        if (o == 0) *p.nbt[i] += 1;
      } else {
        mean = p.rmean[i][o]; var = p.rvar[i][o];
      }
      const float rstd = 1.0f / sqrtf(var + 1e-5f);
      s_mean[o] = mean; s_rstd[o] = rstd;
      p.stat[(i * 2 + 0) * 32 + o] = mean; p.stat[(i * 2 + 1) * 32 + o] = rstd;
    }
    __syncthreads();
    for (int idx = tid; idx < B * O; idx += blockDim.x) {
      const int b = idx / O, o = idx - b * O;
      float v = fmaxf(fmaf((z[idx] - s_mean[o]) * s_rstd[o], p.gamma[i][o], p.beta[i][o]), 0.f);
      if (p.mask != nullptr) v *= p.mask[i * B + b];
      a[idx] = v;
    }
    __syncthreads();
    in = a;
  }
  const int F = p.width[MLP_LAYERS], C = p.C;
  const float* cf = p.a + mlp_off(p, MLP_LAYERS - 1);
  for (int idx = tid; idx < B * C; idx += blockDim.x) {
    const int b = idx / C, c = idx - b * C;
    float o = p.bo[c];
    for (int k = 0; k < F; ++k) o = fmaf(p.img_f[b * F + k], p.Wo[c * 2 * F + k], o);
    for (int k = 0; k < F; ++k) o = fmaf(cf[b * F + k], p.Wo[c * 2 * F + F + k], o);
    p.preds[idx] = o;
    if (p.blend) {
      float ip = p.bi[c], cp = p.bc[c];
      for (int k = 0; k < F; ++k) { ip = fmaf(p.img_f[b * F + k], p.Wi[c * F + k], ip); cp = fmaf(cf[b * F + k], p.Wc[c * F + k], cp); }
      p.preds[B * C + idx] = ip;
      p.preds[2 * B * C + idx] = cp;
    }
  }
}

__global__ void __launch_bounds__(256) mlp_heads_bwd_kernel(const __grid_constant__ MlpArgs p) {
  __shared__ float s_c1[32], s_c2[32];
  const int tid = threadIdx.x, B = p.B, C = p.C, F = p.width[MLP_LAYERS];
  const float* cf = p.a + mlp_off(p, MLP_LAYERS - 1);
  const float* dout = p.dpreds;
  const float* dip = p.dpreds + B * C;
  const float* dcp = p.dpreds + 2 * B * C;
  // heads: parameter gradients
  for (int idx = tid; idx < C * 2 * F; idx += blockDim.x) {
    const int c = idx / (2 * F), k = idx - c * 2 * F;
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc = fmaf(dout[b * C + c], k < F ? p.img_f[b * F + k] : cf[b * F + k - F], acc);
    p.dWo[idx] = acc;
  }
  for (int idx = tid; idx < C * F; idx += blockDim.x) {
    const int c = idx / F, k = idx - c * F;
    float ai = 0.f, ac = 0.f;
    if (p.blend)
      for (int b = 0; b < B; ++b) { ai = fmaf(dip[b * C + c], p.img_f[b * F + k], ai); ac = fmaf(dcp[b * C + c], cf[b * F + k], ac); }
    p.dWi[idx] = ai; p.dWc[idx] = ac;
  }
  for (int c = tid; c < C; c += blockDim.x) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (int b = 0; b < B; ++b) { s0 += dout[b * C + c]; if (p.blend) { s1 += dip[b * C + c]; s2 += dcp[b * C + c]; } }
    p.dbo[c] = s0; p.dbi[c] = s1; p.dbc[c] = s2;
  }
  // heads: feature gradients
  float* da = p.scratch;            // gradient w.r.t. the current layer's output activation [B][width]
  float* dnext = p.scratch + B * 32;
  for (int idx = tid; idx < B * F; idx += blockDim.x) {
    const int b = idx / F, k = idx - b * F;
    float gi = 0.f, gc = 0.f;
    for (int c = 0; c < C; ++c) {
      gi = fmaf(dout[b * C + c], p.Wo[c * 2 * F + k], gi);
      gc = fmaf(dout[b * C + c], p.Wo[c * 2 * F + F + k], gc);
      if (p.blend) { gi = fmaf(dip[b * C + c], p.Wi[c * F + k], gi); gc = fmaf(dcp[b * C + c], p.Wc[c * F + k], gc); }
    }
    p.d_img_f[idx] = gi;
    da[idx] = gc;
  }
  __syncthreads();
  for (int i = MLP_LAYERS - 1; i >= 0; --i) {
    const int K = p.width[i], O = p.width[i + 1];
    const float* z = p.z + mlp_off(p, i);
    const float* in = i == 0 ? p.x : p.a + mlp_off(p, i - 1);
    const float* mean = p.stat + (i * 2 + 0) * 32;
    const float* rstd = p.stat + (i * 2 + 1) * 32;
    // dr = da * mask * relu'(pre);  per-channel sums for the BN backward
    for (int o = tid; o < O; o += blockDim.x) {
      float s1 = 0.f, s2 = 0.f;
      for (int b = 0; b < B; ++b) {
        const float xh = (z[b * O + o] - mean[o]) * rstd[o];
        const float pre = fmaf(xh, p.gamma[i][o], p.beta[i][o]);
        float dr = pre > 0.f ? da[b * O + o] : 0.f;
        if (p.mask != nullptr) dr *= p.mask[i * B + b];
        s1 += dr; s2 = fmaf(dr, xh, s2);
      }
      p.dgamma[i][o] = s2; p.dbeta[i][o] = s1;
      s_c1[o] = p.training ? s1 / (float)B : 0.f;
      s_c2[o] = p.training ? s2 / (float)B : 0.f;
    }
    __syncthreads();
    // dz (stored in place of da)
    for (int idx = tid; idx < B * O; idx += blockDim.x) {
      const int b = idx / O, o = idx - b * O;
      const float xh = (z[idx] - mean[o]) * rstd[o];
      const float pre = fmaf(xh, p.gamma[i][o], p.beta[i][o]);
      float dr = pre > 0.f ? da[idx] : 0.f;
      if (p.mask != nullptr) dr *= p.mask[i * B + b];
      da[idx] = p.gamma[i][o] * rstd[o] * (dr - s_c1[o] - xh * s_c2[o]);
    }
    __syncthreads();
    for (int idx = tid; idx < O * K; idx += blockDim.x) {
      const int o = idx / K, k = idx - o * K;
      float acc = 0.f;
      for (int b = 0; b < B; ++b) acc = fmaf(da[b * O + o], in[b * K + k], acc);
      p.dW[i][idx] = acc;
    }
    for (int o = tid; o < O; o += blockDim.x) {
      float acc = 0.f;
      for (int b = 0; b < B; ++b) acc += da[b * O + o];
      p.db[i][o] = acc;
    }
    if (i > 0) {
      for (int idx = tid; idx < B * K; idx += blockDim.x) {
        const int b = idx / K, k = idx - b * K;
        float acc = 0.f;
        for (int o = 0; o < O; ++o) acc = fmaf(da[b * O + o], p.W[i][o * K + k], acc);
        dnext[idx] = acc;
      }
    }
    __syncthreads();
    float* t = da; da = dnext; dnext = t;
  }
}

// ---------------------------------------------------------------------------------------------- Cox partial likelihood
// pycox cox_ph_loss (restated in oracle/cox.py) for S independent segments in one launch (segment = (head, class)):
//   order rows by sort key DEscending (stable: ties keep original order), gamma = max h,
//   S_i = cumsum_i exp(h - gamma) + eps,  loss = -sum_i w_i (h_i - log S_i - gamma) / sum_i w_i
//   dloss/dh_j = -(w_j - p_j * sum_{i>=j} w_i / S_i) / sum w     (gamma treated as a constant)
// One CTA per segment; block-wide scans are warp-shuffle scans with a per-warp carry.
constexpr int COX_THREADS = 1024;

__device__ __forceinline__ float block_scan_inclusive(float v, float* warp_sums, float& carry_inout) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += n;
  }
  if (lane == 31) warp_sums[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float w = warp_sums[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float n = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += n;
    }
    warp_sums[lane] = w;
  }
  __syncthreads();
  const float prefix = (warp > 0 ? warp_sums[warp - 1] : 0.f) + carry_inout;
  const float total = warp_sums[31];
  __syncthreads();
  carry_inout += total;
  return v + prefix;
}

struct CoxArgs {
  const float* h; long long h_seg_stride, h_stride;       // log-hazards: h[seg*h_seg_stride + i*h_stride]
  const double* key; long long key_seg_stride, key_stride; // sort key  (pycox "durations" slot)
  const double* w; long long w_seg_stride, w_stride;       // row weight (pycox "events" slot)
  const int* perm;       // optional [S][N] precomputed descending order, or null (then N <= COX_SORT_MAX, sorted here)
  int N, S;
  float eps;
  float* loss;           // [S]
  float* grad;           // [S][N] dloss/dh
};
constexpr int COX_SORT_MAX = 4096;

__global__ void __launch_bounds__(COX_THREADS) cox_nll_kernel(const __grid_constant__ CoxArgs p) {
  extern __shared__ unsigned char cox_smem[];
  int* idx = reinterpret_cast<int*>(cox_smem);                 // [Npad]
  float* pv = reinterpret_cast<float*>(idx + p.N + 32);        // [N]   exp(h-gamma), later w/S
  double* sk = reinterpret_cast<double*>(pv + p.N + 32);       // [Npow2] sort keys (only when sorting here)
  __shared__ float warp_sums[32];
  __shared__ float s_red[32];
  const int seg = blockIdx.x, tid = threadIdx.x, N = p.N;
  const float* h = p.h + seg * p.h_seg_stride;
  const double* key = p.key + seg * p.key_seg_stride;
  const double* w = p.w + seg * p.w_seg_stride;
  if (p.perm != nullptr) {
    for (int i = tid; i < N; i += COX_THREADS) idx[i] = p.perm[(size_t)seg * N + i];
  } else {
    // bitonic sort of (key desc, index asc) on a power-of-two padded array
    int P = 1;
    while (P < N) P <<= 1;
    int* sidx = reinterpret_cast<int*>(sk + P);
    for (int i = tid; i < P; i += COX_THREADS) {
      sk[i] = i < N ? key[i * p.key_stride] : -INFINITY;
      sidx[i] = i < N ? i : 0x7fffffff;
    }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < P; i += COX_THREADS) {
          const int l = i ^ j;
          if (l > i) {
            const double a = sk[i], b = sk[l];
            const int ia = sidx[i], ib = sidx[l];
            // "a before b" in the final (descending, stable) order
            const bool a_first = (a > b) || (a == b && ia < ib);
            const bool up = (i & k) == 0;
            if (up ? !a_first : a_first) { sk[i] = b; sk[l] = a; sidx[i] = ib; sidx[l] = ia; }
          }
        }
        __syncthreads();
      }
    }
    for (int i = tid; i < N; i += COX_THREADS) idx[i] = sidx[i];
  }
  __syncthreads();
  // gamma = max h
  float m = -INFINITY;
  for (int i = tid; i < N; i += COX_THREADS) m = fmaxf(m, h[i * p.h_stride]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((tid & 31) == 0) s_red[tid >> 5] = m;
  __syncthreads();
  m = s_red[0];
  for (int i = 1; i < COX_THREADS / 32; ++i) m = fmaxf(m, s_red[i]);
  const float gamma = m;
  __syncthreads();
  // forward scan: S_i, accumulate numerator and total weight
  float carry = 0.f, num = 0.f, wsum = 0.f;
  for (int base = 0; base < N; base += COX_THREADS) {
    const int i = base + tid;
    float pe = 0.f, hi = 0.f, wi = 0.f;
    if (i < N) { const int j = idx[i]; hi = h[j * p.h_stride]; wi = (float)w[j * p.w_stride]; pe = expf(hi - gamma); }
    const float S = block_scan_inclusive(pe, warp_sums, carry) + p.eps;
    if (i < N) {
      num += (hi - (logf(S) + gamma)) * wi;
      wsum += wi;
      pv[i] = wi / S;          // for the reverse scan
      p.grad[(size_t)seg * N + idx[i]] = pe;   // stash p_j in the output slot of row j
    }
  }
  // block reduce num, wsum
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { num += __shfl_xor_sync(0xffffffffu, num, o); wsum += __shfl_xor_sync(0xffffffffu, wsum, o); }
  __shared__ float s_num[32], s_w[32];
  if ((tid & 31) == 0) { s_num[tid >> 5] = num; s_w[tid >> 5] = wsum; }
  __syncthreads();
  float tn = 0.f, tw = 0.f;
  for (int i = 0; i < COX_THREADS / 32; ++i) { tn += s_num[i]; tw += s_w[i]; }
  if (tid == 0) p.loss[seg] = -tn / tw;
  __syncthreads();
  // reverse scan of w/S: tail_j = sum_{i>=j} w_i/S_i ; walk chunks from the end
  carry = 0.f;
  for (int base = 0; base < N; base += COX_THREADS) {
    const int r = base + tid;            // position from the end
    const int i = N - 1 - r;
    const float v = (r < N) ? pv[i] : 0.f;
    const float tail = block_scan_inclusive(v, warp_sums, carry);
    if (r < N) {
      const int j = idx[i];
      const float pe = p.grad[(size_t)seg * N + j];
      const float wi = (float)w[j * p.w_stride];
      p.grad[(size_t)seg * N + j] = -(wi - pe * tail) / tw;
    }
  }
}

// ---------------------------------------------------------------------------------------------- bootstrap C-index
// lifelines concordance_index restated (oracle/cindex.py) for R bootstrap resamples of one patient set, exact in
// integers.  Patients are pre-sorted by (time asc, deaths before censored); a resample is a multiplicity vector
// w = bincount(indices).  One warp sweeps one resample with a Fenwick tree over score ranks held in shared memory:
// lanes own one tree level each, so a prefix query / an insertion is one shared-memory access per lane + a warp sum.
struct CindexArgs {
  const int* rank;        // [N] score rank (0-based, dense) of the sorted patients
  const int* is_death;    // [N]
  const int* group_end;   // [N] index one past the end of the equal-time group containing i
  const int* orig;        // [N] original patient index of sorted position i
  const int* resample;    // [R][N] indices into the ORIGINAL patient order
  int N, R, nranks;
  long long* counts;      // [R][3] correct, tied, pairs
};

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(32) cindex_bootstrap_kernel(const __grid_constant__ CindexArgs p) {
  extern __shared__ int ci_smem[];
  int* tree = ci_smem;               // [nranks + 1] Fenwick tree of inserted death multiplicities
  int* mult = ci_smem + p.nranks + 1;  // [N] multiplicity of each ORIGINAL patient in this resample
  const int r = blockIdx.x, lane = threadIdx.x;
  for (int i = lane; i <= p.nranks; i += 32) tree[i] = 0;
  for (int i = lane; i < p.N; i += 32) mult[i] = 0;
  __syncwarp();
  for (int i = lane; i < p.N; i += 32) atomicAdd(&mult[p.resample[(size_t)r * p.N + i]], 1);
  __syncwarp();
  long long correct = 0, tied = 0, pairs = 0;
  long long pool = 0;
  // prefix(q) = number of inserted with rank < q : sum over tree nodes q, q - lowbit(q), ...  (one node per lane)
  auto prefix = [&](int q) -> long long {
    int node = q;
    for (int l = 0; l < lane && node > 0; ++l) node -= node & (-node);
    long long v = (node > 0) ? tree[node] : 0;
    // lanes beyond the chain length hold node == 0
    return warp_sum_ll(v);
  };
  int g0 = 0;
  while (g0 < p.N) {
    const int g1 = p.group_end[g0];
    // deaths of this time group come first: count against the pool BEFORE inserting them
    int gd = g0;
    while (gd < g1 && p.is_death[gd]) ++gd;
    for (int i = g0; i < gd; ++i) {
      const int wgt = mult[p.orig[i]];
      if (wgt == 0) continue;
      const int rk = p.rank[i];
      const long long lt = prefix(rk), le = prefix(rk + 1);
      pairs += (long long)wgt * pool; correct += (long long)wgt * lt; tied += (long long)wgt * (le - lt);
    }
    for (int i = g0; i < gd; ++i) {
      const int wgt = mult[p.orig[i]];
      if (wgt == 0) continue;
      // insert at rank rk: nodes rk+1, then += lowbit ... (one node per lane)
      int node = p.rank[i] + 1;
      for (int l = 0; l < lane && node <= p.nranks; ++l) node += node & (-node);
      if (node <= p.nranks) tree[node] += wgt;
      __syncwarp();
      pool += wgt;
    }
    for (int i = gd; i < g1; ++i) {
      const int wgt = mult[p.orig[i]];
      if (wgt == 0) continue;
      const int rk = p.rank[i];
      const long long lt = prefix(rk), le = prefix(rk + 1);
      pairs += (long long)wgt * pool; correct += (long long)wgt * lt; tied += (long long)wgt * (le - lt);
    }
    g0 = g1;
  }
  if (lane == 0) {
    p.counts[(size_t)r * 3 + 0] = correct; p.counts[(size_t)r * 3 + 1] = tied; p.counts[(size_t)r * 3 + 2] = pairs;
  }
}

// ---------------------------------------------------------------------------------------------- GradCAM attention maps
// Batched replacement of MultiModalGradCAM.attentionMaps (/root/reference/utils/utils.py:293-344) for an eval-mode model.
// The hooked layer is the last conv2 of the last dense block: its 32 output channels are channels [coff, coff + 32) of
// the block buffer, and they reach the outputs only through norm5 (eval: a fixed affine map) -> ReLU -> global average
// pool -> feature_layer -> output_head.  So the pooled gradient GradCAM reads has a closed form (no trunk backward):
//   alpha[b][c][k] = (sum_f Wo[c][f] Wf[f][k']) * gamma5[k'] / sqrt(rvar5[k'] + eps) * count_v(y[b][v][k'] > 0) / V^2,
// k' = coff + k.  Then the reference's map arithmetic: the activations are re-weighted IN PLACE class after class (class c
// sees alpha[0] * .. * alpha[c]), cam = channel mean, cam -= min, cam /= max (a constant cam gives NaN, as there), and
// F.interpolate(mode='trilinear', align_corners=False) to the volume size.  The cam stays 3-D: unlike the reference's
// .squeeze(), a trunk dimension of size 1 is fine.
// One launch: CTA (chunk, b) rebuilds sample b's C normalised cams in shared memory (V*32 activations + V*32 signs of y),
// then streams its range of the [C][X][Y] output rows, Z contiguous floats each.  Every reduction runs in a fixed order.
struct GradcamArgs {
  const bf16* act;       // last dense block buffer, storage dtype (fp16 / bf16 per kActF16), [B*V][Ctot]
  const float* y;        // trunk output (norm5 output) fp32 NDHWC [B*V][Ctot]
  const float* gamma5;   // norm5.weight        [Ctot]
  const float* rvar5;    // norm5.running_var   [Ctot]
  const float* Wf;       // feature_layer.weight [F][Ctot]
  const float* Wo;       // output_head.weight   [C][2F] (image features first)
  float* maps;           // [B][C][X][Y][Z]
  float eps;
  int Ctot, coff;
  int B, C, F;
  int d, h, w;           // trunk dims
  int X, Y, Z;           // map dims
};
constexpr int GC_CH = 32;          // growth rate: channels of the hooked conv
constexpr int GC_THREADS = 256;
constexpr size_t GC_SMEM_MAX = 200 * 1024;

__device__ __forceinline__ float gc_act(const bf16* p) {
  if constexpr (kActF16) return __half2float(*reinterpret_cast<const __half*>(p));
  else return __bfloat162float(*p);
}

// min / max that return NaN when either operand is NaN (torch.min / torch.max semantics; fminf / fmaxf skip NaN)
__device__ __forceinline__ float gc_nanmin(float a, float b) { return (a != a || a < b) ? a : b; }
__device__ __forceinline__ float gc_nanmax(float a, float b) { return (a != a || a > b) ? a : b; }

// PyTorch's trilinear source index (align_corners=False, size given): src = max(scale (dst + 0.5) - 0.5, 0)
struct GcLerp { int i0, i1; float l0, l1; };
__device__ __forceinline__ GcLerp gc_lerp(int dst, float scale, int in) {
  const float src = fmaxf(scale * ((float)dst + 0.5f) - 0.5f, 0.f);
  GcLerp r;
  r.i0 = (int)src;
  r.i1 = r.i0 + (r.i0 < in - 1 ? 1 : 0);
  r.l1 = src - (float)r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}

template <bool VEC>
__global__ void __launch_bounds__(GC_THREADS) gradcam_maps_kernel(const __grid_constant__ GradcamArgs p, int rows_per_cta) {
  extern __shared__ float gc_smem[];
  const int C = p.C, V = p.d * p.h * p.w, b = blockIdx.y, tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nthr = blockDim.x * blockDim.y, lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
  float* s_cam = gc_smem;                        // [C][V]
  float* s_alpha = s_cam + (size_t)C * V;        // [C][32]
  float* s_line = s_alpha + C * GC_CH;           // [blockDim.y][w]
  int* s_cnt = reinterpret_cast<int*>(s_line + blockDim.y * p.w);   // [32]
  const size_t row0 = (size_t)b * V;

  // 1. per-channel positive counts of y (exact integers), the head weights A[c][k] * norm5 scale
  if (tid < GC_CH) s_cnt[tid] = 0;
  __syncthreads();
  {
    int cnt = 0;                                 // nthr % 32 == 0: this thread always sees channel k = lane
    for (int i = tid; i < V * GC_CH; i += nthr) cnt += p.y[(row0 + i / GC_CH) * p.Ctot + p.coff + lane] > 0.f ? 1 : 0;
    if (cnt) atomicAdd(&s_cnt[lane], cnt);
  }
  for (int i = tid; i < C * GC_CH; i += nthr) {
    const int c = i / GC_CH, k = i - c * GC_CH, kk = p.coff + k;
    float a = 0.f;
    for (int f = 0; f < p.F; ++f) a = fmaf(p.Wo[(size_t)c * 2 * p.F + f], p.Wf[(size_t)f * p.Ctot + kk], a);
    s_alpha[i] = a * (p.gamma5[kk] / sqrtf(p.rvar5[kk] + p.eps));
  }
  __syncthreads();
  const float v2 = (float)V * (float)V;
  for (int i = tid; i < C * GC_CH; i += nthr) s_alpha[i] = s_alpha[i] * ((float)s_cnt[i % GC_CH] / v2);
  __syncthreads();

  // 2. cams: weighted[k] *= alpha[c][k] class after class (the reference's in-place quirk), cam[c][v] = mean_k weighted[k]
  for (int v = tid; v < V; v += nthr) {
    const bf16* a = p.act + (row0 + v) * p.Ctot + p.coff;
    float wk[GC_CH];
#pragma unroll
    for (int k = 0; k < GC_CH; ++k) wk[k] = gc_act(a + k);
    for (int c = 0; c < C; ++c) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < GC_CH; ++k) { wk[k] *= s_alpha[c * GC_CH + k]; s += wk[k]; }
      s_cam[(size_t)c * V + v] = s / (float)GC_CH;
    }
  }
  __syncthreads();

  // 3. cam -= min; cam /= max (one warp per class, fixed reduction order).  NaN propagates as in torch.min / torch.max: a
  // cam holding a NaN (a non-finite activation) normalises to all-NaN, like the reference's.
  for (int c = warp; c < C; c += nwarps) {
    float* cam = s_cam + (size_t)c * V;
    float mn = INFINITY, mx = -INFINITY;
    for (int v = lane; v < V; v += 32) { mn = gc_nanmin(mn, cam[v]); mx = gc_nanmax(mx, cam[v]); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = gc_nanmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = gc_nanmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    const float range = mx - mn;                 // == max(cam - min): x -> fl(x - mn) is monotonic
    for (int v = lane; v < V; v += 32) cam[v] = (cam[v] - mn) / range;
  }
  __syncthreads();

  // 4. trilinear up-sampling of rows [r0, r1) of the flattened [C][X][Y] rows.  Row r is owned by the threads with
  // threadIdx.y == r % blockDim.y (one warp holds whole rows): they first blend the row's line over (x, y) --
  // line[j] = lerp_x lerp_y cam[c][.][.][j], j < w -- then write Z outputs, each a lerp of two line entries.
  const int XY = p.X * p.Y, total = C * XY;
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(total, r0 + rows_per_cta);
  const float sx = (float)p.d / (float)p.X, sy = (float)p.h / (float)p.Y, sz = (float)p.w / (float)p.Z;
  float* line = s_line + threadIdx.y * p.w;
  float* out_b = p.maps + (size_t)b * total * p.Z;
  const int nz = VEC ? p.Z / 4 : p.Z;
  for (int base = r0; base < r1; base += blockDim.y) {
    const int r = base + threadIdx.y;
    const bool active = r < r1;
    if (active) {
      const int c = r / XY, xy = r - c * XY, x = xy / p.Y, yy = xy - x * p.Y;
      const GcLerp lx = gc_lerp(x, sx, p.d), ly = gc_lerp(yy, sy, p.h);
      const float* cc = s_cam + (size_t)c * V;
      const float* p00 = cc + ((size_t)lx.i0 * p.h + ly.i0) * p.w;
      const float* p01 = cc + ((size_t)lx.i0 * p.h + ly.i1) * p.w;
      const float* p10 = cc + ((size_t)lx.i1 * p.h + ly.i0) * p.w;
      const float* p11 = cc + ((size_t)lx.i1 * p.h + ly.i1) * p.w;
      for (int j = threadIdx.x; j < p.w; j += blockDim.x)
        line[j] = lx.l0 * (ly.l0 * p00[j] + ly.l1 * p01[j]) + lx.l1 * (ly.l0 * p10[j] + ly.l1 * p11[j]);
    }
    __syncwarp();
    if (active) {
      float* orow = out_b + (size_t)r * p.Z;
      for (int q = threadIdx.x; q < nz; q += blockDim.x) {
        if constexpr (VEC) {
          float o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const GcLerp lz = gc_lerp(4 * q + j, sz, p.w);
            o[j] = lz.l0 * line[lz.i0] + lz.l1 * line[lz.i1];
          }
          __stcs(reinterpret_cast<float4*>(orow) + q, make_float4(o[0], o[1], o[2], o[3]));
        } else {
          const GcLerp lz = gc_lerp(q, sz, p.w);
          __stcs(orow + q, lz.l0 * line[lz.i0] + lz.l1 * line[lz.i1]);
        }
      }
    }
    __syncwarp();
  }
}

}  // namespace mmnn_heads
using namespace mmnn_heads;

// ------------------------------------------------------------------------------------------------- BCE with logits
// nn.BCEWithLogitsLoss(pos_weight) as the reference's classification path builds it (/root/reference/main.py:148-153):
//   l = (1 - y) x + (1 + (pw - 1) y) * (log1p(exp(-|x|)) + max(-x, 0))          (torch's stable form), elementwise,
//   dl/dx = (1 - y) - (1 + (pw - 1) y) * (1 - sigmoid(x)),
// for all stacked heads in one launch; plus the F1 counters of main.py:226-229 (sigmoid(x) > thr vs. label) per class
// for the first `count_rows` rows (the multimodal head).  x, y: [rows][C] (y broadcast over heads by the caller's view).
__global__ void __launch_bounds__(256) bce_logits_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ pw,
                                                         long long n, int C, long long y_rows_elems, float* __restrict__ loss, float* __restrict__ grad,
                                                         float thr, long long count_elems, int* __restrict__ counts /*[3][C] tp fp fn or null*/) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % C);
    const float xv = x[i], yv = y[i % y_rows_elems];
    const float w = 1.f + ((pw != nullptr ? pw[c] : 1.f) - 1.f) * yv;
    const float sp = log1pf(expf(-fabsf(xv))) + fmaxf(-xv, 0.f);
    loss[i] = (1.f - yv) * xv + w * sp;
    const float sig = 1.f / (1.f + expf(-xv));
    grad[i] = (1.f - yv) - w * (1.f - sig);
    if (counts != nullptr && i < count_elems) {
      const bool pred = sig > thr, pos = yv == 1.f, neg = yv == 0.f;
      if (pred && pos) atomicAdd(counts + c, 1);
      if (pred && neg) atomicAdd(counts + C + c, 1);
      if (!pred && pos) atomicAdd(counts + 2 * C + c, 1);
    }
  }
}

extern "C" {

int mmnn_gap_linear_fwd(const float* y, int B, int V, int C, const float* W, const float* bias, const float* mask, int F,
                        float* pooled, float* out, void* stream) {
  mmnn::ProfScope ps_(mmnn::PC_HEADS, (cudaStream_t)stream, 1);
  gap_linear_fwd_kernel<<<B, 256, C * sizeof(float), (cudaStream_t)stream>>>(y, V, C, W, bias, mask, F, pooled, out);
  LAUNCH_RET();
  return 0;
}

int mmnn_gap_linear_bwd(const float* y, const float* pooled, int B, int V, int C, const float* W, const float* dout,
                        const float* mask, int F, float* dy, float* dW, float* db, void* stream) {
  mmnn::ProfScope ps_(mmnn::PC_HEADS, (cudaStream_t)stream, 2);
  gap_linear_bwd_dy_kernel<<<B, 256, F * sizeof(float), (cudaStream_t)stream>>>(y, V, C, W, dout, mask, F, dy);
  LAUNCH_RET();
  gap_linear_bwd_w_kernel<<<(F * C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(pooled, dout, mask, B, C, F, dW, db);
  LAUNCH_RET();
  return 0;
}


int mmnn_mlp_heads(const MlpArgs* args, int backward, void* stream) {
  if (args->B < 1 || args->B > 1024) return -2;
  for (int i = 1; i <= MLP_LAYERS; ++i)
    if (args->width[i] > 32) return -3;
  mmnn::ProfScope ps_(mmnn::PC_HEADS, (cudaStream_t)stream);
  if (backward) mlp_heads_bwd_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(*args);
  else mlp_heads_fwd_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(*args);
  LAUNCH_RET();
  return 0;
}
int mmnn_sizeof_mlp_args() { return (int)sizeof(MlpArgs); }

int mmnn_cox_nll(const CoxArgs* a, void* stream) {
  if (a->N < 1) return -2;
  size_t smem = (size_t)(a->N + 32) * 8;
  if (a->perm == nullptr) {
    if (a->N > COX_SORT_MAX) return -3;
    int P = 1;
    while (P < a->N) P <<= 1;
    smem += (size_t)P * 12 + 16;
  }
  if (smem > 220 * 1024) return -4;
  cudaError_t e = cudaFuncSetAttribute(cox_nll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  mmnn::ProfScope ps_(mmnn::PC_HEADS, (cudaStream_t)stream, 1);
  cox_nll_kernel<<<a->S, COX_THREADS, smem, (cudaStream_t)stream>>>(*a);
  LAUNCH_RET();
  return 0;
}
int mmnn_sizeof_cox_args() { return (int)sizeof(CoxArgs); }

}  // extern "C"

namespace {
struct GcLaunch { bool vec; dim3 grid, block; size_t smem; int rows_per_cta; };
constexpr int GC_MAX_DEVICES = 64;
struct GcVariantCache { size_t smem = 0, smem_attr = 0; int per_sm = 0; };   // last occupancy query; largest smem attribute set
struct GcDeviceCache { int sms = 0; GcVariantCache variant[2]; };
GcDeviceCache g_gc_cache[GC_MAX_DEVICES];
std::mutex g_gc_cache_mutex;

// Launch shape of mmnn_gradcam_maps; 0 or the error code it returns.
int gradcam_launch_config(const GradcamArgs* a, GcLaunch* L) {
  if (a->B < 1 || a->B > 65535 || a->C < 1 || a->F < 1 || a->d < 1 || a->h < 1 || a->w < 1 || a->X < 1 || a->Y < 1 ||
      a->Z < 1 || a->coff < 0 || a->coff + GC_CH > a->Ctot)
    return -2;
  const long long V = (long long)a->d * a->h * a->w, rows = (long long)a->C * a->X * a->Y;
  if (rows > INT_MAX / 2 || V * GC_CH > INT_MAX / 2) return -2;
  L->vec = a->Z % 4 == 0 && ((uintptr_t)a->maps & 15) == 0;
  const int nz = L->vec ? a->Z / 4 : a->Z;
  int bx = 1;
  while (bx < nz && bx < 32) bx <<= 1;           // threads along Z: a power of two <= 32, so a warp holds whole rows
  L->block = dim3(bx, GC_THREADS / bx);
  L->smem = ((size_t)a->C * V + (size_t)a->C * GC_CH + (size_t)L->block.y * a->w + GC_CH) * sizeof(float);
  if (L->smem > GC_SMEM_MAX) return -3;
  // >= 2 full waves: CTAs resident per SM x SMs x 2, split evenly over the samples.  The device queries (SM count, the
  // dynamic shared memory attribute, occupancy) run once per (device, variant, shared memory size), not per batch.
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  if (dev < 0 || dev >= GC_MAX_DEVICES) return -2;
  std::lock_guard<std::mutex> lock(g_gc_cache_mutex);
  GcDeviceCache& dc = g_gc_cache[dev];
  if (dc.sms == 0 && (e = cudaDeviceGetAttribute(&dc.sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
  GcVariantCache& vc = dc.variant[L->vec ? 1 : 0];
  if (vc.smem != L->smem) {
    auto kern = L->vec ? gradcam_maps_kernel<true> : gradcam_maps_kernel<false>;
    if (L->smem > vc.smem_attr) {
      if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L->smem)) != cudaSuccess) return (int)e;
      vc.smem_attr = L->smem;
    }
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GC_THREADS, L->smem)) != cudaSuccess) return (int)e;
    vc.per_sm = per_sm > 0 ? per_sm : 1;
    vc.smem = L->smem;
  }
  const int sms = dc.sms, per_sm = vc.per_sm;
  const long long target = 2LL * sms * per_sm;
  const long long chunks = std::min<long long>(rows, (target + a->B - 1) / a->B);
  L->rows_per_cta = (int)((rows + chunks - 1) / chunks);
  L->grid = dim3((unsigned)((rows + L->rows_per_cta - 1) / L->rows_per_cta), (unsigned)a->B);
  return 0;
}
}  // namespace

extern "C" {

// Batched GradCAM maps (MultiModalGradCAM.attentionMaps, /root/reference/utils/utils.py:293-344, for every sample of an
// eval-mode forward at once).  Shared memory: C*V cams + C*32 weights + one line of w floats per row in flight; -3 when
// that exceeds GC_SMEM_MAX, -2 for inconsistent sizes.
int mmnn_gradcam_maps(const GradcamArgs* a, void* stream) {
  GcLaunch L;
  const int rc = gradcam_launch_config(a, &L);
  if (rc != 0) return rc;
  mmnn::ProfScope ps_(mmnn::PC_HEADS, (cudaStream_t)stream, 1);
  if (L.vec) gradcam_maps_kernel<true><<<L.grid, L.block, L.smem, (cudaStream_t)stream>>>(*a, L.rows_per_cta);
  else gradcam_maps_kernel<false><<<L.grid, L.block, L.smem, (cudaStream_t)stream>>>(*a, L.rows_per_cta);
  LAUNCH_RET();
  return 0;
}
// CTAs mmnn_gradcam_maps launches for these arguments (each reads its sample's V x 32 activations and signs of y once):
// the byte count of a bandwidth figure.  Negative: the error code mmnn_gradcam_maps would return.
long long mmnn_gradcam_ctas(const GradcamArgs* a) {
  GcLaunch L;
  const int rc = gradcam_launch_config(a, &L);
  return rc != 0 ? rc : (long long)L.grid.x * L.grid.y;
}
int mmnn_sizeof_gradcam_args() { return (int)sizeof(GradcamArgs); }

int mmnn_cindex_bootstrap(const CindexArgs* a, void* stream) {
  const size_t smem = (size_t)(a->nranks + 1 + a->N) * sizeof(int);
  if (smem > 220 * 1024) return -4;
  cudaError_t e = cudaFuncSetAttribute(cindex_bootstrap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  mmnn::ProfScope ps_(mmnn::PC_HEADS, (cudaStream_t)stream, 1);
  cindex_bootstrap_kernel<<<a->R, 32, smem, (cudaStream_t)stream>>>(*a);
  LAUNCH_RET();
  return 0;
}
int mmnn_sizeof_cindex_args() { return (int)sizeof(CindexArgs); }

// x [n] logits of all stacked heads ([H][N][C] flattened), y [y_elems] targets ([N][C], reused by every head),
// pos_weight [C] or NULL; loss / grad [n] elementwise; counts int32 [3][C] (tp, fp, fn; caller-zeroed) over the first
// count_elems elements, or NULL.
int mmnn_bce_logits(const float* x, const float* y, const float* pos_weight, long long n, int C, long long y_elems, float* loss,
                    float* grad, float threshold, long long count_elems, int* counts, void* stream) {
  if (n <= 0) return 0;
  if (C <= 0 || y_elems <= 0 || y_elems % C != 0) return -2;
  mmnn::ProfScope ps_(mmnn::PC_HEADS, (cudaStream_t)stream, 1);
  long long blocks = (n + 255) / 256;
  bce_logits_kernel<<<(unsigned)(blocks > 1184 ? 1184 : blocks), 256, 0, (cudaStream_t)stream>>>(x, y, pos_weight, n, C, y_elems, loss,
                                                                                                 grad, threshold, count_elems, counts);
  LAUNCH_RET();
  return 0;
}

}  // extern "C"
