// b200seg — multi-class segmentation on fp32 NCHW logits [N, K, H, W] (2 <= K <= 8, the head kernel's limit) and
// integer label maps [N, H, W] (uint8 or int64):
//   softmax cross-entropy (nn.CrossEntropyLoss(weight, ignore_index) semantics) + soft Dice over the foreground classes,
//   per-sample / per-class confusion counts of argmax vs label, and the argmax label map.
// The K logits of a pixel sit H*W apart: consecutive threads take consecutive pixels (four per thread, one float4 per
// class, when H*W % 4 == 0), and max -> log-sum-exp -> softmax stay in registers.  One reduction pass (fp64 block
// partials, atomics or the deterministic rows of DetBuf) yields every sum the loss, its gradient and the training IoU
// need; the gradient is one elementwise pass.  Layout of the sums: include/b200seg.h (B2_CE_*).
// argmax takes the LOWEST index among equal maxima (torch.argmax); labels outside [0, K) that are not ignore_index are
// counted, not trusted: the loss becomes NaN (torch raises a device-side assert there) and such pixels, like ignored
// ones, contribute to no sum, count or gradient.
#include "common.cuh"

namespace b2 {

constexpr int kMcThreads = 256;

// pixels p0 .. p0 + VEC - 1 (same sample: VEC divides H*W): logits v[j][c] and labels y[j]
template <int K, int VEC, typename L>
__device__ __forceinline__ void mc_load(const float* __restrict__ z, const L* __restrict__ lab, long long hw, long long p0,
                                        float (&v)[VEC][K], long long (&y)[VEC]) {
  const long long n = p0 / hw, s = p0 - n * hw;
  const float* zp = z + n * K * hw + s;
  if constexpr (VEC == 4) {
#pragma unroll
    for (int c = 0; c < K; ++c) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(zp + c * hw));
      v[0][c] = q.x;
      v[1][c] = q.y;
      v[2][c] = q.z;
      v[3][c] = q.w;
    }
    if constexpr (sizeof(L) == 1) {
      const uchar4 u = __ldg(reinterpret_cast<const uchar4*>(lab + p0));
      y[0] = u.x;
      y[1] = u.y;
      y[2] = u.z;
      y[3] = u.w;
    } else {
      const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(lab + p0));
      const longlong2 b = __ldg(reinterpret_cast<const longlong2*>(lab + p0 + 2));
      y[0] = a.x;
      y[1] = a.y;
      y[2] = b.x;
      y[3] = b.y;
    }
  } else {
#pragma unroll
    for (int c = 0; c < K; ++c) v[0][c] = __ldg(zp + c * hw);
    y[0] = (long long)__ldg(lab + p0);
  }
}

// max and the first index attaining it (torch.argmax), softmax numerators e[c] = exp(v[c] - max) and their sum
template <int K>
__device__ __forceinline__ void mc_softmax(const float (&v)[K], float& m, int& am, float (&e)[K], float& s) {
  m = v[0];
  am = 0;
#pragma unroll
  for (int c = 1; c < K; ++c) {
    if (v[c] > m) {
      m = v[c];
      am = c;
    }
  }
  s = 0.f;
#pragma unroll
  for (int c = 0; c < K; ++c) {
    e[c] = expf(v[c] - m);
    s += e[c];
  }
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int K, int VEC, typename L>
__global__ void __launch_bounds__(kMcThreads) ce_loss_fwd_kernel(const float* __restrict__ z, const L* __restrict__ lab,
                                                                 long long npix, long long hw,
                                                                 const float* __restrict__ wt, long long ignore,
                                                                 double* __restrict__ sums, DetBuf det) {
  constexpr int NS = B2_CE_NSUMS(K);
  float a[NS];
#pragma unroll
  for (int k = 0; k < NS; ++k) a[k] = 0.f;
  const long long groups = npix / VEC;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups;
       g += (long long)gridDim.x * blockDim.x) {
    float v[VEC][K];
    long long y[VEC];
    mc_load<K, VEC, L>(z, lab, hw, g * VEC, v, y);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      if (y[j] == ignore) continue;
      if (y[j] < 0 || y[j] >= K) {
        a[B2_CE_INVALID(K)] += 1.f;
        continue;
      }
      const int yc = (int)y[j];
      float m, e[K], s;
      int am;
      mc_softmax<K>(v[j], m, am, e, s);
      float zy = v[j][0];
#pragma unroll
      for (int c = 1; c < K; ++c) zy = c == yc ? v[j][c] : zy;
      const float wy = wt != nullptr ? __ldg(wt + yc) : 1.f;
      a[B2_CE_LOSS] += wy * ((m - zy) + logf(s));        // lse - z_y, without cancellation in lse
      a[B2_CE_WSUM] += wy;
      const float rs = 1.f / s;
#pragma unroll
      for (int c = 0; c < K; ++c) {
        const float p = e[c] * rs;
        const bool t = c == yc, pr = c == am;
        a[B2_CE_PT(K) + c] += t ? p : 0.f;
        a[B2_CE_P(K) + c] += p;
        a[B2_CE_T(K) + c] += t ? 1.f : 0.f;
        a[B2_CE_INTER(K) + c] += (t && pr) ? 1.f : 0.f;
        a[B2_CE_UNION(K) + c] += (t || pr) ? 1.f : 0.f;
      }
    }
  }
  __shared__ double sh[NS][kMcThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < NS; ++k) {
    const double d = warp_sum_f64((double)a[k]);
    if (lane == 0) sh[k][warp] = d;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < NS; k += blockDim.x) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[k][w];
    red_out(sums, det, k, s);
  }
}

__global__ void ce_loss_finalize_kernel(const double* __restrict__ sums, int K, float w_ce, float w_dice, float smooth,
                                        float* __restrict__ loss) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double valid = 0.0;
  for (int c = 0; c < K; ++c) valid += sums[B2_CE_T(K) + c];
  if (sums[B2_CE_INVALID(K)] != 0.0 || valid == 0.0) {
    *loss = __int_as_float(0x7fc00000);       // NaN: a label outside [0, K), or every pixel ignored
    return;
  }
  double l = 0.0;
  if (w_ce != 0.f) l += (double)w_ce * sums[B2_CE_LOSS] / sums[B2_CE_WSUM];
  if (w_dice != 0.f) {
    double dice = 0.0;
    for (int c = 1; c < K; ++c)
      dice += (2.0 * sums[B2_CE_PT(K) + c] + smooth) / (sums[B2_CE_P(K) + c] + sums[B2_CE_T(K) + c] + smooth);
    l += (double)w_dice * (1.0 - dice / (K - 1));
  }
  *loss = (float)l;
}

// dz_j = g * [w_ce w[y] / sum w * (p_j - [j = y]) + p_j (d_j - sum_c p_c d_c)],
// d_c = -w_dice / (K - 1) * (2 [y = c] den_c - num_c) / den_c^2 for c >= 1, d_0 = 0; zero on ignored / invalid pixels
template <int K, int VEC, typename L>
__global__ void __launch_bounds__(kMcThreads) ce_loss_bwd_kernel(const float* __restrict__ z, const L* __restrict__ lab,
                                                                 long long npix, long long hw,
                                                                 const float* __restrict__ wt, long long ignore,
                                                                 const double* __restrict__ sums, float w_ce,
                                                                 float w_dice, float smooth,
                                                                 const float* __restrict__ grad_out,
                                                                 float* __restrict__ dz) {
  const float go = grad_out != nullptr ? __ldg(grad_out) : 1.f;
  const float kce = w_ce != 0.f ? (float)((double)w_ce / sums[B2_CE_WSUM]) : 0.f;
  float dA[K], dB[K];               // d_c = dA[c] [y = c] + dB[c]
  dA[0] = dB[0] = 0.f;
#pragma unroll
  for (int c = 1; c < K; ++c) {
    if (w_dice != 0.f) {
      const double num = 2.0 * sums[B2_CE_PT(K) + c] + smooth;
      const double den = sums[B2_CE_P(K) + c] + sums[B2_CE_T(K) + c] + smooth;
      const double f = (double)w_dice / (K - 1);
      dA[c] = (float)(-2.0 * f / den);
      dB[c] = (float)(f * num / (den * den));
    } else {
      dA[c] = dB[c] = 0.f;
    }
  }
  const long long groups = npix / VEC;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups;
       g += (long long)gridDim.x * blockDim.x) {
    float v[VEC][K];
    long long y[VEC];
    const long long p0 = g * VEC;
    mc_load<K, VEC, L>(z, lab, hw, p0, v, y);
    float o[VEC][K];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const bool ok = y[j] != ignore && y[j] >= 0 && y[j] < K;
      const int yc = ok ? (int)y[j] : -1;
      float m, e[K], s;
      int am;
      mc_softmax<K>(v[j], m, am, e, s);
      const float rs = 1.f / s;
      const float cy = ok ? go * kce * (wt != nullptr ? __ldg(wt + yc) : 1.f) : 0.f;
      const float gd = ok ? go : 0.f;
      float p[K], d[K], pd = 0.f;
#pragma unroll
      for (int c = 0; c < K; ++c) {
        p[c] = e[c] * rs;
        d[c] = (c == yc ? dA[c] : 0.f) + dB[c];
        pd += p[c] * d[c];
      }
#pragma unroll
      for (int c = 0; c < K; ++c) o[j][c] = cy * (p[c] - (c == yc ? 1.f : 0.f)) + gd * p[c] * (d[c] - pd);
    }
    const long long n = p0 / hw, s0 = p0 - n * hw;
    float* dp = dz + n * K * hw + s0;
#pragma unroll
    for (int c = 0; c < K; ++c) {
      if constexpr (VEC == 4) {
        *reinterpret_cast<float4*>(dp + c * hw) = make_float4(o[0][c], o[1][c], o[2][c], o[3][c]);
      } else {
        dp[c * hw] = o[0][c];
      }
    }
  }
}

// counts[n][c] = {TP, #pred, #target} of class c in sample n, pred = argmax; ignored / invalid pixels excluded
template <int K, int VEC, typename L>
__global__ void __launch_bounds__(kMcThreads) seg_counts_mc_kernel(const float* __restrict__ z, const L* __restrict__ lab,
                                                                   long long hw, long long ignore,
                                                                   unsigned long long* __restrict__ counts) {
  const int n = blockIdx.y;
  unsigned cnt[3 * K];
#pragma unroll
  for (int k = 0; k < 3 * K; ++k) cnt[k] = 0u;
  const long long groups = hw / VEC;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups;
       g += (long long)gridDim.x * blockDim.x) {
    float v[VEC][K];
    long long y[VEC];
    mc_load<K, VEC, L>(z, lab, hw, (long long)n * hw + g * VEC, v, y);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      if (y[j] == ignore || y[j] < 0 || y[j] >= K) continue;
      float m = v[j][0];
      int am = 0;
#pragma unroll
      for (int c = 1; c < K; ++c) {
        if (v[j][c] > m) {
          m = v[j][c];
          am = c;
        }
      }
#pragma unroll
      for (int c = 0; c < K; ++c) {
        const bool t = c == (int)y[j], pr = c == am;
        cnt[3 * c + 0] += (t && pr) ? 1u : 0u;
        cnt[3 * c + 1] += pr ? 1u : 0u;
        cnt[3 * c + 2] += t ? 1u : 0u;
      }
    }
  }
  __shared__ unsigned sh[3 * K][kMcThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 3 * K; ++k) {
    const unsigned s = __reduce_add_sync(0xffffffffu, cnt[k]);
    if (lane == 0) sh[k][warp] = s;
  }
  __syncthreads();
  if (threadIdx.x < 3 * K) {
    unsigned long long s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[threadIdx.x][w];
    if (s) atomicAdd(&counts[(long long)n * 3 * K + threadIdx.x], s);
  }
}

// label map = argmax over the K logits (first maximum), uint8
template <int K, int VEC>
__global__ void __launch_bounds__(kMcThreads) logits_to_labels_kernel(const float* __restrict__ z, long long npix,
                                                                      long long hw, uint8_t* __restrict__ out) {
  const long long groups = npix / VEC;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups;
       g += (long long)gridDim.x * blockDim.x) {
    const long long p0 = g * VEC, n = p0 / hw, s = p0 - n * hw;
    const float* zp = z + n * K * hw + s;
    if constexpr (VEC == 4) {
      float4 m = __ldg(reinterpret_cast<const float4*>(zp));
      uchar4 am = make_uchar4(0, 0, 0, 0);
#pragma unroll
      for (int c = 1; c < K; ++c) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(zp + c * hw));
        if (q.x > m.x) { m.x = q.x; am.x = (uint8_t)c; }
        if (q.y > m.y) { m.y = q.y; am.y = (uint8_t)c; }
        if (q.z > m.z) { m.z = q.z; am.z = (uint8_t)c; }
        if (q.w > m.w) { m.w = q.w; am.w = (uint8_t)c; }
      }
      *reinterpret_cast<uchar4*>(out + p0) = am;
    } else {
      float m = __ldg(zp);
      uint8_t am = 0;
#pragma unroll
      for (int c = 1; c < K; ++c) {
        const float q = __ldg(zp + c * hw);
        if (q > m) { m = q; am = (uint8_t)c; }
      }
      out[p0] = am;
    }
  }
}

static int mc_grid(long long groups) {
  long long g = (groups + kMcThreads - 1) / kMcThreads;
  const long long cap = (long long)num_sms() * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

static bool aligned(const void* p, int bytes) { return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0; }

// four pixels per thread when the planes allow it: H*W % 4 == 0 and every pointer aligned for the vector access
static int mc_vec(long long hw, const float* z, const void* lab, int label_bytes, const void* out, int out_bytes) {
  if (hw % 4 != 0 || !aligned(z, 16)) return 1;
  if (lab != nullptr && !aligned(lab, 4 * label_bytes)) return 1;
  if (out != nullptr && !aligned(out, 4 * out_bytes)) return 1;
  return 4;
}

// F<K, VEC, L>::run(args...) for the runtime (k, vec, label bytes)
template <template <int, int, typename> class F, typename... A>
static int mc_dispatch(int k, int vec, int label_bytes, A&&... args) {
#define B2_MC_CASE(KK)                                                                             \
  case KK:                                                                                         \
    if (label_bytes == 1)                                                                          \
      return vec == 4 ? F<KK, 4, uint8_t>::run(args...) : F<KK, 1, uint8_t>::run(args...);        \
    return vec == 4 ? F<KK, 4, int64_t>::run(args...) : F<KK, 1, int64_t>::run(args...);
  switch (k) {
    B2_MC_CASE(2)
    B2_MC_CASE(3)
    B2_MC_CASE(4)
    B2_MC_CASE(5)
    B2_MC_CASE(6)
    B2_MC_CASE(7)
    B2_MC_CASE(8)
  }
#undef B2_MC_CASE
  B2_REQUIRE(false, B2_ERR_SHAPE, "class count %d outside [2, 8]", k);
}

template <int K, int VEC, typename L>
struct CeFwd {
  static int run(const float* z, const void* lab, long long npix, long long hw, const float* wt, long long ignore,
                 double* sums, cudaStream_t st) {
    const int grid = mc_grid(npix / VEC);
    constexpr int NS = B2_CE_NSUMS(K);
    DetBuf det;
    int rc = det_begin(&det, grid, NS, st);
    if (rc) return rc;
    ce_loss_fwd_kernel<K, VEC, L><<<grid, kMcThreads, 0, st>>>(z, static_cast<const L*>(lab), npix, hw, wt, ignore,
                                                               sums, det);
    B2_LAUNCH_CHECK();
    if (det.partial) return det_finish(det.partial, grid, NS, NS, sums, st);
    return B2_OK;
  }
};

template <int K, int VEC, typename L>
struct CeBwd {
  static int run(const float* z, const void* lab, long long npix, long long hw, const float* wt, long long ignore,
                 const double* sums, float w_ce, float w_dice, float smooth, const float* grad_out, float* dz,
                 cudaStream_t st) {
    ce_loss_bwd_kernel<K, VEC, L><<<mc_grid(npix / VEC), kMcThreads, 0, st>>>(
        z, static_cast<const L*>(lab), npix, hw, wt, ignore, sums, w_ce, w_dice, smooth, grad_out, dz);
    B2_LAUNCH_CHECK();
    return B2_OK;
  }
};

template <int K, int VEC, typename L>
struct CountsMc {
  static int run(const float* z, const void* lab, int n, long long hw, long long ignore, uint64_t* counts,
                 cudaStream_t st) {
    long long gx = (hw / VEC + kMcThreads * 4 - 1) / (kMcThreads * 4);
    const long long cap = ((long long)num_sms() * 8 + n - 1) / n;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    seg_counts_mc_kernel<K, VEC, L><<<dim3((unsigned)gx, (unsigned)n), kMcThreads, 0, st>>>(
        z, static_cast<const L*>(lab), hw, ignore, reinterpret_cast<unsigned long long*>(counts));
    B2_LAUNCH_CHECK();
    return B2_OK;
  }
};

template <int K, int VEC, typename L>
struct ToLabels {
  static int run(const float* z, long long npix, long long hw, uint8_t* out, cudaStream_t st) {
    logits_to_labels_kernel<K, VEC><<<mc_grid(npix / VEC), kMcThreads, 0, st>>>(z, npix, hw, out);
    B2_LAUNCH_CHECK();
    return B2_OK;
  }
};

static int mc_check(int32_t n, int32_t k, int64_t hw, int32_t label_bytes) {
  B2_REQUIRE(n > 0 && hw > 0 && k >= 2 && k <= 8, B2_ERR_SHAPE, "bad multi-class extent n=%d k=%d hw=%lld", n, k,
             (long long)hw);
  B2_REQUIRE(label_bytes == 1 || label_bytes == 8, B2_ERR_SHAPE, "labels must be uint8 or int64 (got %d bytes)",
             label_bytes);
  return B2_OK;
}

}  // namespace b2

using namespace b2;

extern "C" int b2_ce_loss_fwd(const float* z, const void* labels, int32_t label_bytes, int32_t n, int32_t k,
                              int64_t hw, const float* weight, int64_t ignore_index, double* sums,
                              b2_stream_t stream) {
  int rc = mc_check(n, k, hw, label_bytes);
  if (rc) return rc;
  const long long npix = (long long)n * hw;
  return mc_dispatch<CeFwd>(k, mc_vec(hw, z, labels, label_bytes, nullptr, 0), label_bytes, z, labels, npix,
                            (long long)hw, weight, (long long)ignore_index, sums, (cudaStream_t)stream);
}

extern "C" int b2_ce_loss_finalize(const double* sums, int32_t k, float w_ce, float w_dice, float smooth, float* loss,
                                   b2_stream_t stream) {
  B2_REQUIRE(k >= 2 && k <= 8, B2_ERR_SHAPE, "class count %d outside [2, 8]", k);
  ce_loss_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(sums, k, w_ce, w_dice, smooth, loss);
  B2_LAUNCH_CHECK();
  return B2_OK;
}

extern "C" int b2_ce_loss_bwd(const float* z, const void* labels, int32_t label_bytes, int32_t n, int32_t k,
                              int64_t hw, const float* weight, int64_t ignore_index, const double* sums, float w_ce,
                              float w_dice, float smooth, const float* grad_out, float* dz, b2_stream_t stream) {
  int rc = mc_check(n, k, hw, label_bytes);
  if (rc) return rc;
  const long long npix = (long long)n * hw;
  return mc_dispatch<CeBwd>(k, mc_vec(hw, z, labels, label_bytes, dz, 4), label_bytes, z, labels, npix,
                            (long long)hw, weight, (long long)ignore_index, sums, w_ce, w_dice, smooth, grad_out, dz,
                            (cudaStream_t)stream);
}

extern "C" int b2_seg_counts_mc(const float* z, const void* labels, int32_t label_bytes, int32_t n, int32_t k,
                                int64_t hw, int64_t ignore_index, uint64_t* counts, b2_stream_t stream) {
  int rc = mc_check(n, k, hw, label_bytes);
  if (rc) return rc;
  B2_REQUIRE(n <= 65535, B2_ERR_SHAPE, "seg_counts_mc: %d samples (at most 65535)", n);
  B2_CHECK_CUDA(cudaMemsetAsync(counts, 0, (size_t)n * k * 3 * sizeof(uint64_t), (cudaStream_t)stream));
  return mc_dispatch<CountsMc>(k, mc_vec(hw, z, labels, label_bytes, nullptr, 0), label_bytes, z, labels, (int)n,
                               (long long)hw, (long long)ignore_index, counts, (cudaStream_t)stream);
}

extern "C" int b2_logits_to_labels(const float* z, int32_t n, int32_t k, int64_t hw, uint8_t* labels,
                                   b2_stream_t stream) {
  int rc = mc_check(n, k, hw, 1);
  if (rc) return rc;
  const long long npix = (long long)n * hw;
  return mc_dispatch<ToLabels>(k, mc_vec(hw, z, nullptr, 1, labels, 1), 1, z, npix, (long long)hw, labels,
                               (cudaStream_t)stream);
}
