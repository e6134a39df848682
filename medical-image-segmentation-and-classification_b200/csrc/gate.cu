// b200seg — attention gate (AttentionUNet.py:29-54, R2AttU_Net.py:61-86):
//     out = x * sigmoid(BN1(psi . relu(BN_g(W_g g) + BN_x(W_x x))))
// The two 1x1 GEMMs (W_g, W_x) run on tcgen05 through b2_conv_fprop with the BN-statistics epilogue; everything
// after them is memory-bound and lives here.  Train-mode BatchNorm puts two grid-wide reductions inside the gate
// (statistics of the psi pre-activation, and of its gradient), hence forward = {psi_fwd, apply_fwd} and
// backward = {apply_bwd, psi_bwd_reduce, psi_bwd_apply}; `a = relu(..)` is recomputed, never stored.
// Rounding points mirror autocast: every BN output, the g1+x1 sum, the psi conv output and sigmoid are bf16.
#include <stdlib.h>

#include "common.cuh"

namespace b2 {

__device__ __forceinline__ void g_unpack8(const uint4& u, float* f) {
  f[0] = bf16lo(u.x); f[1] = bf16hi(u.x); f[2] = bf16lo(u.y); f[3] = bf16hi(u.y);
  f[4] = bf16lo(u.z); f[5] = bf16hi(u.z); f[6] = bf16lo(u.w); f[7] = bf16hi(u.w);
}
__device__ __forceinline__ uint4 g_pack8(const float* f) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]),
                    pack_bf16x2(f[6], f[7]));
}
__device__ __forceinline__ void g_load8(const float* p, bool has, float* f) {
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = has ? __ldg(p + j) : 0.f;
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// block-wide sum of two floats held by arbitrary threads -> dst[0], dst[1] (fp64 atomics, or the block's partial row)
__device__ __forceinline__ void block_sum2_out(float a, float b, double* dst, const DetBuf& det) {
  __shared__ float sh[2][8];
  a = warp_sum(a);
  b = warp_sum(b);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    sh[0][warp] = a;
    sh[1][warp] = b;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float ta = 0.f, tb = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) {
      ta += sh[0][i];
      tb += sh[1][i];
    }
    red_out(dst, det, 0, (double)ta);
    red_out(dst, det, 1, (double)tb);
  }
}

// ---------------------------------------------------------------------------------------------------------
// forward phase B: q = psi_conv(relu(bn_g(g1p) + bn_x(x1p)))  + statistics of q
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gate_psi_fwd_kernel(
    const __nv_bfloat16* __restrict__ g1p, const __nv_bfloat16* __restrict__ x1p, int ld, long long npix, int fint,
    int L, const float* __restrict__ scale_g, const float* __restrict__ shift_g, const float* __restrict__ scale_x,
    const float* __restrict__ shift_x, const float* __restrict__ wpsi, const float* __restrict__ bpsi,
    __nv_bfloat16* __restrict__ q, double* __restrict__ qstats, DetBuf det) {
  pdl_enter();
  const int lig = threadIdx.x % L, grp = threadIdx.x / L, gpb = blockDim.x / L;
  const bool has = lig * 8 < fint;
  float sg[8], hg[8], sx[8], hx[8], wp[8];
  g_load8(scale_g + lig * 8, has, sg);
  g_load8(shift_g + lig * 8, has, hg);
  g_load8(scale_x + lig * 8, has, sx);
  g_load8(shift_x + lig * 8, has, hx);
  g_load8(wpsi + lig * 8, has, wp);
#pragma unroll
  for (int j = 0; j < 8; ++j) wp[j] = bf16_round(wp[j]);
  const float bp = bpsi ? __ldg(bpsi) : 0.f;
  float lsum = 0.f, lsq = 0.f;
  for (long long base = (long long)blockIdx.x * gpb; base < npix; base += (long long)gridDim.x * gpb) {
    const long long p = base + grp;
    const bool live = p < npix;
    float s = 0.f;
    if (has && live) {
      float g[8], x[8];
      g_unpack8(__ldg(reinterpret_cast<const uint4*>(g1p + p * ld + lig * 8)), g);
      g_unpack8(__ldg(reinterpret_cast<const uint4*>(x1p + p * ld + lig * 8)), x);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gb = bf16_round(fmaf(g[j], sg[j], hg[j]));
        const float xb = bf16_round(fmaf(x[j], sx[j], hx[j]));
        const float a = fmaxf(bf16_round(gb + xb), 0.f);
        s = fmaf(a, wp[j], s);
      }
    }
    for (int o = L >> 1; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lig == 0 && live) {
      const __nv_bfloat16 qb = __float2bfloat16_rn(s + bp);
      q[p] = qb;
      const float qf = __bfloat162float(qb);
      lsum += qf;
      lsq += qf * qf;
    }
  }
  block_sum2_out(lsum, lsq, qstats, det);
}

// forward phase C: psi = sigmoid(bn1(q)); out = x * psi      (thread owns an 8-channel group, walks pixels)
__global__ void __launch_bounds__(256) gate_apply_fwd_kernel(const __nv_bfloat16* __restrict__ x, int ldx,
                                                             const __nv_bfloat16* __restrict__ q, long long npix,
                                                             int tpp, int rows, const float* __restrict__ scale1,
                                                             const float* __restrict__ shift1,
                                                             __nv_bfloat16* __restrict__ psi,
                                                             __nv_bfloat16* __restrict__ out, int ldo) {
  pdl_enter();
  const int g = threadIdx.x % tpp, r = threadIdx.x / tpp;
  if (r >= rows) return;
  const float s1 = __ldg(scale1), h1 = __ldg(shift1);
  for (long long p = (long long)blockIdx.x * rows + r; p < npix; p += (long long)gridDim.x * rows) {
    const float qv = __bfloat162float(q[p]);
    const float ps = bf16_round(sigmoidf_(bf16_round(fmaf(qv, s1, h1))));
    float f[8];
    g_unpack8(__ldg(reinterpret_cast<const uint4*>(x + p * ldx + g * 8)), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] *= ps;
    *reinterpret_cast<uint4*>(out + p * ldo + g * 8) = g_pack8(f);
    if (g == 0) psi[p] = __float2bfloat16_rn(ps);
  }
}

// backward phase 1: dx = dout*psi ; dsig = (sum_c dout*x) * psi (1-psi) ; sums1 += (dsig, dsig*qhat)
__global__ void __launch_bounds__(256) gate_apply_bwd_kernel(
    const __nv_bfloat16* __restrict__ dout, int lddout, const __nv_bfloat16* __restrict__ x, int ldx,
    const __nv_bfloat16* __restrict__ psi, const __nv_bfloat16* __restrict__ q, long long npix, int cg, int L,
    const float* __restrict__ mean1, const float* __restrict__ invstd1, __nv_bfloat16* __restrict__ dx, int lddx,
    float* __restrict__ dsig, double* __restrict__ sums1, DetBuf det) {
  pdl_enter();
  const int lig = threadIdx.x % L, grp = threadIdx.x / L, gpb = blockDim.x / L;
  const float mu1 = __ldg(mean1), is1 = __ldg(invstd1);
  float l0 = 0.f, l1 = 0.f;
  const long long stride = (long long)gridDim.x * gpb;
  constexpr int U = 2;                        // pixels in flight per thread (cg <= L: one 8-channel group each)
  for (long long base = (long long)blockIdx.x * gpb; base < npix; base += U * stride) {
    float s[U], ps[U];
    bool live[U];
    if (cg <= L) {
      uint4 dv[U], fv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long p = base + u * stride + grp;
        live[u] = p < npix;
        const bool ld = live[u] && lig < cg;
        const long long pc = live[u] ? p : 0;
        ps[u] = __bfloat162float(psi[pc]);
        dv[u] = ld ? __ldg(reinterpret_cast<const uint4*>(dout + pc * lddout + lig * 8)) : make_uint4(0, 0, 0, 0);
        fv[u] = ld ? __ldg(reinterpret_cast<const uint4*>(x + pc * ldx + lig * 8)) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long p = base + u * stride + grp;
        float d[8], f[8];
        g_unpack8(dv[u], d);
        g_unpack8(fv[u], f);
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc = fmaf(d[j], f[j], acc);
          d[j] *= ps[u];
        }
        s[u] = acc;
        if (live[u] && lig < cg) *reinterpret_cast<uint4*>(dx + p * lddx + lig * 8) = g_pack8(d);
      }
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long p = base + u * stride + grp;
        live[u] = p < npix;
        s[u] = 0.f;
        ps[u] = 0.f;
        if (live[u]) {
          ps[u] = __bfloat162float(psi[p]);
          for (int k = lig; k < cg; k += L) {
            float d[8], f[8];
            g_unpack8(__ldg(reinterpret_cast<const uint4*>(dout + p * lddout + k * 8)), d);
            g_unpack8(__ldg(reinterpret_cast<const uint4*>(x + p * ldx + k * 8)), f);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              s[u] = fmaf(d[j], f[j], s[u]);
              d[j] *= ps[u];
            }
            *reinterpret_cast<uint4*>(dx + p * lddx + k * 8) = g_pack8(d);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float su = s[u];
      for (int o = L >> 1; o > 0; o >>= 1) su += __shfl_xor_sync(0xffffffffu, su, o);
      const long long p = base + u * stride + grp;
      if (lig == 0 && live[u]) {
        const float ds = su * ps[u] * (1.f - ps[u]);
        dsig[p] = ds;
        const float qh = (__bfloat162float(q[p]) - mu1) * is1;
        l0 += ds;
        l1 += ds * qh;
      }
    }
  }
  block_sum2_out(l0, l1, sums1, det);
}

struct GateBwdCoef {
  const float *scale_g, *shift_g, *mean_g, *invstd_g, *gamma_g;
  const float *scale_x, *shift_x, *mean_x, *invstd_x, *gamma_x;
  const float *gamma1, *mean1, *invstd1;
  const float* wpsi;
};

// dq for one pixel from dsig via BN1 backward
__device__ __forceinline__ float gate_dq(float ds, float qv, float g1, float mu1, float is1, int training,
                                         float k0, float k1) {
  const float qh = (qv - mu1) * is1;
  return training ? g1 * is1 * (ds - k0 - qh * k1) : g1 * is1 * ds;
}

// ---------------------------------------------------------------------------------------------------------
// The two psi-backward kernels are templates on V = channels per thread: V = 8 (16-byte accesses) or V = 4 (8-byte
// accesses, half the per-channel register state: <= 80 registers, three blocks per SM and room next to a persistent
// weight-gradient CTA of the side stream).  V = 4 is used whenever F_int / 4 threads per pixel fit a block.
// U = pixels in flight per thread: 4 (two blocks per SM) for F_int <= 128, where it measured 4-9 % faster than 2
// (three blocks per SM); the kernels are as much instruction- as latency-bound (B200SEG_GATE_U forces either).
// ---------------------------------------------------------------------------------------------------------
template <int V> struct GVec;
template <> struct GVec<8> { using T = uint4; };
template <> struct GVec<4> { using T = uint2; };
template <int V> __device__ __forceinline__ void gv_unpack(const typename GVec<V>::T& u, float* f);
template <> __device__ __forceinline__ void gv_unpack<8>(const uint4& u, float* f) { g_unpack8(u, f); }
template <> __device__ __forceinline__ void gv_unpack<4>(const uint2& u, float* f) {
  f[0] = bf16lo(u.x); f[1] = bf16hi(u.x); f[2] = bf16lo(u.y); f[3] = bf16hi(u.y);
}
template <int V> __device__ __forceinline__ typename GVec<V>::T gv_pack(const float* f);
template <> __device__ __forceinline__ uint4 gv_pack<8>(const float* f) { return g_pack8(f); }
template <> __device__ __forceinline__ uint2 gv_pack<4>(const float* f) {
  return make_uint2(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]));
}
template <int V> __device__ __forceinline__ void gv_loadf(const float* p, bool has, float* f) {
#pragma unroll
  for (int j = 0; j < V; ++j) f[j] = has ? __ldg(p + j) : 0.f;
}

// backward phase 2: reductions for BN_g, BN_x and the psi conv
template <int V, int U, int MINB>
__global__ void __launch_bounds__(256, MINB) gate_psi_bwd_reduce_kernel(
    const float* __restrict__ dsig, const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ g1p,
    const __nv_bfloat16* __restrict__ x1p, int ld, long long npix, int fint, int L, GateBwdCoef c,
    const double* __restrict__ sums1, int training, double* __restrict__ sums, float* __restrict__ dwpsi,
    float* __restrict__ dbpsi, int slice, DetBuf det) {
  pdl_enter();
  using VT = typename GVec<V>::T;
  // gridDim.y channel slices of `slice` channels (0: one slice = all of F_int): a block then ends in 5 * slice global
  // atomics instead of 5 * F_int, and gridDim.x (= blocks adding to one address) shrinks by the slice count — the
  // same-address atomics of ~1200 blocks were a fixed 30-90 us per launch, whatever the tensor size.
  const int c_off = slice ? blockIdx.y * slice : 0;
  const int fw = slice ? (fint - c_off < slice ? fint - c_off : slice) : fint;      // channels of this slice
  g1p += c_off;
  x1p += c_off;
  c.scale_g += c_off; c.shift_g += c_off; c.mean_g += c_off; c.invstd_g += c_off;
  c.scale_x += c_off; c.shift_x += c_off; c.mean_x += c_off; c.invstd_x += c_off;
  c.wpsi += c_off;
  extern __shared__ float red[];   // [4][fw] + 1
  for (int i = threadIdx.x; i < 4 * fw + 1; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  const int lig = threadIdx.x % L, grp = threadIdx.x / L, gpb = blockDim.x / L;
  const bool has = lig * V < fw;
  // per-channel constants kept in registers: BN affine (mask recomputation), means (centred sums), psi weights.
  // The xhat sums are accumulated as sum da * (v - mean) and scaled by invstd once per block.
  float sg[V], hg[V], mg[V], sx[V], hx[V], mx[V], wp[V];
  gv_loadf<V>(c.scale_g + lig * V, has, sg);
  gv_loadf<V>(c.shift_g + lig * V, has, hg);
  gv_loadf<V>(c.mean_g + lig * V, has, mg);
  gv_loadf<V>(c.scale_x + lig * V, has, sx);
  gv_loadf<V>(c.shift_x + lig * V, has, hx);
  gv_loadf<V>(c.mean_x + lig * V, has, mx);
  gv_loadf<V>(c.wpsi + lig * V, has, wp);
#pragma unroll
  for (int j = 0; j < V; ++j) wp[j] = bf16_round(wp[j]);
  const float g1 = __ldg(c.gamma1), mu1 = __ldg(c.mean1), is1 = __ldg(c.invstd1);
  const float k0 = (float)(sums1[0] / (double)npix), k1 = (float)(sums1[1] / (double)npix);
  float ab[V], agg[V], agx[V], aw[V], abp = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) ab[j] = agg[j] = agx[j] = aw[j] = 0.f;
  if (has) {
    const long long stride = (long long)gridDim.x * gpb;
    // U pixels in flight per thread (all loads issued before the math)
    for (long long p0 = (long long)blockIdx.x * gpb + grp; p0 < npix; p0 += U * stride) {
      VT gv[U], xv[U];
      float ds[U], qv[U];
      bool ok[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long p = p0 + u * stride;
        ok[u] = p < npix;
        const long long pc = ok[u] ? p : p0;
        gv[u] = __ldg(reinterpret_cast<const VT*>(g1p + pc * ld + lig * V));
        xv[u] = __ldg(reinterpret_cast<const VT*>(x1p + pc * ld + lig * V));
        ds[u] = __ldg(dsig + pc);
        qv[u] = __bfloat162float(q[pc]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float dq = ok[u] ? gate_dq(ds[u], qv[u], g1, mu1, is1, training, k0, k1) : 0.f;
        float g[V], x[V];
        gv_unpack<V>(gv[u], g);
        gv_unpack<V>(xv[u], x);
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float gb = bf16_round(fmaf(g[j], sg[j], hg[j]));
          const float xb = bf16_round(fmaf(x[j], sx[j], hx[j]));
          const float a = fmaxf(bf16_round(gb + xb), 0.f);
          const float da = a > 0.f ? dq * wp[j] : 0.f;
          ab[j] += da;
          agg[j] = fmaf(da, g[j] - mg[j], agg[j]);
          agx[j] = fmaf(da, x[j] - mx[j], agx[j]);
          aw[j] = fmaf(dq, a, aw[j]);
        }
        if (lig == 0) abp += dq;
      }
    }
    if (det.partial == nullptr) {
#pragma unroll
      for (int j = 0; j < V; ++j) {
        atomicAdd(&red[0 * fw + lig * V + j], ab[j]);
        atomicAdd(&red[1 * fw + lig * V + j], agg[j] * __ldg(c.invstd_g + lig * V + j));
        atomicAdd(&red[2 * fw + lig * V + j], agx[j] * __ldg(c.invstd_x + lig * V + j));
        atomicAdd(&red[3 * fw + lig * V + j], aw[j]);
      }
      if (lig == 0) atomicAdd(&red[4 * fw], abp);
    }
  }
  if (det.partial != nullptr) {
    // deterministic mode: the pixel groups of the block add their sums one after the other (fixed order)
    for (int gsel = 0; gsel < gpb; ++gsel) {
      if (grp == gsel && has) {
#pragma unroll
        for (int j = 0; j < V; ++j) {
          red[0 * fw + lig * V + j] += ab[j];
          red[1 * fw + lig * V + j] += agg[j] * __ldg(c.invstd_g + lig * V + j);
          red[2 * fw + lig * V + j] += agx[j] * __ldg(c.invstd_x + lig * V + j);
          red[3 * fw + lig * V + j] += aw[j];
        }
        if (lig == 0) red[4 * fw] += abp;
      }
      __syncthreads();
    }
  }
  __syncthreads();
  // partial-row layout in deterministic mode: [0, 4 fint) = sums, [4 fint, 5 fint) = dwpsi, [5 fint] = dbpsi
  for (int i = threadIdx.x; i < fw; i += blockDim.x) {
    const int ci = c_off + i;
    red_out(sums, det, 0 * fint + ci, (double)red[0 * fw + i]);   // dbeta_g
    red_out(sums, det, 1 * fint + ci, (double)red[1 * fw + i]);   // dgamma_g
    red_out(sums, det, 2 * fint + ci, (double)red[0 * fw + i]);   // dbeta_x (same upstream gradient)
    red_out(sums, det, 3 * fint + ci, (double)red[2 * fw + i]);   // dgamma_x
    if (det.partial != nullptr) det.partial[(size_t)blockIdx.x * det.n + 4 * fint + ci] = (double)red[3 * fw + i];
    else atomicAdd(&dwpsi[ci], red[3 * fw + i]);
  }
  if (threadIdx.x == 0 && blockIdx.y == 0) {       // every slice sees all pixels: sum dq is taken by the first one
    if (det.partial != nullptr) det.partial[(size_t)blockIdx.x * det.n + 5 * fint] = (double)red[4 * fw];
    else atomicAdd(dbpsi, red[4 * fw]);
  }
}

// backward phase 3: gradients w.r.t. the two pre-BN GEMM outputs.  Per channel the BatchNorm backward collapses to
//   dg1p = Wg*dq*[a>0] + Bg*g + Cg     with Wg = gamma*invstd*wpsi, Bg = -gamma*invstd^2*dgamma/m,
//                                           Cg = -gamma*invstd*dbeta/m - Bg*mean          (same for the x branch)
// so only the mask coefficients and three constants per branch stay in registers.  Also accumulates the column sums
// of the ROUNDED outputs = bias gradients of the W_g / W_x convolutions (dbias[0][c], dbias[1][c]).
template <int V, int U, int MINB>
__global__ void __launch_bounds__(256, MINB) gate_psi_bwd_apply_kernel(
    const float* __restrict__ dsig, const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ g1p,
    const __nv_bfloat16* __restrict__ x1p, int ld, long long npix, int fint, int tpp, int rows, GateBwdCoef c,
    const double* __restrict__ sums1, int training, const double* __restrict__ sums,
    __nv_bfloat16* __restrict__ dg1p, __nv_bfloat16* __restrict__ dx1p, float* __restrict__ dgamma_beta,
    float* __restrict__ dbn1, float* __restrict__ dbias, DetBuf det) {
  pdl_enter();
  using VT = typename GVec<V>::T;
  __shared__ float red[256 * V];
  // gridDim.y channel slices of tpp * V channels (see the reduce kernel)
  const int c_off = blockIdx.y * (tpp * V);
  g1p += c_off;
  x1p += c_off;
  dg1p += c_off;
  dx1p += c_off;
  const int gch = threadIdx.x % tpp, r = threadIdx.x / tpp;
  const bool active = r < rows && c_off + gch * V < fint;
  float bsg[V], bsx[V];
#pragma unroll
  for (int j = 0; j < V; ++j) bsg[j] = bsx[j] = 0.f;
  if (active) {
    float sg[V], hg[V], sx[V], hx[V], wg[V], bg[V], cg[V], wx[V], bx[V], cx[V];
    gv_loadf<V>(c.scale_g + c_off + gch * V, true, sg);
    gv_loadf<V>(c.shift_g + c_off + gch * V, true, hg);
    gv_loadf<V>(c.scale_x + c_off + gch * V, true, sx);
    gv_loadf<V>(c.shift_x + c_off + gch * V, true, hx);
    const double inv_m = 1.0 / (double)npix;
#pragma unroll
    for (int j = 0; j < V; ++j) {
      const int ch = c_off + gch * V + j;
      const float wp = bf16_round(__ldg(c.wpsi + ch));
      const float igv = __ldg(c.invstd_g + ch), mgv = __ldg(c.mean_g + ch);
      const float ixv = __ldg(c.invstd_x + ch), mxv = __ldg(c.mean_x + ch);
      const float cgv = __ldg(c.gamma_g + ch) * igv, cxv = __ldg(c.gamma_x + ch) * ixv;
      const double dbg = sums[0 * fint + ch], dgg = sums[1 * fint + ch], dgx = sums[3 * fint + ch];
      const float kb = training ? (float)(dbg * inv_m) : 0.f;
      const float kgg = training ? (float)(dgg * inv_m) : 0.f;
      const float kgx = training ? (float)(dgx * inv_m) : 0.f;
      wg[j] = cgv * wp;
      bg[j] = -cgv * kgg * igv;
      cg[j] = -cgv * kb - bg[j] * mgv;
      wx[j] = cxv * wp;
      bx[j] = -cxv * kgx * ixv;
      cx[j] = -cxv * kb - bx[j] * mxv;
      if (blockIdx.x == 0 && r == 0) {
        dgamma_beta[0 * fint + ch] = (float)dgg;
        dgamma_beta[1 * fint + ch] = (float)dbg;
        dgamma_beta[2 * fint + ch] = (float)dgx;
        dgamma_beta[3 * fint + ch] = (float)dbg;
      }
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
      dbn1[0] = (float)sums1[1];   // dgamma1
      dbn1[1] = (float)sums1[0];   // dbeta1
    }
    const float g1 = __ldg(c.gamma1), mu1 = __ldg(c.mean1), is1 = __ldg(c.invstd1);
    const float k0 = (float)(sums1[0] * inv_m), k1 = (float)(sums1[1] * inv_m);
    const long long stride = (long long)gridDim.x * rows;
    // U pixels in flight per thread
    for (long long p0 = (long long)blockIdx.x * rows + r; p0 < npix; p0 += U * stride) {
      VT gv[U], xv[U];
      float ds[U], qv[U];
      bool ok[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long p = p0 + u * stride;
        ok[u] = p < npix;
        const long long pc = ok[u] ? p : p0;
        gv[u] = __ldg(reinterpret_cast<const VT*>(g1p + pc * ld + gch * V));
        xv[u] = __ldg(reinterpret_cast<const VT*>(x1p + pc * ld + gch * V));
        ds[u] = __ldg(dsig + pc);
        qv[u] = __bfloat162float(q[pc]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (!ok[u]) continue;
        const long long p = p0 + u * stride;
        const float dq = gate_dq(ds[u], qv[u], g1, mu1, is1, training, k0, k1);
        float g[V], x[V];
        gv_unpack<V>(gv[u], g);
        gv_unpack<V>(xv[u], x);
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float gb = bf16_round(fmaf(g[j], sg[j], hg[j]));
          const float xb = bf16_round(fmaf(x[j], sx[j], hx[j]));
          const float dqm = bf16_round(gb + xb) > 0.f ? dq : 0.f;
          g[j] = fmaf(wg[j], dqm, fmaf(bg[j], g[j], cg[j]));
          x[j] = fmaf(wx[j], dqm, fmaf(bx[j], x[j], cx[j]));
        }
        const VT og = gv_pack<V>(g), ox = gv_pack<V>(x);
        *reinterpret_cast<VT*>(dg1p + p * ld + gch * V) = og;
        *reinterpret_cast<VT*>(dx1p + p * ld + gch * V) = ox;
        if (dbias != nullptr) {
          gv_unpack<V>(og, g);
          gv_unpack<V>(ox, x);
#pragma unroll
          for (int j = 0; j < V; ++j) {
            bsg[j] += g[j];
            bsx[j] += x[j];
          }
        }
      }
    }
  }
  if (dbias != nullptr) {
    for (int which = 0; which < 2; ++which) {
      float* v = which == 0 ? bsg : bsx;
      __syncthreads();
      if (active) {
#pragma unroll
        for (int j = 0; j < V; ++j) red[(r * tpp + gch) * V + j] = v[j];
      }
      __syncthreads();
      if (active && r == 0) {
#pragma unroll
        for (int j = 0; j < V; ++j) {
          float s = 0.f;
          for (int rr = 0; rr < rows; ++rr) s += red[(rr * tpp + gch) * V + j];
          red_out(dbias, det, which * fint + c_off + gch * V + j, s);
        }
      }
    }
  }
}

static int g_pow2ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}
// 4 channels per thread when F_int / 4 threads per pixel fit a 256-thread block (B200SEG_GATE_LIGHT=0: always 8)
static bool gate_light(int fint) {
  static const bool enabled = [] {
    const char* e = getenv("B200SEG_GATE_LIGHT");
    return !(e != nullptr && atoi(e) == 0);
  }();
  return enabled && fint % 4 == 0 && fint / 4 <= 256;
}
static int g_grid(long long units, int per_block, int waves) {
  long long g = (units + per_block - 1) / per_block;
  const long long cap = (long long)num_sms() * waves;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}
static bool g_al(const void* p, int ld) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && ld % 8 == 0; }

}  // namespace b2

using namespace b2;

extern "C" int b2_gate_psi_fwd(const void* g1p, const void* x1p, int32_t ld, int64_t npix, int32_t fint,
                               const float* scale_g, const float* shift_g, const float* scale_x,
                               const float* shift_x, const float* wpsi, const float* bpsi, void* q,
                               double* qstats, b2_stream_t stream) {
  B2_REQUIRE(fint % 8 == 0 && fint <= 256, B2_ERR_SHAPE, "F_int=%d must be a multiple of 8, <= 256", fint);
  B2_REQUIRE(g_al(g1p, ld) && g_al(x1p, ld), B2_ERR_ALIGN, "gate operands misaligned");
  const int L = g_pow2ceil(fint / 8);
  const int grid = g_grid(npix, 256 / L, 8);
  DetBuf det;
  int rc = det_begin(&det, grid, 2, (cudaStream_t)stream);
  if (rc) return rc;
  B2_CHECK_CUDA(launch_chain(gate_psi_fwd_kernel, dim3(grid), dim3(256), (size_t)(0), (cudaStream_t)stream, 1,
      (long long)npix * fint * 2, (const __nv_bfloat16*)g1p, (const __nv_bfloat16*)x1p, ld, npix, fint, L, scale_g,
      shift_g, scale_x, shift_x, wpsi, bpsi, (__nv_bfloat16*)q, qstats, det));
  B2_LAUNCH_CHECK();
  if (det.partial) return det_finish(det.partial, grid, det.n, 2, qstats, (cudaStream_t)stream);
  return B2_OK;
}

extern "C" int b2_gate_apply_fwd(const void* x, int32_t ldx, const void* q, int64_t npix, int32_t c,
                                 const float* scale1, const float* shift1, void* psi, void* out, int32_t ldo,
                                 b2_stream_t stream) {
  B2_REQUIRE(c % 8 == 0 && c <= 2048, B2_ERR_SHAPE, "gate C=%d must be a multiple of 8, <= 2048", c);
  B2_REQUIRE(g_al(x, ldx) && g_al(out, ldo), B2_ERR_ALIGN, "gate operands misaligned");
  const int tpp = c / 8, rows = 256 / tpp;
  B2_CHECK_CUDA(launch_chain(gate_apply_fwd_kernel, dim3(g_grid(npix, rows, 16)), dim3(256), (size_t)(0),
      (cudaStream_t)stream, 1, (long long)npix * c * 2, (const __nv_bfloat16*)x, ldx, (const __nv_bfloat16*)q, npix,
      tpp, rows, scale1, shift1, (__nv_bfloat16*)psi, (__nv_bfloat16*)out, ldo));
  B2_LAUNCH_CHECK();
  return B2_OK;
}

extern "C" int b2_gate_apply_bwd(const void* dout, int32_t lddout, const void* x, int32_t ldx, const void* psi,
                                 const void* q, int64_t npix, int32_t c, const float* mean1, const float* invstd1,
                                 void* dx, int32_t lddx, float* dsig, double* sums1, b2_stream_t stream) {
  B2_REQUIRE(c % 8 == 0, B2_ERR_SHAPE, "gate C=%d must be a multiple of 8", c);
  B2_REQUIRE(g_al(dout, lddout) && g_al(x, ldx) && g_al(dx, lddx), B2_ERR_ALIGN, "gate operands misaligned");
  int L = g_pow2ceil(c / 8);
  if (L > 32) L = 32;
  const int grid = g_grid(npix, 256 / L, 8);
  DetBuf det;
  int rc = det_begin(&det, grid, 2, (cudaStream_t)stream);
  if (rc) return rc;
  B2_CHECK_CUDA(launch_chain(gate_apply_bwd_kernel, dim3(grid), dim3(256), (size_t)(0), (cudaStream_t)stream, 1,
      (long long)npix * c * 2, (const __nv_bfloat16*)dout, lddout, (const __nv_bfloat16*)x, ldx,
      (const __nv_bfloat16*)psi, (const __nv_bfloat16*)q, npix, c / 8, L, mean1, invstd1, (__nv_bfloat16*)dx, lddx,
      dsig, sums1, det));
  B2_LAUNCH_CHECK();
  if (det.partial) return det_finish(det.partial, grid, det.n, 2, sums1, (cudaStream_t)stream);
  return B2_OK;
}

static GateBwdCoef make_coef(const b2_gate_coef* k) {
  GateBwdCoef c;
  c.scale_g = k->scale_g; c.shift_g = k->shift_g; c.mean_g = k->mean_g; c.invstd_g = k->invstd_g;
  c.gamma_g = k->gamma_g;
  c.scale_x = k->scale_x; c.shift_x = k->shift_x; c.mean_x = k->mean_x; c.invstd_x = k->invstd_x;
  c.gamma_x = k->gamma_x;
  c.gamma1 = k->gamma1; c.mean1 = k->mean1; c.invstd1 = k->invstd1;
  c.wpsi = k->wpsi;
  return c;
}

extern "C" int b2_gate_psi_bwd_reduce(const float* dsig, const void* q, const void* g1p, const void* x1p,
                                      int32_t ld, int64_t npix, int32_t fint, const b2_gate_coef* coef,
                                      const double* sums1, int32_t training, double* sums, float* dwpsi,
                                      float* dbpsi, b2_stream_t stream) {
  B2_REQUIRE(fint % 8 == 0 && fint <= 256, B2_ERR_SHAPE, "F_int=%d must be a multiple of 8, <= 256", fint);
  B2_REQUIRE(g_al(g1p, ld) && g_al(x1p, ld), B2_ERR_ALIGN, "gate operands misaligned");
  const bool light = gate_light(fint);
  // 64-channel slices (gridDim.y) once F_int exceeds one: 16 threads per pixel, 16 pixels per block iteration
  const int slice = (light && fint > 64 && env_switch("B200SEG_GATE_SLICE", 1) != 0) ? 64 : 0;
  const int slices = slice ? (fint + slice - 1) / slice : 1;
  const size_t smem = (size_t)(4 * (slice ? slice : fint) + 1) * sizeof(float);
  const int L = g_pow2ceil((slice ? slice : fint) / (light ? 4 : 8));
  int grid = g_grid(npix, 256 / L, light ? 8 : 4);
  grid = (grid + slices - 1) / slices;
  DetBuf det;
  int rc = det_begin(&det, grid, 5 * fint + 1, (cudaStream_t)stream);
  if (rc) return rc;
  if (light && env_switch("B200SEG_GATE_U", fint <= 128 ? 4 : 2) == 4) {
    B2_CHECK_CUDA(launch_chain(gate_psi_bwd_reduce_kernel<4, 4, 2>, dim3(grid, slices), dim3(256), (size_t)(smem),
        (cudaStream_t)stream, 1, (long long)npix * fint * 2, dsig, (const __nv_bfloat16*)q, (const __nv_bfloat16*)g1p,
        (const __nv_bfloat16*)x1p, ld, npix, fint, L, make_coef(coef), sums1, training, sums, dwpsi, dbpsi, slice,
        det));
  } else if (light) {
    B2_CHECK_CUDA(launch_chain(gate_psi_bwd_reduce_kernel<4, 2, 3>, dim3(grid, slices), dim3(256), (size_t)(smem),
        (cudaStream_t)stream, 1, (long long)npix * fint * 2, dsig, (const __nv_bfloat16*)q, (const __nv_bfloat16*)g1p,
        (const __nv_bfloat16*)x1p, ld, npix, fint, L, make_coef(coef), sums1, training, sums, dwpsi, dbpsi, slice,
        det));
  } else {
    B2_CHECK_CUDA(launch_chain(gate_psi_bwd_reduce_kernel<8, 2, 2>, dim3(grid), dim3(256), (size_t)(smem),
        (cudaStream_t)stream, 1, (long long)npix * fint * 2, dsig, (const __nv_bfloat16*)q, (const __nv_bfloat16*)g1p,
        (const __nv_bfloat16*)x1p, ld, npix, fint, L, make_coef(coef), sums1, training, sums, dwpsi, dbpsi, 0, det));
  }
  B2_LAUNCH_CHECK();
  if (det.partial) {
    const DetSeg seg[3] = {det_seg(0, 4 * fint, sums), det_seg(4 * fint, fint, dwpsi), det_seg(5 * fint, 1, dbpsi)};
    return det_finish(det.partial, grid, det.n, seg, 3, (cudaStream_t)stream);
  }
  return B2_OK;
}

extern "C" int b2_gate_psi_bwd_apply(const float* dsig, const void* q, const void* g1p, const void* x1p,
                                     int32_t ld, int64_t npix, int32_t fint, const b2_gate_coef* coef,
                                     const double* sums1, int32_t training, const double* sums, void* dg1p,
                                     void* dx1p, float* dgamma_beta, float* dbn1, float* dbias,
                                     b2_stream_t stream) {
  B2_REQUIRE(fint % 8 == 0 && fint <= 256, B2_ERR_SHAPE, "F_int=%d must be a multiple of 8, <= 256", fint);
  B2_REQUIRE(g_al(g1p, ld) && g_al(x1p, ld) && g_al(dg1p, ld) && g_al(dx1p, ld), B2_ERR_ALIGN,
             "gate operands misaligned");
  const bool light = gate_light(fint);
  int tpp = fint / (light ? 4 : 8), slices = 1;
  if (light && fint > 64 && env_switch("B200SEG_GATE_SLICE", 1) != 0) {
    tpp = 16;                                     // 64-channel slices
    slices = (fint + 63) / 64;
  }
  const int rows = 256 / tpp;
  int grid = g_grid(npix, rows, 8);
  grid = (grid + slices - 1) / slices;
  DetBuf det;
  det.partial = nullptr;
  det.n = 2 * fint;
  if (dbias != nullptr) {
    int rc = det_begin(&det, grid, 2 * fint, (cudaStream_t)stream);
    if (rc) return rc;
  }
  if (light && env_switch("B200SEG_GATE_U", fint <= 128 ? 4 : 2) == 4) {
    B2_CHECK_CUDA(launch_chain(gate_psi_bwd_apply_kernel<4, 4, 2>, dim3(grid, slices), dim3(256), (size_t)(0),
        (cudaStream_t)stream, 1, (long long)npix * fint * 2, dsig, (const __nv_bfloat16*)q, (const __nv_bfloat16*)g1p,
        (const __nv_bfloat16*)x1p, ld, npix, fint, tpp, rows, make_coef(coef), sums1, training, sums,
        (__nv_bfloat16*)dg1p, (__nv_bfloat16*)dx1p, dgamma_beta, dbn1, dbias, det));
  } else if (light) {
    B2_CHECK_CUDA(launch_chain(gate_psi_bwd_apply_kernel<4, 2, 3>, dim3(grid, slices), dim3(256), (size_t)(0),
        (cudaStream_t)stream, 1, (long long)npix * fint * 2, dsig, (const __nv_bfloat16*)q, (const __nv_bfloat16*)g1p,
        (const __nv_bfloat16*)x1p, ld, npix, fint, tpp, rows, make_coef(coef), sums1, training, sums,
        (__nv_bfloat16*)dg1p, (__nv_bfloat16*)dx1p, dgamma_beta, dbn1, dbias, det));
  } else {
    B2_CHECK_CUDA(launch_chain(gate_psi_bwd_apply_kernel<8, 2, 2>, dim3(grid), dim3(256), (size_t)(0),
        (cudaStream_t)stream, 1, (long long)npix * fint * 2, dsig, (const __nv_bfloat16*)q, (const __nv_bfloat16*)g1p,
        (const __nv_bfloat16*)x1p, ld, npix, fint, tpp, rows, make_coef(coef), sums1, training, sums,
        (__nv_bfloat16*)dg1p, (__nv_bfloat16*)dx1p, dgamma_beta, dbn1, dbias, det));
  }
  B2_LAUNCH_CHECK();
  if (det.partial) return det_finish(det.partial, grid, det.n, 2 * fint, dbias, (cudaStream_t)stream);
  return B2_OK;
}
