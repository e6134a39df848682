// b200seg — CUDA-core convolutions for the two shapes that are memory-bound by construction:
//   * image stem, Cin <= 4 (AttentionUNet.py:6 basic_block(3,64) first conv; R2U_Net.py:43 RRCNN1.conv_1x1 3->64):
//     K = 27 (or 3) is far below one MMA K step, the layer is 0.17 % of the step FLOPs and bound by the 64-channel
//     output write;
//   * Cout <= 8 1x1 heads (AttentionUNet.py:84 `out`, R2U_Net.py:76 `conv_1x1`, ResnetUnet.py:58 `out`): a dot
//     product per pixel.
// Weights are rounded to bf16 on load, matching what autocast feeds the reference convolution.
#include "common.cuh"

namespace b2 {

// ------------------------------------------------------------------------------------------------------------
// stem forward: x4 NHWC bf16 (4 channels, zero padded), wk fp32 [cout][taps][4]
// ------------------------------------------------------------------------------------------------------------
template <int KS>
__global__ void __launch_bounds__(128) smallc_fprop_kernel(const uint2* __restrict__ x4, int n, int h, int w,
                                                           const float* __restrict__ wk,
                                                           const float* __restrict__ bias, int cout,
                                                           __nv_bfloat16* __restrict__ y, int ldy, int relu) {
  constexpr int TAPS = KS * KS;
  extern __shared__ float sm[];
  float* sw = sm;                       // [cout][TAPS][4]
  float* sb = sm + cout * TAPS * 4;     // [cout]
  for (int i = threadIdx.x; i < cout * TAPS * 4; i += blockDim.x) sw[i] = bf16_round(wk[i]);
  for (int i = threadIdx.x; i < cout; i += blockDim.x) sb[i] = bias ? bias[i] : 0.f;
  __syncthreads();
  const long long total = (long long)n * h * w;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total;
       p += (long long)gridDim.x * blockDim.x) {
    const int xx = (int)(p % w);
    const int yy = (int)((p / w) % h);
    float in[TAPS][4];
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
      const int dy = (KS == 3) ? t / 3 - 1 : 0, dx = (KS == 3) ? t % 3 - 1 : 0;
      const int y2 = yy + dy, x2 = xx + dx;
      uint2 u = make_uint2(0u, 0u);
      if (y2 >= 0 && y2 < h && x2 >= 0 && x2 < w) u = __ldg(x4 + p + (long long)dy * w + dx);
      in[t][0] = bf16lo(u.x); in[t][1] = bf16hi(u.x); in[t][2] = bf16lo(u.y); in[t][3] = bf16hi(u.y);
    }
    __nv_bfloat16* yp = y + p * ldy;
    for (int co = 0; co < cout; co += 8) {
      float acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float a = sb[co + j];
        const float4* wp = reinterpret_cast<const float4*>(sw + (size_t)(co + j) * TAPS * 4);
#pragma unroll
        for (int t = 0; t < TAPS; ++t) {
          const float4 wv = wp[t];
          a = fmaf(in[t][0], wv.x, a);
          a = fmaf(in[t][1], wv.y, a);
          a = fmaf(in[t][2], wv.z, a);
          a = fmaf(in[t][3], wv.w, a);
        }
        acc[j] = relu ? fmaxf(a, 0.f) : a;
      }
      *reinterpret_cast<uint4*>(yp + co) = make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]),
                                                      pack_bf16x2(acc[4], acc[5]), pack_bf16x2(acc[6], acc[7]));
    }
  }
}

// stem weight gradient: dw[co][tap][c] += sum_p dy[p][co] * x4[p (+) tap][c]      (cout == 64)
// Register-tiled CUDA-core GEMM  [64 co] x [TAPS*4 columns] over K = pixels: a block stages 128 pixels of dY (bf16)
// and their im2col rows (fp32) in shared memory; thread (co, group) keeps CPG accumulators and reads the im2col row
// as warp-wide broadcasts.  Partial sums go to dw with fp32 atomics (one per accumulator per block).
template <int KS>
__global__ void __launch_bounds__(256) smallc_wgrad_kernel(const __nv_bfloat16* __restrict__ dy, int lddy,
                                                           const uint2* __restrict__ x4, int n, int h, int w,
                                                           float* __restrict__ dw, DetBuf det) {
  constexpr int TAPS = KS * KS;
  constexpr int NC = TAPS * 4;                 // im2col columns
  constexpr int CPG = (NC + 3) / 4;            // columns per thread group (9 or 1)
  constexpr int GST = (CPG + 3) / 4 * 4;       // padded group stride in floats (12 or 4) -> 16 B aligned rows
  constexpr int TP = 128;                      // pixels per tile
  __shared__ __align__(16) __nv_bfloat16 dy_s[TP][64];
  __shared__ __align__(16) float xc_s[TP][4 * GST];
  const int t = threadIdx.x;
  const int co = t & 63, grp = t >> 6;
  float acc[CPG];
#pragma unroll
  for (int k = 0; k < CPG; ++k) acc[k] = 0.f;
  const long long total = (long long)n * h * w;
  const long long tiles = (total + TP - 1) / TP;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long p0 = tile * TP;
    // dY tile: 128 px x 64 co bf16 = 1024 x 16 B
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = t + i * 256;
      const int px = idx >> 3, c8 = idx & 7;
      const long long p = p0 + px;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (p < total) v = __ldg(reinterpret_cast<const uint4*>(dy + p * lddy + c8 * 8));
      *reinterpret_cast<uint4*>(&dy_s[px][c8 * 8]) = v;
    }
    // im2col rows: two threads per pixel, taps split between them
    {
      const int px = t & 127, half = t >> 7;
      const long long p = p0 + px;
      const int xx = (int)(p % w);
      const int yy = (int)((p / w) % h);
#pragma unroll
      for (int tp = 0; tp < TAPS; ++tp) {
        if ((tp & 1) != half) continue;
        const int ddy = (KS == 3) ? tp / 3 - 1 : 0, ddx = (KS == 3) ? tp % 3 - 1 : 0;
        const int y2 = yy + ddy, x2 = xx + ddx;
        uint2 u = make_uint2(0u, 0u);
        if (p < total && y2 >= 0 && y2 < h && x2 >= 0 && x2 < w) u = __ldg(x4 + p + (long long)ddy * w + ddx);
        const float f[4] = {bf16lo(u.x), bf16hi(u.x), bf16lo(u.y), bf16hi(u.y)};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int col = tp * 4 + c;
          xc_s[px][(col / CPG) * GST + col % CPG] = f[c];
        }
      }
    }
    __syncthreads();
#pragma unroll 4
    for (int px = 0; px < TP; ++px) {
      const float a = __bfloat162float(dy_s[px][co]);
      const float* xr = &xc_s[px][grp * GST];
#pragma unroll
      for (int k = 0; k < CPG; ++k) acc[k] = fmaf(a, xr[k], acc[k]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < CPG; ++k) {
    const int col = grp * CPG + k;
    if (col < NC) red_out(dw, det, co * NC + col, acc[k]);
  }
}

// ------------------------------------------------------------------------------------------------------------
// heads: y[b][co][hw] = sum_c x[p][c] * w[co][c] + bias[co]      (fp32 out, NCHW)
// L lanes cooperate on one pixel, each lane owns 8 channels (requires cin/8 <= L <= 32).
// ------------------------------------------------------------------------------------------------------------
template <int CO>
__global__ void __launch_bounds__(256) head_fwd_kernel(const __nv_bfloat16* __restrict__ x, int ldx,
                                                       long long npix, int hw, int cin,
                                                       const float* __restrict__ w, const float* __restrict__ bias,
                                                       int cout, int L, float* __restrict__ y) {
  const int lig = threadIdx.x % L;           // lane in group
  const int grp = threadIdx.x / L;
  const int gpb = blockDim.x / L;
  const bool has = lig * 8 < cin;
  float wr[CO][8];
#pragma unroll
  for (int co = 0; co < CO; ++co)
#pragma unroll
    for (int j = 0; j < 8; ++j) wr[co][j] = (has && co < cout) ? bf16_round(w[co * cin + lig * 8 + j]) : 0.f;
  // block-uniform trip count so the full-mask shuffles below are always executed by every lane
  constexpr int U = CO <= 2 ? 4 : 2;            // pixels in flight per thread
  const long long stride = (long long)gridDim.x * gpb;
  for (long long base = (long long)blockIdx.x * gpb; base < npix; base += U * stride) {
    uint4 u[U];
    bool live[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const long long p = base + k * stride + grp;
      live[k] = p < npix;
      u[k] = (has && live[k]) ? __ldg(reinterpret_cast<const uint4*>(x + p * ldx + lig * 8)) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const long long p = base + k * stride + grp;
      float f[8];
      f[0] = bf16lo(u[k].x); f[1] = bf16hi(u[k].x); f[2] = bf16lo(u[k].y); f[3] = bf16hi(u[k].y);
      f[4] = bf16lo(u[k].z); f[5] = bf16hi(u[k].z); f[6] = bf16lo(u[k].w); f[7] = bf16hi(u[k].w);
      // (pixel counts are far below 2^31: 32-bit division)
      const unsigned b = (unsigned)p / (unsigned)hw, r = (unsigned)p - b * (unsigned)hw;
#pragma unroll
      for (int co = 0; co < CO; ++co) {
        if (co < cout) {
          float s = 0.f;
#pragma unroll
          for (int j = 0; j < 8; ++j) s = fmaf(f[j], wr[co][j], s);
          for (int o = L >> 1; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
          if (lig == 0 && live[k]) y[((long long)b * cout + co) * hw + r] = s + (bias ? bias[co] : 0.f);
        }
      }
    }
  }
}

template <int CO>
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ dy,
                                                       const __nv_bfloat16* __restrict__ x, int ldx,
                                                       long long npix, int hw, int cin,
                                                       const float* __restrict__ w, int cout, int L,
                                                       __nv_bfloat16* __restrict__ dx, int lddx,
                                                       float* __restrict__ dw, float* __restrict__ db, DetBuf det) {
  extern __shared__ float sacc[];   // [cout][cin] + [cout]
  for (int i = threadIdx.x; i < cout * cin + cout; i += blockDim.x) sacc[i] = 0.f;
  __syncthreads();
  const int lig = threadIdx.x % L;
  const int grp = threadIdx.x / L;
  const int gpb = blockDim.x / L;
  const bool has = lig * 8 < cin;
  float wr[CO][8], aw[CO][8], ab[CO];
#pragma unroll
  for (int co = 0; co < CO; ++co) {
    ab[co] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      wr[co][j] = (has && co < cout) ? bf16_round(w[co * cin + lig * 8 + j]) : 0.f;
      aw[co][j] = 0.f;
    }
  }
  constexpr int U = CO <= 2 ? 4 : 2;            // pixels in flight per thread (loads issued before the math)
  const long long pstride = (long long)gridDim.x * gpb;
  for (long long p0 = (long long)blockIdx.x * gpb + grp; p0 < npix; p0 += U * pstride) {
    uint4 xu[U];
    float dv[U][CO];
    bool live[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const long long p = p0 + k * pstride;
      live[k] = p < npix;
      const long long pc = live[k] ? p : p0;
      const long long b = (unsigned)pc / (unsigned)hw, r = (unsigned)pc - (unsigned)b * (unsigned)hw;   // npix < 2^31
      xu[k] = has ? __ldg(reinterpret_cast<const uint4*>(x + pc * ldx + lig * 8)) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int co = 0; co < CO; ++co) dv[k][co] = (co < cout && live[k]) ? __ldg(dy + (b * cout + co) * hw + r) : 0.f;
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      if (!live[k]) continue;
      const long long p = p0 + k * pstride;
      float f[8], g[8];
      f[0] = bf16lo(xu[k].x); f[1] = bf16hi(xu[k].x); f[2] = bf16lo(xu[k].y); f[3] = bf16hi(xu[k].y);
      f[4] = bf16lo(xu[k].z); f[5] = bf16hi(xu[k].z); f[6] = bf16lo(xu[k].w); f[7] = bf16hi(xu[k].w);
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] = 0.f;
#pragma unroll
      for (int co = 0; co < CO; ++co) {
        if (co < cout) {
          const float d = dv[k][co];
          if (lig == 0) ab[co] += d;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            g[j] = fmaf(d, wr[co][j], g[j]);
            aw[co][j] = fmaf(d, f[j], aw[co][j]);
          }
        }
      }
      if (has && dx != nullptr) {
        *reinterpret_cast<uint4*>(dx + p * lddx + lig * 8) =
            make_uint4(pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]), pack_bf16x2(g[4], g[5]),
                       pack_bf16x2(g[6], g[7]));
      }
    }
  }
  if (det.partial == nullptr) {
    if (has) {
#pragma unroll
      for (int co = 0; co < CO; ++co) {
        if (co < cout) {
#pragma unroll
          for (int j = 0; j < 8; ++j) atomicAdd(&sacc[co * cin + lig * 8 + j], aw[co][j]);
          if (lig == 0) atomicAdd(&sacc[cout * cin + co], ab[co]);
        }
      }
    }
  } else {
    // deterministic mode: the pixel groups of the block add their sums one after the other (fixed order)
    for (int gsel = 0; gsel < gpb; ++gsel) {
      if (grp == gsel && has) {
#pragma unroll
        for (int co = 0; co < CO; ++co) {
          if (co < cout) {
#pragma unroll
            for (int j = 0; j < 8; ++j) sacc[co * cin + lig * 8 + j] += aw[co][j];
            if (lig == 0) sacc[cout * cin + co] += ab[co];
          }
        }
      }
      __syncthreads();
    }
  }
  __syncthreads();
  // partial-row layout in deterministic mode: [0, cout*cin) = dw, [cout*cin, cout*cin + cout) = db
  for (int i = threadIdx.x; i < cout * cin + cout; i += blockDim.x) {
    if (det.partial != nullptr) det.partial[(size_t)blockIdx.x * det.n + i] = (double)sacc[i];
    else if (i < cout * cin) atomicAdd(&dw[i], sacc[i]);
    else atomicAdd(&db[i - cout * cin], sacc[i]);
  }
}

static int pow2ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

}  // namespace b2

using namespace b2;

extern "C" int b2_conv_smallc_fprop(const void* x4, int32_t n, int32_t h, int32_t w, int32_t ksize,
                                    const float* wk, const float* bias, int32_t cout, void* y, int32_t ldy,
                                    int32_t relu, b2_stream_t stream) {
  B2_REQUIRE(ksize == 1 || ksize == 3, B2_ERR_SHAPE, "ksize %d unsupported", ksize);
  B2_REQUIRE(cout % 8 == 0 && cout <= 512, B2_ERR_SHAPE, "cout=%d must be a multiple of 8, <= 512", cout);
  B2_REQUIRE(ldy % 8 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0, B2_ERR_ALIGN, "y misaligned");
  const long long total = (long long)n * h * w;
  long long grid = (total + 127) / 128;
  const long long cap = (long long)num_sms() * 16;
  if (grid > cap) grid = cap;
  const int taps = ksize * ksize;
  const size_t smem = (size_t)cout * taps * 4 * sizeof(float) + cout * sizeof(float);
  if (ksize == 3)
    smallc_fprop_kernel<3><<<(unsigned)grid, 128, smem, (cudaStream_t)stream>>>(
        (const uint2*)x4, n, h, w, wk, bias, cout, (__nv_bfloat16*)y, ldy, relu);
  else
    smallc_fprop_kernel<1><<<(unsigned)grid, 128, smem, (cudaStream_t)stream>>>(
        (const uint2*)x4, n, h, w, wk, bias, cout, (__nv_bfloat16*)y, ldy, relu);
  B2_LAUNCH_CHECK();
  return B2_OK;
}

extern "C" int b2_conv_smallc_wgrad(const void* dy, int32_t lddy, const void* x4, int32_t n, int32_t h, int32_t w,
                                    int32_t ksize, int32_t cout, float* dw, b2_stream_t stream) {
  B2_REQUIRE(ksize == 1 || ksize == 3, B2_ERR_SHAPE, "ksize %d unsupported", ksize);
  B2_REQUIRE(cout == 64, B2_ERR_SHAPE, "stem wgrad supports cout == 64 (got %d)", cout);
  B2_REQUIRE(lddy % 8 == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0, B2_ERR_ALIGN, "dy misaligned");
  const long long tiles = ((long long)n * h * w + 127) / 128;
  long long grid = (long long)num_sms() * 5;
  if (grid > tiles) grid = tiles;
  const int ncol = cout * ksize * ksize * 4;
  DetBuf det;
  int rc = det_begin(&det, grid, ncol, (cudaStream_t)stream);
  if (rc) return rc;
  if (ksize == 3)
    smallc_wgrad_kernel<3><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)dy, lddy,
                                                                             (const uint2*)x4, n, h, w, dw, det);
  else
    smallc_wgrad_kernel<1><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)dy, lddy,
                                                                             (const uint2*)x4, n, h, w, dw, det);
  B2_LAUNCH_CHECK();
  if (det.partial) return det_finish(det.partial, grid, det.n, ncol, dw, (cudaStream_t)stream);
  return B2_OK;
}

extern "C" int b2_head_fwd(const void* x, int32_t ldx, int64_t npix, int32_t hw, int32_t cin, const float* w,
                           const float* bias, int32_t cout, float* y, b2_stream_t stream) {
  B2_REQUIRE(cin % 8 == 0 && cin <= 256, B2_ERR_SHAPE, "head cin=%d must be a multiple of 8, <= 256", cin);
  B2_REQUIRE(cout >= 1 && cout <= 8, B2_ERR_SHAPE, "head cout=%d must be in 1..8", cout);
  B2_REQUIRE(npix > 0 && npix < (1ll << 31) && hw > 0, B2_ERR_SHAPE, "head: pixel count out of range");
  B2_REQUIRE(ldx % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, B2_ERR_ALIGN, "x misaligned");
  const int L = pow2ceil(cin / 8);
  const int gpb = 256 / L;
  long long grid = (npix + gpb - 1) / gpb;
  const long long cap = (long long)num_sms() * 8;
  if (grid > cap) grid = cap;
#define B2_HEAD_FWD(CO) head_fwd_kernel<CO><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>( \
      (const __nv_bfloat16*)x, ldx, npix, hw, cin, w, bias, cout, L, y)
  if (cout == 1) B2_HEAD_FWD(1); else if (cout == 2) B2_HEAD_FWD(2); else if (cout <= 4) B2_HEAD_FWD(4); else B2_HEAD_FWD(8);
#undef B2_HEAD_FWD
  B2_LAUNCH_CHECK();
  return B2_OK;
}

extern "C" int b2_head_bwd(const float* dy, const void* x, int32_t ldx, int64_t npix, int32_t hw, int32_t cin,
                           const float* w, int32_t cout, void* dx, int32_t lddx, float* dw, float* db,
                           b2_stream_t stream) {
  B2_REQUIRE(cin % 8 == 0 && cin <= 256, B2_ERR_SHAPE, "head cin=%d must be a multiple of 8, <= 256", cin);
  B2_REQUIRE(cout >= 1 && cout <= 8, B2_ERR_SHAPE, "head cout=%d must be in 1..8", cout);
  B2_REQUIRE(npix > 0 && npix < (1ll << 31) && hw > 0, B2_ERR_SHAPE, "head: pixel count out of range");
  B2_REQUIRE(ldx % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, B2_ERR_ALIGN, "x misaligned");
  B2_REQUIRE(dx == nullptr || (lddx % 8 == 0 && (reinterpret_cast<uintptr_t>(dx) & 15) == 0), B2_ERR_ALIGN,
             "dx misaligned");
  const int L = pow2ceil(cin / 8);
  const int gpb = 256 / L;
  long long grid = (npix + gpb - 1) / gpb;
  // (every block ends in cout * (cin + 1) atomics on the same addresses: few, long-running blocks)
  const long long cap = (long long)num_sms() * 6;
  if (grid > cap) grid = cap;
  const size_t smem = (size_t)(cout * cin + cout) * sizeof(float);
  DetBuf det;
  int rc = det_begin(&det, grid, cout * cin + cout, (cudaStream_t)stream);
  if (rc) return rc;
#define B2_HEAD_BWD(CO) head_bwd_kernel<CO><<<(unsigned)grid, 256, smem, (cudaStream_t)stream>>>( \
      dy, (const __nv_bfloat16*)x, ldx, npix, hw, cin, w, cout, L, (__nv_bfloat16*)dx, lddx, dw, db, det)
  if (cout == 1) B2_HEAD_BWD(1); else if (cout == 2) B2_HEAD_BWD(2); else if (cout <= 4) B2_HEAD_BWD(4); else B2_HEAD_BWD(8);
#undef B2_HEAD_BWD
  B2_LAUNCH_CHECK();
  if (det.partial) {
    const DetSeg seg[2] = {det_seg(0, cout * cin, dw), det_seg(cout * cin, cout, db)};
    return det_finish(det.partial, grid, det.n, seg, 2, (cudaStream_t)stream);
  }
  return B2_OK;
}
