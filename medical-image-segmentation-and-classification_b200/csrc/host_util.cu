// b200seg — host utilities: thread-local error string, arch check, TMA descriptor encoding.
#include <stdarg.h>
#include <stdlib.h>
#include <map>
#include <mutex>
#include <string>

#include "common.cuh"

namespace b2 {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return B2_ERR_CUDA;
}

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// ---------------------------------------------------------------------------------------------
// environment switches, read once
// ---------------------------------------------------------------------------------------------
static std::mutex g_env_mu;
static std::map<std::string, int> g_env_cache;

int env_switch(const char* name, int dflt) {
  std::lock_guard<std::mutex> lk(g_env_mu);
  auto it = g_env_cache.find(name);
  if (it != g_env_cache.end()) return it->second == INT32_MIN ? dflt : it->second;
  const char* v = getenv(name);
  const int val = v ? atoi(v) : INT32_MIN;       // INT32_MIN = "not set": the caller's default applies
  g_env_cache.emplace(name, val);
  return v ? val : dflt;
}

// ---------------------------------------------------------------------------------------------
// deterministic-reduction workspace
// ---------------------------------------------------------------------------------------------
static std::mutex g_det_mu;
static double* g_det_ws[64] = {nullptr};       // per device
static long long g_det_doubles[64] = {0};

static bool det_lookup(double** ws, long long* n) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return false;
  std::lock_guard<std::mutex> lk(g_det_mu);
  *ws = g_det_ws[dev];
  *n = g_det_doubles[dev];
  return *ws != nullptr;
}

bool det_enabled() {
  double* ws;
  long long n;
  return det_lookup(&ws, &n);
}

int det_begin(DetBuf* out, long long rows, int n, cudaStream_t stream, long long keep) {
  (void)stream;
  out->partial = nullptr;
  out->n = n;
  double* ws;
  long long cap;
  if (!det_lookup(&ws, &cap)) return B2_OK;
  const long long need = rows * (long long)n;
  B2_REQUIRE(keep + need <= cap, B2_ERR_WORKSPACE,
             "deterministic workspace too small: need %lld B, have %lld B (b2_set_deterministic)",
             (keep + need) * 8, cap * 8);
  out->partial = ws + keep;
  return B2_OK;
}

// Finish: one block per slab of up to 32 consecutive columns of one segment.  The block streams chunks of the slab's
// rows (kFinChunk doubles: 96 rows of 32 columns, 3072 rows of one column) through two shared-memory buffers, every
// thread holding kFinChunk / kFinThreads independent loads in flight, while one lane per column adds the previous
// chunk in row order.  The sum of a column is the same chain of fp64 additions as a serial loop over the rows, so the
// result does not depend on the slab width or the chunking; the loads no longer sit on that chain.
static constexpr int kFinThreads = 256;
static constexpr int kFinChunk = 3072;
static constexpr int kFinLoads = kFinChunk / kFinThreads;

struct DetFinishJob {
  const double* partial;
  long long rows;
  int row_stride;
  int nseg;
  DetSeg seg[kDetMaxSeg];
  int first_block[kDetMaxSeg + 1];    // blocks [first_block[s], first_block[s + 1]) finish segment s
};

__global__ void __launch_bounds__(kFinThreads) det_finish_kernel(DetFinishJob j) {
  __shared__ double buf[2][kFinChunk];
  pdl_enter();          // the producer has completed: its partial rows are complete and visible
  int s = 0;
  while (s + 1 < j.nseg && (int)blockIdx.x >= j.first_block[s + 1]) ++s;
  const DetSeg sg = j.seg[s];
  const int c0 = ((int)blockIdx.x - j.first_block[s]) * 32;
  const int w = sg.count - c0 < 32 ? sg.count - c0 : 32;        // columns of this slab
  const int ch = kFinChunk / w;                                  // rows per chunk
  const int per = ch * w;
  const long long rows = j.rows;
  const double* src = j.partial + sg.offset + c0;
  // element e = k * kFinThreads + threadIdx.x of a chunk is (row e / w, column e % w): a warp reads whole rows
  int er[kFinLoads], eo[kFinLoads];
#pragma unroll
  for (int k = 0; k < kFinLoads; ++k) {
    const int e = k * kFinThreads + (int)threadIdx.x;
    er[k] = e < per ? e / w : INT32_MAX;
    eo[k] = e < per ? er[k] * j.row_stride + (e - er[k] * w) : 0;
  }
  double v[kFinLoads];
  auto load = [&](long long r0) {
    const double* base = src + r0 * j.row_stride;
#pragma unroll
    for (int k = 0; k < kFinLoads; ++k) v[k] = r0 + er[k] < rows ? __ldg(base + eo[k]) : 0.0;
  };
  auto stash = [&](double* b) {
#pragma unroll
    for (int k = 0; k < kFinLoads; ++k)
      if (k * kFinThreads + (int)threadIdx.x < per) b[k * kFinThreads + threadIdx.x] = v[k];
  };
  const long long nchunks = (rows + ch - 1) / ch;
  load(0);
  stash(buf[0]);
  __syncthreads();
  double acc = 0.0;
  for (long long q = 0; q < nchunks; ++q) {
    if (q + 1 < nchunks) load((q + 1) * ch);                     // in flight while the chunk q is added
    if ((int)threadIdx.x < w) {
      const double* b = buf[q & 1] + threadIdx.x;
      const int n = rows - q * ch < ch ? (int)(rows - q * ch) : ch;
#pragma unroll 8
      for (int r = 0; r < n; ++r) acc += b[r * w];
    }
    if (q + 1 < nchunks) stash(buf[(q + 1) & 1]);                // buffer (q + 1) & 1 was last read before the
    __syncthreads();                                             // previous barrier
  }
  if ((int)threadIdx.x < w) {
    const int i = c0 + (int)threadIdx.x;
    if (sg.f64) {
      double* d = static_cast<double*>(sg.dst);
      d[i] = d[i] + acc;
    } else {
      float* d = static_cast<float*>(sg.dst);
      d[i] = (float)((double)d[i] + acc);
    }
  }
}

int det_finish(const double* partial, long long rows, int row_stride, const DetSeg* seg, int nseg,
               cudaStream_t stream) {
  B2_REQUIRE(nseg >= 1 && nseg <= kDetMaxSeg && rows >= 1, B2_ERR_SHAPE, "det_finish: %d segments, %lld rows",
             nseg, rows);
  DetFinishJob j;
  j.partial = partial;
  j.rows = rows;
  j.row_stride = row_stride;
  j.nseg = nseg;
  int blocks = 0;
  for (int s = 0; s < nseg; ++s) {
    B2_REQUIRE(seg[s].count >= 0 && seg[s].offset >= 0 && seg[s].offset + seg[s].count <= row_stride, B2_ERR_SHAPE,
               "det_finish: segment %d (offset %d, count %d) outside a row of %d", s, seg[s].offset, seg[s].count,
               row_stride);
    j.seg[s] = seg[s];
    j.first_block[s] = blocks;
    blocks += (seg[s].count + 31) / 32;
  }
  j.first_block[nseg] = blocks;
  if (blocks == 0) return B2_OK;
  B2_CHECK_CUDA(launch_chain(det_finish_kernel, dim3(blocks), dim3(kFinThreads), (size_t)0, stream, 1,
                             rows * row_stride * (long long)sizeof(double), j));
  return B2_OK;
}
int det_finish(const double* partial, long long rows, int row_stride, int count, double* dst, cudaStream_t stream) {
  const DetSeg s = det_seg(0, count, dst);
  return det_finish(partial, rows, row_stride, &s, 1, stream);
}
int det_finish(const double* partial, long long rows, int row_stride, int count, float* dst, cudaStream_t stream) {
  const DetSeg s = det_seg(0, count, dst);
  return det_finish(partial, rows, row_stride, &s, 1, stream);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeTiledFn>(p);
    }
  });
  return fn;
}

int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz,
                     const uint32_t* elem_strides) {
  EncodeTiledFn fn = get_encode_fn();
  B2_REQUIRE(fn != nullptr, B2_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable (no driver?)");
  B2_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, B2_ERR_ALIGN, "TMA base pointer not 16B aligned");
  cuuint64_t gdim[5];
  cuuint64_t gstr[5];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = elem_strides ? elem_strides[i] : 1;
    if (i > 0) {
      gstr[i - 1] = strides_bytes[i];
      B2_REQUIRE((strides_bytes[i] & 15) == 0, B2_ERR_ALIGN, "TMA stride %d = %llu B not a multiple of 16", i,
                 (unsigned long long)strides_bytes[i]);
    }
  }
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr,
                  bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu,%llu,%llu,%llu] box [%u,%u,%u,%u]", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
              rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
    return B2_ERR_CUDA;
  }
  return B2_OK;
}

}  // namespace b2

extern "C" {

const char* b2_last_error(void) { return b2::g_err; }
int b2_abi_version(void) { return B2_ABI_VERSION; }
int b2_num_sms(void) { return b2::num_sms(); }

int b2_set_deterministic(void* workspace, int64_t bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return b2::cuda_fail(e, "cudaGetDevice");
  B2_REQUIRE(dev >= 0 && dev < 64, B2_ERR_SHAPE, "device index %d out of range", dev);
  B2_REQUIRE(workspace == nullptr || (bytes >= (1 << 20) && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0),
             B2_ERR_WORKSPACE, "deterministic workspace must be 16 B aligned and >= 1 MiB");
  std::lock_guard<std::mutex> lk(b2::g_det_mu);
  b2::g_det_ws[dev] = static_cast<double*>(workspace);
  b2::g_det_doubles[dev] = workspace ? bytes / 8 : 0;
  return B2_OK;
}

int b2_get_deterministic(void) { return b2::det_enabled() ? 1 : 0; }

int b2_det_finish(const double* partial, int64_t rows, int32_t row_stride, int32_t nseg, const int32_t* offsets,
                  const int32_t* counts, void* const* dsts, const int32_t* dst_f64, b2_stream_t stream) {
  B2_REQUIRE(nseg >= 1 && nseg <= b2::kDetMaxSeg, B2_ERR_SHAPE, "b2_det_finish: %d segments (1..%d)", nseg,
             b2::kDetMaxSeg);
  b2::DetSeg seg[b2::kDetMaxSeg];
  for (int s = 0; s < nseg; ++s) seg[s] = {offsets[s], counts[s], dsts[s], dst_f64[s] != 0 ? 1 : 0};
  return b2::det_finish(partial, rows, row_stride, seg, nseg, (cudaStream_t)stream);
}

int b2_reload_env(void) {
  std::lock_guard<std::mutex> lk(b2::g_env_mu);
  b2::g_env_cache.clear();
  return B2_OK;
}

int b2_arch_check(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return b2::cuda_fail(e, "cudaGetDevice");
  int major = 0, minor = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return b2::cuda_fail(e, "cudaDeviceGetAttribute");
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10 || minor != 0) {
    b2::set_error("libb200seg is built for sm_100a only; device %d is sm_%d%d", dev, major, minor);
    return B2_ERR_ARCH;
  }
  return B2_OK;
}

}  // extern "C"
