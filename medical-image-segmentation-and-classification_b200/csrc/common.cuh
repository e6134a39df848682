// b200seg — shared device/host helpers for the sm_100a kernels.
// Hand-written PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/b200seg.h"

namespace b2 {

// ---------------------------------------------------------------------------------------------
// host-side error plumbing (thread-local message, negative error codes; see include/b200seg.h)
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what);

#define B2_CHECK_CUDA(expr)                                            \
  do {                                                                 \
    cudaError_t _e = (expr);                                           \
    if (_e != cudaSuccess) return ::b2::cuda_fail(_e, #expr);          \
  } while (0)

#define B2_REQUIRE(cond, code, ...)                                    \
  do {                                                                 \
    if (!(cond)) { ::b2::set_error(__VA_ARGS__); return (code); }      \
  } while (0)

#define B2_LAUNCH_CHECK() B2_CHECK_CUDA(cudaGetLastError())

int num_sms();

// B200SEG_* switches are read from the environment ONCE (mutex-guarded cache; b2_reload_env() re-reads them): a launch
// costs no getenv scans, and concurrent forward / autograd-engine threads see one consistent configuration.
int env_switch(const char* name, int dflt);

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (B200SEG_PDL, default 2 = the size rule below).  A kernel launched through
// launch_chain() with the rule satisfied carries cudaLaunchAttributeProgrammaticStreamSerialization: its CTAs may
// become resident while the previous kernel of the stream is still draining, so its launch latency and prologue
// (barrier init, TMEM allocation, descriptor prefetch) overlap that kernel's tail — inside a captured graph the edge
// becomes a programmatic dependency.  EVERY kernel launched this way executes pdl_wait() on all threads before its
// first global-memory access (reads AND writes: the previous kernel may still be reading what this one overwrites);
// pdl_trigger() comes after the wait, so when a dependent's CTAs start, everything older than their direct
// predecessor has completed, and completion stays transitive along the chain.  Without the trigger the next kernel
// becomes resident when the CTAs exit.
// Both instructions are no-ops in a launch without the attribute.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() {
  pdl_wait();
  pdl_trigger();
}

// B200SEG_PDL: 0 off; 1 every chain launch; 2 (default) only launches whose tensor is at most B200SEG_PDL_MB (default 16) MiB —
// the launch-bound regime (batch-1 inference, a few images per GPU); a long memory-bound kernel whose CTAs sit
// resident behind the previous kernel only takes SM slots from the weight-gradient stream.
inline bool pdl_allowed(long long work_bytes) {
  const int mode = env_switch("B200SEG_PDL", 2);
  if (mode == 0) return false;
  if (mode == 1) return true;
  return work_bytes <= (long long)env_switch("B200SEG_PDL_MB", 16) * (1ll << 20);
}

// <<<grid, block, smem, stream>>> with the programmatic-serialization attribute when pdl_allowed(work_bytes) (the
// kernel must call pdl_wait() / pdl_enter() first thing).  `cluster` > 1 adds the cluster dimension.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                int cluster, long long work_bytes, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[2];
  unsigned n = 0;
  if (cluster > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = (unsigned)cluster;
    at[n].val.clusterDim.y = 1;
    at[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl_allowed(work_bytes)) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = at;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// TMA descriptor encode (driver entry point fetched through the runtime; no libcuda link dependency).
// dims/strides innermost-first; strides in BYTES for dims 1..rank-1; bf16 elements.
int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz,
                     const uint32_t* elem_strides = nullptr);

// ---------------------------------------------------------------------------------------------
// Deterministic-reduction mode (b2_set_deterministic, include/b200seg.h).  Kernels whose last step is a cross-block
// atomicAdd write ONE ROW of per-block partials into the registered workspace instead; det_finish adds the rows to the
// destination in block order.  With the mode off (`partial == nullptr`) the kernels use their atomics.
// The rows are not cleared: a producer writes every slot of its rows exactly once, or zeroes its own rows itself, and
// only after its pdl_wait() — every reduction reuses the start of the workspace, and the previous finish may still
// be reading it until then.
// ---------------------------------------------------------------------------------------------
struct DetBuf {
  double* partial;   // [rows][n] or nullptr
  int n;             // row length in doubles
};
// Reserve rows*n doubles of the workspace for a launch on `stream`.  out->partial stays nullptr when the mode is
// off.  Consecutive reservations of ONE entry point may coexist (`keep` = doubles already reserved by it).
int det_begin(DetBuf* out, long long rows, int n, cudaStream_t stream, long long keep = 0);
// dst[i] += sum over rows r (in order) of partial[r * row_stride + offset + i], i < count, for up to kDetMaxSeg
// segments of the same rows in ONE launch (dst double when f64, float otherwise)
static constexpr int kDetMaxSeg = 4;
struct DetSeg {
  int offset;
  int count;
  void* dst;
  int f64;
};
inline DetSeg det_seg(int offset, int count, double* dst) { return DetSeg{offset, count, dst, 1}; }
inline DetSeg det_seg(int offset, int count, float* dst) { return DetSeg{offset, count, dst, 0}; }
int det_finish(const double* partial, long long rows, int row_stride, const DetSeg* seg, int nseg, cudaStream_t stream);
int det_finish(const double* partial, long long rows, int row_stride, int count, double* dst, cudaStream_t stream);
int det_finish(const double* partial, long long rows, int row_stride, int count, float* dst, cudaStream_t stream);
bool det_enabled();

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
// final cross-block accumulation of a per-block value: atomics, or this block's slot of the partial rows
template <typename T>
__device__ __forceinline__ void red_out(T* dst, const DetBuf& d, int idx, T v) {
  if (d.partial != nullptr) d.partial[(size_t)blockIdx.x * d.n + idx] = (double)v;
  else atomicAdd(dst + idx, v);
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug becomes a trapped launch (reported as a CUDA error) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) { __trap(); }
  }
}

// ---- TMA loads (tile mode), completion on an mbarrier ----
__device__ __forceinline__ void tma_load_2d(void* smem, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// ---- thread-block clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {     // every thread of every CTA in the cluster
  asm volatile("barrier.cluster.arrive.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
}
// ---- CTA pairs (tcgen05 cta_group::2): the two CTAs of a 2-cluster feed ONE M = 256 MMA issued by the rank-0 CTA.
// Both CTAs load their own operand slices into their own shared memory, but the completion bytes are signalled on the
// LEADER's mbarrier (the MMA-issuing thread waits there), hence the .cta_group::2 form with a cluster-mapped barrier.
__device__ __forceinline__ uint32_t mapa_shared(uint32_t smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
// arrive on the mbarrier at this smem offset in CTA `cta_rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta_rank) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(mapa_shared(smem_u32(bar), cta_rank)) : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(void* smem, const CUtensorMap* tm, uint32_t leader_bar, int c0, int c1,
                                                 int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
      "[%2];" ::"r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(void* smem, const CUtensorMap* tm, uint32_t leader_bar, int c0, int c1,
                                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6}], [%2];" ::"r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_pair(void* smem, const CUtensorMap* tm, uint32_t leader_bar, int c0, int c1,
                                                 int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6, %7}], [%2];" ::"r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

// ---- tcgen05 ----
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// cta_group::2 forms: executed by the same warp of BOTH CTAs of the pair (same smem slot offset)
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate. One thread issues.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// M = 256 across the CTA pair: rows 0..127 accumulate in the leader's TMEM, rows 128..255 in the peer's; A comes from
// each CTA's own smem, B is N/2 rows from each (same smem offsets in both CTAs).  Issued by the LEADER only.
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs -> the mbarrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets TMEM lane (base_lane + i).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory matrix descriptor (sm_100 "version 1"), 128-byte swizzle.
//   start address >>4 in [0,14); LBO>>4 in [16,30); SBO>>4 in [32,46); version=1 in [46,48); layout type in [61,64)
// K-major  SW128: rows (M/N) are 128 B apart, 8-row groups SBO apart (1024 B when dense); LBO unused.
// MN-major SW128: 64-element MN blocks are LBO apart, 8-row K groups are SBO apart (1024 B when dense).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B and fp32 D.
__host__ __device__ __forceinline__ uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// One elected lane of a converged warp (elect.sync): the compiler knows the region is single-threaded, so TMA /
// MMA operands are moved to uniform registers once instead of through per-lane broadcast loops.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Column sums over the 32 lanes of a warp for 32 per-lane values (31 shuffles instead of 160).
// On return v[0] of lane l holds sum over all lanes of the original v[l].
__device__ __forceinline__ float warp_transpose_sum32(float* v, int lane) {
#pragma unroll
  for (int off = 16, n = 16; off >= 1; off >>= 1, n >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < n; ++i) {
      const float send = upper ? v[i] : v[i + n];
      const float keep = upper ? v[i + n] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }
#endif  // __CUDACC__

}  // namespace b2
