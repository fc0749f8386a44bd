// Shared helpers for the koemorph_b200 CUDA sources (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include "../../include/koemorph_b200.h"

namespace koe {

// ---- error plumbing for the C ABI ---------------------------------------------------------------
inline char* err_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}
inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}
inline std::atomic<int64_t>& launch_counter() {
  static std::atomic<int64_t> c{0};
  return c;
}
inline void count_launch(int n = 1) { launch_counter().fetch_add(n, std::memory_order_relaxed); }

#define KOE_CUDA(expr)                                                                            \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return koe::fail((int)_e, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                       __LINE__);                                                                 \
  } while (0)

// launch with programmatic stream serialisation (see pdl_wait below)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_after_primary_starts(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                               cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  static const bool no_pdl = getenv("KOE_NO_PDL") != nullptr;  // experiment switch
  cfg.numAttrs = no_pdl ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// the number of SMs of the current device, queried once per device
inline cudaError_t sm_count(int* n) {
  static std::atomic<int> cached[64];
  *n = 0;
  int dev = 0;
  if (cudaError_t e = cudaGetDevice(&dev)) return e;
  const bool cacheable = dev >= 0 && dev < 64;
  if (cacheable && (*n = cached[dev].load(std::memory_order_relaxed)) > 0) return cudaSuccess;
  if (cudaError_t e = cudaDeviceGetAttribute(n, cudaDevAttrMultiProcessorCount, dev)) return e;
  if (cacheable) cached[dev].store(*n, std::memory_order_relaxed);
  return cudaSuccess;
}

#define KOE_REQUIRE(cond, ...)                                   \
  do {                                                           \
    if (!(cond)) return koe::fail(KOE_E_INVALID, __VA_ARGS__);   \
  } while (0)

// Pinned host staging of small per-call tables (csrc/staging.cu): acquire a buffer of >= ints entries that no queued copy
// reads any more, fill host[0, ints), then upload_tables: one cudaMemcpyAsync to the device tables and the event that frees
// the buffer again.  check_capture refuses a call whose stream is capturing a CUDA graph (its tables change every call).
struct TableStaging {
  int32_t* host = nullptr;
  size_t ints = 0;
  cudaEvent_t copied = nullptr;
};
int acquire_table_staging(void* stream, size_t ints, TableStaging** out);
int upload_tables(TableStaging* b, int32_t* dev_tables, size_t ints, cudaStream_t stream);
int check_capture(void* stream, const char* what);

// ---- log-mel frontend launches (csrc/logmel.cu) -------------------------------------------------------------------------
enum class FrontendMode {
  Frames,      // frame j of clip c to row j of clip c's block of power / frame_max
  SplitPairs,  // the same for the even frames; frame 2j + 1 to row j of power_b / frame_max_b (the streaming step)
  Varlen,      // a packed variable-length batch (VarlenTables; default bank only)
};

// Packed variable-length batch: frame pair k of the launch is pair k - pair_base[c] of clip c (pair_base[c] <= k <
// pair_base[c + 1], `pairs` in all); clip c is `length[c]` samples at audio + sample_off[c] and has row_base[c + 1] -
// row_base[c] frames in this launch, frame j centred on sample (frame_offset + j * frame_step) * hop of the clip (window
// edges as lo_rel_hops / hi_rel_hops), stored to row row_base[c] + j of power / frame_max.  Of the koe_logmel_args it
// reads audio, hop, frame_offset, frame_step, lo/hi_rel_hops, power and frame_max.
struct VarlenTables {
  const long long* sample_off;
  const int* length;
  const int* pair_base;
  const int* row_base;
  int n_clips;
  long long pairs;
};

// Early release of the core (csrc/session.cu): the frontend counts up *flag once clips [0, clips) are stored.  The
// launcher sets `target` to the count that means so, or to 0 when this launch does not signal.
struct EarlyRelease {
  int clips;
  unsigned* flag;
  unsigned target;
};

// One frontend launch.  `follows_frontend_launch`: the kernel queued just before this one on `stream` is another frontend
// launch of the same forward, writing other buffers.  `early`: only a Frames launch with the default bank signals.
int launch_logmel(const koe_frontend_t* fe, const koe_logmel_args* a, FrontendMode mode, bool follows_frontend_launch,
                  void* stream, EarlyRelease* early = nullptr, const VarlenTables* varlen = nullptr);

// Destination of one mel-row variant: clip c's rows at power + c * power_stride, its maxima at frame_max + c * fmax_stride.
struct MelRows {
  float* power;
  float* frame_max;
  int64_t power_stride, fmax_stride;
};

// The frontend launches of one streaming hop (csrc/session.cu) over n_streams tails of tail_len samples, the newest
// complete frame centred `half` samples in: rows[v] receives mel-row variant v = F, R0, L0, R1, L1 (1 + 2 n_edge of them).
int launch_hop_frontend(const koe_frontend_t* fe, const float* tail, int n_streams, int tail_len, int half, int hop,
                        int n_edge, const MelRows* rows, void* stream);

// ---- device helpers ----------------------------------------------------------------------------
// Programmatic dependent launch (sm_90+): a kernel launched with launch_after_primary_starts() may begin while the
// previous kernel of the stream is still running, as soon as every CTA of that kernel has executed
// pdl_launch_dependents() (or exited) and an SM has room; it must execute pdl_wait() before it touches anything the
// previous kernel writes -- pdl_wait() returns once the previous kernel has completed and its writes are visible.
// Without the launch attribute both instructions are no-ops, so every kernel stays correct under a plain launch.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
constexpr unsigned kFullMask = 0xffffffffu;

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFullMask, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}

// librosa.power_to_db constants (amin = 1e-10, top_db = 80) -- see oracle/koemorph_oracle.py::power_to_db
constexpr float kAmin = 1e-10f;
constexpr float kTopDb = 80.0f;

__device__ __forceinline__ float power_db(float p) { return 10.0f * log10f(fmaxf(p, kAmin)); }
// dB value relative to ref_db, clamped at -top_db, optionally rescaled to [0, 1] by (x + 80) / 80
__device__ __forceinline__ float normalise_db(float db, float ref_db, bool rescale) {
  float x = fmaxf(db - ref_db, -kTopDb);
  return rescale ? (x + 80.0f) / 80.0f : x;
}

// ---- mbarrier + bulk copy (TMA, cp.async.bulk) wrappers for kernels that stream operands through a shared-memory ring
__device__ __forceinline__ uint32_t smem_u32addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbarrier_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbarrier_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbarrier_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded spin: a protocol bug traps (error to the host) instead of hanging the GPU
__device__ __forceinline__ void mbarrier_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  for (uint32_t spin = 0; !ok; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!ok && spin > (1u << 22)) __trap();
  }
}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

}  // namespace koe
