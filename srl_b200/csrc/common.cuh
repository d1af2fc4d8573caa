// Shared helpers for the srl_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/srl_b200.h"

namespace srl {

// ---- error plumbing: status codes + thread-local message, never abort() --------------------
void set_error(const char* fmt, ...);

#define SRL_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      ::srl::set_error(__VA_ARGS__);  \
      return (code);                  \
    }                                 \
  } while (0)

#define SRL_CUDA(call)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (call);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ::srl::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return SRL_ERR_CUDA;                                                                 \
    }                                                                                      \
  } while (0)

int sm_count();  // cached per device

// Programmatic dependent launch (srl_set_pdl / SRL_PDL, api.cu): a kernel launched with launch_pdl() may become
// resident while the kernel before it on the stream still runs -- once every CTA of that kernel has executed
// pdl_launch_dependents() (or exited) -- and must execute pdl_wait() before it touches anything the earlier kernel
// writes.  Off: plain launches (the device-side instructions are no-ops then).
bool pdl_enabled();
// The scan may only start ahead of the kernel before it when that kernel is this library's permutation kernel (which
// writes nothing the scan reads): srl_philox_perm notes its launch, the scan's launcher takes the note (once).  Behind
// anything else the scan is an ordinary launch -- it executes griddepcontrol.wait only at its end, so a programmatic
// launch behind a kernel that PRODUCES its inputs would read them without a visibility guarantee.
void pdl_note_perm(cudaStream_t st);
bool pdl_take_perm(cudaStream_t st);
// ... and the other way round (the order HotPath uses: the scan is the long pole of the step and starts first): the
// permutation kernel directly behind a scan starts beside it (it touches nothing the scan touches) and executes
// griddepcontrol.wait at ITS end, so that "permutation complete" implies "scan complete and visible" for the loss kernel
// behind it.  Only one of the two kernels of a pair is ever launched programmatically.
void pdl_note_scan(cudaStream_t st);
bool pdl_take_scan(cudaStream_t st);
void pdl_forget();

inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

// ---- device helpers ------------------------------------------------------------------------
#ifdef __CUDACC__

// Streaming (read-once / write-once) accesses: evict-first cache hints through the compiler intrinsics.
// (Not `asm volatile`: volatile asm pins the loads in program order, which serialises one DRAM round trip
// per loop iteration -- measured in profiles/r1_notes.md.  The intrinsics stay schedulable, so independent
// loads are hoisted and overlap.)
__device__ __forceinline__ float ldg_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ float2 ldg_stream(const float2* p) { return __ldcs(p); }
__device__ __forceinline__ float4 ldg_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ uint32_t ldg_stream(const uint32_t* p) { return __ldcs(p); }
__device__ __forceinline__ uint8_t ldg_stream(const uint8_t* p) { return __ldcs(p); }
__device__ __forceinline__ int4 ldg_stream(const int4* p) { return __ldcs(p); }
__device__ __forceinline__ __nv_bfloat16 ldg_stream(const __nv_bfloat16* p) { return __ldcs(p); }
__device__ __forceinline__ void stg_stream(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void stg_stream(float2* p, float2 v) { __stcs(p, v); }
__device__ __forceinline__ void stg_stream(float4* p, float4 v) { __stcs(p, v); }
__device__ __forceinline__ void stg_stream(int4* p, int4 v) { __stcs(p, v); }
__device__ __forceinline__ void stg_stream(__nv_bfloat16* p, __nv_bfloat16 v) { __stcs(p, v); }

// griddepcontrol.wait returns once every prerequisite grid has COMPLETED and its memory is visible (immediately when the
// kernel was launched without the programmatic attribute).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <class... KArgs, class... Args>
inline cudaError_t launch_maybe_pdl(bool programmatic, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                    cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (programmatic && pdl_enabled()) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
// a kernel that waits (pdl_wait) BEFORE it reads anything: always safe to launch programmatically (the loss kernels)
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  pdl_forget();
  return launch_maybe_pdl(true, kern, grid, block, smem, st, static_cast<Args&&>(args)...);
}
// the scan kernels (pdl_wait only at their end): programmatic only directly behind srl_philox_perm on the same stream
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl_scan(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                   Args&&... args) {
  const bool programmatic = pdl_take_perm(st);
  const cudaError_t e = launch_maybe_pdl(programmatic, kern, grid, block, smem, st, static_cast<Args&&>(args)...);
  if (!programmatic) pdl_note_scan(st);  // a permutation launched next on this stream may start beside this scan
  return e;
}

// Lets kernel KERN use up to `bytes` of dynamic shared memory on the current device.  The driver is asked once per device
// (one flag table per kernel, not per signature), so later launches -- stream capture included -- cost nothing.
template <auto KERN>
inline int opt_in_smem(size_t bytes) {
  static bool opted_in[64] = {};
  int dev = 0;
  SRL_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && !opted_in[dev]) {
    SRL_CUDA(cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
    opted_in[dev] = true;
  }
  return SRL_OK;
}

// ---- debug timeline (profiles/microbench/timeline.py; library built with -DSRL_TIMELINE, never the product build) ------
// One record per (kernel, CTA, slot): %globaltimer (ns, common to all SMs) and the SM's clock64.  The buffer pointer is a
// per-translation-unit device symbol set through the TU's own exported setter; a null pointer switches the stamps off.
#ifdef SRL_TIMELINE
namespace tl {
struct Rec {
  unsigned long long gt, clk;
};
constexpr int kCtas = 2048, kSlots = 16;
static __device__ Rec* g_buf;
__device__ __forceinline__ void stamp(int kernel, int cta, int slot) {
  Rec* b = g_buf;
  if (b != nullptr && cta < kCtas) {
    // reading %globaltimer costs ~250 cycles: only a CTA's entry stamp (slot 0) carries it; every other stamp is the SM's
    // cycle counter alone (the host places it on the global axis through the entry stamp of the same CTA)
    unsigned long long g = 0;
    if (slot == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
    Rec r;
    r.gt = g;
    r.clk = static_cast<unsigned long long>(clock64());
    b[(static_cast<size_t>(kernel) * kCtas + cta) * kSlots + slot] = r;
  }
}
}  // namespace tl
#define SRL_TL(kernel, cta, slot) ::srl::tl::stamp(kernel, cta, slot)
#define SRL_TL_SETTER(name)                                                                                  \
  extern "C" int name(void* p) {                                                                             \
    return cudaMemcpyToSymbol(::srl::tl::g_buf, &p, sizeof(p)) == cudaSuccess ? 0 : 1;                      \
  }
#else
#define SRL_TL(kernel, cta, slot) ((void)0)
#define SRL_TL_SETTER(name)
#endif

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

#endif  // __CUDACC__
}  // namespace srl
