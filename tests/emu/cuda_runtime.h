// TEST INFRASTRUCTURE ONLY -- a functional CPU emulation of the small part of the CUDA programming model that the
// kernels of libd3h_tets.so use, so that their LOGIC (index arithmetic, scans, sorts, table look-ups, float op order)
// can be exercised by the parity tests on a machine without a GPU.  The product never builds or loads this:
// d3human-code_b200/build.py compiles the kernels with nvcc for sm_100a only; tests/emu/build_emu.py compiles the very
// same .cu files with g++ against THIS header (it shadows <cuda_runtime.h>) into tests/emu/_build/, and only
// tests/test_emu_parity.py loads the result.
//
// Model: one OS thread.  Every CUDA thread of a block is a fibre (ucontext); blocks run one after the other.  A fibre
// runs until it reaches a block barrier or a warp collective, where it yields to the scheduler; the collective completes
// when every lane named in its mask has arrived.  There is no real concurrency, so atomics are plain read-modify-writes
// and memory ordering is sequential: data races and missing fences are NOT detected, performance means nothing.
// Two things a GPU does are imitated to make order / initialisation bugs visible: __shared__ variables live in one ELF
// section that is filled with 0xCB before every block (a fresh CTA's shared memory is arbitrary), and the schedule can be
// shuffled (D3H_EMU_SHUFFLE / d3h_emu_set_shuffle: random block order, random start and direction of every thread sweep).
#pragma once
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <type_traits>

#define D3H_CPU_EMU 1
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __restrict__
#define __launch_bounds__(...)
// every __shared__ variable lands in one ELF section so that the scheduler can poison it before each block runs
#define __shared__ static __attribute__((section("emu_shared")))
#define __constant__
#define __grid_constant__
#define __align__(n) __attribute__((aligned(n)))

// ---- vector types -----------------------------------------------------------------------------------------------
struct dim3 { unsigned x, y, z; dim3(unsigned a = 1, unsigned b = 1, unsigned c = 1) : x(a), y(b), z(c) {} };
struct alignas(8) int2 { int x, y; };
struct alignas(16) int4 { int x, y, z, w; };
struct alignas(8) uint2 { unsigned x, y; };
struct alignas(16) uint4 { unsigned x, y, z, w; };
struct alignas(8) float2 { float x, y; };
struct float3 { float x, y, z; };
struct alignas(16) float4 { float x, y, z, w; };
struct alignas(16) longlong2 { long long x, y; };
static inline int2 make_int2(int a, int b) { return {a, b}; }
static inline int4 make_int4(int a, int b, int c, int d) { return {a, b, c, d}; }
static inline uint2 make_uint2(unsigned a, unsigned b) { return {a, b}; }
static inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { return {a, b, c, d}; }
static inline float2 make_float2(float a, float b) { return {a, b}; }
static inline float3 make_float3(float a, float b, float c) { return {a, b, c}; }
static inline float4 make_float4(float a, float b, float c, float d) { return {a, b, c, d}; }

// ---- scheduler interface (tests/emu/emu_core.cpp) ------------------------------------------------------------------
namespace emu {
struct Idx { unsigned x, y, z; };
extern Idx g_threadIdx, g_blockIdx, g_blockDim, g_gridDim;
void run_grid(dim3 grid, dim3 block, const std::function<void()>& body, size_t dyn_smem_bytes = 0);
void block_barrier();
// warp collective: every lane of `mask` contributes `v`; returns the contributions of all 32 lanes (undefined for lanes
// outside the mask) through `out`
void warp_exchange(unsigned mask, unsigned long long v, unsigned long long out[32]);
unsigned long long now_ns();
void set_shuffle(unsigned long long seed);
void warp_sync_release();
void warp_sync_acquire();
// dynamic shared memory of the running block (1024-byte aligned, poisoned with 0xCB before every block) and its size
unsigned char* dyn_smem();
size_t dyn_smem_bytes();
size_t cvta_generic_to_shared(const void* p);
// the asynchronous part of sm_100 that csrc/d3h_mlp.cu uses: mbarriers, bulk copies global -> shared, tensor memory and
// tcgen05 (emu_core.cpp, written from the PTX ISA's definitions)
void mbar_init(uint64_t* bar, unsigned count);
void mbar_arrive(uint64_t* bar);
void mbar_arrive_expect_tx(uint64_t* bar, unsigned bytes);
void mbar_wait(uint64_t* bar, unsigned parity);
void bulk_copy_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar);
void tmem_alloc(uint32_t* dst, unsigned cols);
void tmem_dealloc(uint32_t taddr, unsigned cols);
void mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, unsigned accumulate);
void mma_commit(uint64_t* bar);
void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]);
// launches: the runtime's error of the last launch, and the dynamic shared memory limit a kernel was given
int take_last_error();
void set_last_error(int e);
int func_max_dynamic_smem(const void* f);
void set_func_max_dynamic_smem(const void* f, int bytes);
}  // namespace emu
// the built-in variables are plain globals (references): struct members named gridDim / blockDim keep working
static emu::Idx& threadIdx = emu::g_threadIdx;
static emu::Idx& blockIdx = emu::g_blockIdx;
static emu::Idx& blockDim = emu::g_blockDim;
static emu::Idx& gridDim = emu::g_gridDim;

// ---- synchronisation ---------------------------------------------------------------------------------------------
static inline void __syncthreads() { emu::block_barrier(); }
static inline void __threadfence() {}
static inline void __threadfence_system() {}
static inline void __threadfence_block() {}
static inline unsigned emu_lane() { return emu::g_threadIdx.x & 31u; }
static inline void __syncwarp(unsigned mask = 0xffffffffu) {  // rendezvous + memory ordering among the named lanes
  unsigned long long o[32];
  emu::warp_sync_release();
  emu::warp_exchange(mask, 0, o);
  emu::warp_sync_acquire();
}
static inline unsigned __ballot_sync(unsigned mask, int pred) {
  unsigned long long o[32];
  emu::warp_exchange(mask, pred ? 1ull : 0ull, o);
  unsigned r = 0;
  for (int l = 0; l < 32; ++l)
    if (((mask >> l) & 1u) && o[l]) r |= 1u << l;
  return r;
}
static inline int __any_sync(unsigned mask, int pred) { return __ballot_sync(mask, pred) != 0u; }
static inline int __all_sync(unsigned mask, int pred) { return __ballot_sync(mask, pred) == mask; }
template <typename T>
static inline unsigned long long emu_bits(T v) {
  static_assert(sizeof(T) <= 8, "shuffle of a wide type");
  unsigned long long b = 0;
  memcpy(&b, &v, sizeof(T));
  return b;
}
template <typename T>
static inline T emu_unbits(unsigned long long b) {
  T v;
  memcpy(&v, &b, sizeof(T));
  return v;
}
template <typename T>
static inline T __shfl_sync(unsigned mask, T v, int src, int width = 32) {
  (void)width;
  unsigned long long o[32];
  emu::warp_exchange(mask, emu_bits(v), o);
  return emu_unbits<T>(o[src & 31]);
}
template <typename T>
static inline T __shfl_up_sync(unsigned mask, T v, unsigned delta, int width = 32) {
  (void)width;
  unsigned long long o[32];
  emu::warp_exchange(mask, emu_bits(v), o);
  const int src = (int)emu_lane() - (int)delta;
  return src < 0 ? v : emu_unbits<T>(o[src]);
}
template <typename T>
static inline T __shfl_down_sync(unsigned mask, T v, unsigned delta, int width = 32) {
  (void)width;
  unsigned long long o[32];
  emu::warp_exchange(mask, emu_bits(v), o);
  const int src = (int)emu_lane() + (int)delta;
  return src > 31 ? v : emu_unbits<T>(o[src]);
}
template <typename T>
static inline T __shfl_xor_sync(unsigned mask, T v, int lane_mask, int width = 32) {
  (void)width;
  unsigned long long o[32];
  emu::warp_exchange(mask, emu_bits(v), o);
  return emu_unbits<T>(o[(emu_lane() ^ (unsigned)lane_mask) & 31]);
}
template <typename T>
static inline unsigned __match_any_sync(unsigned mask, T v) {
  unsigned long long o[32];
  const unsigned long long mine = emu_bits(v);
  emu::warp_exchange(mask, mine, o);
  unsigned r = 0;
  for (int l = 0; l < 32; ++l)
    if (((mask >> l) & 1u) && o[l] == mine) r |= 1u << l;
  return r;
}

// ---- integer / float intrinsics ----------------------------------------------------------------------------------
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __ffs(int v) { return __builtin_ffs(v); }
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned n) {
  return (unsigned)(((((unsigned long long)hi) << 32) | lo) >> (n & 31u));
}
static inline unsigned __fns(unsigned mask, unsigned base, int offset) {  // offset-th set bit at or above `base`
  if (offset <= 0) return 0xffffffffu;  // (negative offsets search downwards; not used by these kernels)
  int seen = 0;
  for (unsigned b = base; b < 32; ++b)
    if ((mask >> b) & 1u)
      if (++seen == offset) return b;
  return 0xffffffffu;
}
static inline float __fadd_rn(float a, float b) { volatile float r = a + b; return r; }
static inline float __fsub_rn(float a, float b) { volatile float r = a - b; return r; }
static inline float __fmul_rn(float a, float b) { volatile float r = a * b; return r; }
static inline float __fdiv_rn(float a, float b) { volatile float r = a / b; return r; }
static inline float __fmaf_rn(float a, float b, float c) { return fmaf(a, b, c); }
static inline float __fsqrt_rn(float a) { return sqrtf(a); }
static inline float __uint_as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }
static inline unsigned __float_as_uint(float f) { unsigned u; memcpy(&u, &f, 4); return u; }
// the fast intrinsics as the GPU evaluates them: __expf(x) = ex2.approx(x * log2(e)), __logf(x) = lg2.approx(x) * ln(2),
// with the multiplications rounded to fp32 (ex2 / lg2 themselves are within 2 ulp; the libm functions stand in for them)
// (glibc declares functions of these names itself: the intrinsics are macros)
static inline float emu_expf(float x) { volatile float t = x * 1.44269504088896341f; return exp2f(t); }
static inline float emu_logf(float x) { volatile float t = log2f(x); return t * 0.693147180559945309f; }
#define __expf(x) emu_expf(x)
#define __logf(x) emu_logf(x)
static inline size_t __cvta_generic_to_shared(const void* p) { return emu::cvta_generic_to_shared(p); }
template <typename T> static inline T __ldg(const T* p) { return *p; }
template <typename T> static inline T emu_load_relaxed(const T* p);
template <typename T> static inline T __ldcg(const T* p) { return emu_load_relaxed(p); }  // L2 loads: may watch atomics
template <typename T> static inline T __ldcs(const T* p) { return emu_load_relaxed(p); }
static inline int min(int a, int b) { return a < b ? a : b; }
static inline int max(int a, int b) { return a > b ? a : b; }
static inline unsigned min(unsigned a, unsigned b) { return a < b ? a : b; }
static inline unsigned max(unsigned a, unsigned b) { return a > b ? a : b; }
static inline long min(long a, long b) { return a < b ? a : b; }   // int64_t is long on LP64: min(int64_t, int64_t)
static inline long max(long a, long b) { return a > b ? a : b; }
static inline long long min(long long a, long long b) { return a < b ? a : b; }
static inline long long max(long long a, long long b) { return a > b ? a : b; }

// ---- atomics ---------------------------------------------------------------------------------------------------------
// Default build: no concurrency, plain read-modify-writes.  EMU_TSAN build: real seq_cst atomics, so that ThreadSanitizer
// treats them as synchronisation (ticket / last-block patterns) and does not report the atomic accesses themselves.
#ifdef EMU_TSAN
template <typename T> static inline T emu_rmw_add(T* p, T v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
static inline float emu_rmw_add(float* p, float v) {
  unsigned* u = reinterpret_cast<unsigned*>(p);
  unsigned old = __atomic_load_n(u, __ATOMIC_RELAXED), want;
  float f;
  do {
    memcpy(&f, &old, 4);
    f += v;
    memcpy(&want, &f, 4);
  } while (!__atomic_compare_exchange_n(u, &old, want, false, __ATOMIC_SEQ_CST, __ATOMIC_RELAXED));
  memcpy(&f, &old, 4);
  return f;
}
template <typename T> static inline T emu_load_relaxed(const T* p) {
  if constexpr (sizeof(T) == 4 || sizeof(T) == 8) {
    typedef typename std::conditional<sizeof(T) == 4, unsigned, unsigned long long>::type U;
    U u = __atomic_load_n(reinterpret_cast<const U*>(p), __ATOMIC_RELAXED);
    T r;
    memcpy(&r, &u, sizeof(T));
    return r;
  } else {
    return *p;
  }
}
template <typename T> static inline void emu_store_relaxed(T* p, T v) {
  typedef typename std::conditional<sizeof(T) == 4, unsigned, unsigned long long>::type U;
  U u;
  memcpy(&u, &v, sizeof(T));
  __atomic_store_n(reinterpret_cast<U*>(p), u, __ATOMIC_RELAXED);
}
static inline unsigned atomicOr(unsigned* p, unsigned v) { return __atomic_fetch_or(p, v, __ATOMIC_SEQ_CST); }
static inline unsigned atomicSub(unsigned* p, unsigned v) { return __atomic_fetch_sub(p, v, __ATOMIC_SEQ_CST); }
static inline unsigned long long atomicCAS(unsigned long long* p, unsigned long long cmp, unsigned long long v) {
  __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST);
  return cmp;
}
static inline unsigned atomicCAS(unsigned* p, unsigned cmp, unsigned v) {
  __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST);
  return cmp;
}
static inline int atomicCAS(int* p, int cmp, int v) {
  __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST);
  return cmp;
}
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) {
  unsigned long long old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (old < v && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_SEQ_CST, __ATOMIC_RELAXED)) {}
  return old;
}
#else
template <typename T> static inline T emu_rmw_add(T* p, T v) { T o = *p; *p = o + v; return o; }
template <typename T> static inline T emu_load_relaxed(const T* p) { return *p; }
template <typename T> static inline void emu_store_relaxed(T* p, T v) { *p = v; }
static inline unsigned atomicOr(unsigned* p, unsigned v) { unsigned o = *p; *p = o | v; return o; }
static inline unsigned atomicSub(unsigned* p, unsigned v) { unsigned o = *p; *p = o - v; return o; }
static inline unsigned long long atomicCAS(unsigned long long* p, unsigned long long cmp, unsigned long long v) {
  unsigned long long o = *p;
  if (o == cmp) *p = v;
  return o;
}
static inline unsigned atomicCAS(unsigned* p, unsigned cmp, unsigned v) {
  unsigned o = *p;
  if (o == cmp) *p = v;
  return o;
}
static inline int atomicCAS(int* p, int cmp, int v) {
  int o = *p;
  if (o == cmp) *p = v;
  return o;
}
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) {
  unsigned long long o = *p;
  if (v > o) *p = v;
  return o;
}
#endif
static inline unsigned atomicAdd(unsigned* p, unsigned v) { return emu_rmw_add(p, v); }
static inline int atomicAdd(int* p, int v) { return emu_rmw_add(p, v); }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { return emu_rmw_add(p, v); }
static inline float atomicAdd(float* p, float v) { return emu_rmw_add(p, v); }
static inline float4 atomicAdd(float4* p, float4 v) {  // the hardware's vector atomic is four independent scalar adds
  float4 o;
  o.x = emu_rmw_add(&p->x, v.x); o.y = emu_rmw_add(&p->y, v.y); o.z = emu_rmw_add(&p->z, v.z); o.w = emu_rmw_add(&p->w, v.w);
  return o;
}

// ---- runtime API: one device, memory = host memory, streams / events are no-ops, graphs unsupported -------------------
typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorInvalidValue = 1, cudaErrorNotSupported = 801 };
typedef struct emu_stream_s* cudaStream_t;
typedef struct emu_event_s* cudaEvent_t;
typedef struct emu_graph_s* cudaGraph_t;
typedef struct emu_graphexec_s* cudaGraphExec_t;
typedef struct emu_graphnode_s* cudaGraphNode_t;
enum cudaStreamCaptureStatus { cudaStreamCaptureStatusNone = 0 };
enum cudaStreamCaptureMode { cudaStreamCaptureModeThreadLocal = 1 };
enum cudaGraphNodeType { cudaGraphNodeTypeKernel = 0 };
enum cudaMemcpyKind { cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3 };
enum cudaMemoryType { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2 };
enum cudaDeviceAttr { cudaDevAttrMultiProcessorCount = 16 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2 };
enum { cudaGraphInstantiateFlagUseNodePriority = 8 };
struct cudaPointerAttributes { cudaMemoryType type; int device; void* devicePointer; void* hostPointer; };
struct cudaKernelNodeParams { void* func; dim3 gridDim, blockDim; unsigned sharedMemBytes; void** kernelParams; void** extra; };
enum cudaLaunchAttributeID { cudaLaunchAttributePriority = 8 };
struct cudaLaunchAttributeValue { int priority; };
struct cudaLaunchAttribute { cudaLaunchAttributeID id; cudaLaunchAttributeValue val; };
struct cudaLaunchConfig_t { dim3 gridDim, blockDim; size_t dynamicSmemBytes; cudaStream_t stream; cudaLaunchAttribute* attrs; unsigned numAttrs; };

static inline const char* cudaGetErrorString(cudaError_t e) {
  return e == 0 ? "no error" : (e == cudaErrorInvalidValue ? "invalid argument" : "emulation: unsupported");
}
static inline cudaError_t cudaGetLastError() { return emu::take_last_error(); }
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return cudaSuccess; }
static inline cudaError_t cudaDeviceGetAttribute(int* v, cudaDeviceAttr, int) { *v = 4; return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
static inline cudaError_t cudaDeviceGetStreamPriorityRange(int* lo, int* hi) { *lo = 0; *hi = -5; return cudaSuccess; }
static inline cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessor(int* n, const void*, int, size_t) { *n = 2; return cudaSuccess; }
template <typename F> static inline cudaError_t cudaFuncSetAttribute(F f, cudaFuncAttribute a, int v) {
  if (a == cudaFuncAttributeMaxDynamicSharedMemorySize) emu::set_func_max_dynamic_smem(reinterpret_cast<const void*>(f), v);
  return cudaSuccess;
}
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = nullptr; return cudaSuccess; }
static inline cudaError_t cudaStreamCreateWithPriority(cudaStream_t* s, unsigned, int) { *s = nullptr; return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaStreamIsCapturing(cudaStream_t, cudaStreamCaptureStatus* s) { *s = cudaStreamCaptureStatusNone; return cudaSuccess; }
static inline cudaError_t cudaStreamBeginCapture(cudaStream_t, cudaStreamCaptureMode) { return cudaErrorNotSupported; }
static inline cudaError_t cudaStreamEndCapture(cudaStream_t, cudaGraph_t*) { return cudaErrorNotSupported; }
static inline cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = nullptr; return cudaSuccess; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = nullptr; return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return cudaSuccess; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaGraphGetNodes(cudaGraph_t, cudaGraphNode_t*, size_t* n) { *n = 0; return cudaErrorNotSupported; }
static inline cudaError_t cudaGraphNodeGetType(cudaGraphNode_t, cudaGraphNodeType*) { return cudaErrorNotSupported; }
static inline cudaError_t cudaGraphKernelNodeGetParams(cudaGraphNode_t, cudaKernelNodeParams*) { return cudaErrorNotSupported; }
static inline cudaError_t cudaGraphInstantiate(cudaGraphExec_t*, cudaGraph_t, unsigned long long) { return cudaErrorNotSupported; }
static inline cudaError_t cudaGraphInstantiateWithFlags(cudaGraphExec_t*, cudaGraph_t, unsigned long long) { return cudaErrorNotSupported; }
static inline cudaError_t cudaGraphExecKernelNodeSetParams(cudaGraphExec_t, cudaGraphNode_t, const cudaKernelNodeParams*) { return cudaErrorNotSupported; }
static inline cudaError_t cudaGraphLaunch(cudaGraphExec_t, cudaStream_t) { return cudaErrorNotSupported; }
static inline cudaError_t cudaGraphDestroy(cudaGraph_t) { return cudaSuccess; }
static inline cudaError_t cudaGraphExecDestroy(cudaGraphExec_t) { return cudaSuccess; }
static inline cudaError_t cudaPointerGetAttributes(cudaPointerAttributes* a, const void* p) {
  a->type = cudaMemoryTypeHost; a->device = 0; a->devicePointer = const_cast<void*>(p); a->hostPointer = const_cast<void*>(p);
  return cudaSuccess;
}
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t) { memmove(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t) { memset(d, v, n); return cudaSuccess; }
template <typename T> static inline cudaError_t cudaMalloc(T** p, size_t n) { *p = (T*)malloc(n); return *p ? cudaSuccess : 2; }
static inline cudaError_t cudaFree(void* p) { free(p); return cudaSuccess; }

template <typename... KArgs, typename... Args>
static inline cudaError_t cudaLaunchKernelEx(const cudaLaunchConfig_t* cfg, void (*kernel)(KArgs...), Args&&... args) {
  // more than 48 KB of dynamic shared memory needs the kernel's cudaFuncAttributeMaxDynamicSharedMemorySize first: the
  // launch fails with cudaErrorInvalidValue (reported by the next cudaGetLastError) and nothing runs
  if (cfg->dynamicSmemBytes > 48u * 1024u &&
      (int64_t)cfg->dynamicSmemBytes > (int64_t)emu::func_max_dynamic_smem(reinterpret_cast<const void*>(kernel))) {
    emu::set_last_error(cudaErrorInvalidValue);
    return cudaErrorInvalidValue;
  }
  auto body = [=]() { kernel(args...); };
  emu::run_grid(cfg->gridDim, cfg->blockDim, body, cfg->dynamicSmemBytes);
  return cudaSuccess;
}
// kernel<<<grid, block, smem, stream>>>(args) of the product sources, spelled EMU_LAUNCH(kernel, grid, block, smem, stream)(args)
template <typename... KArgs>
struct EmuLaunch {
  void (*kernel)(KArgs...);
  cudaLaunchConfig_t cfg;
  template <typename... Args>
  void operator()(Args&&... args) const { cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...); }
};
template <typename... KArgs>
static inline EmuLaunch<KArgs...> emu_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream) {
  EmuLaunch<KArgs...> l;
  memset(&l.cfg, 0, sizeof(l.cfg));
  l.kernel = kernel;
  l.cfg.gridDim = grid;
  l.cfg.blockDim = block;
  l.cfg.dynamicSmemBytes = smem;
  l.cfg.stream = stream;
  return l;
}
