// SDF field query (SURVEY 8f row 3): positional encoding + the MLP of geometry/mlp.py:9-45 on the tensor cores.
//
// Every GEMM of the forward and backward pass is one of two kernels built on the same core:
//
//   * activations are fp32 in global memory; producer warps load 32-column (128-byte) slices with coalesced 16-byte loads
//     (the loads of slice i+1 are in flight while the tensor core works on slice i), split every value into hi (low 13
//     mantissa bits cleared = exactly representable in TF32) and lo = x - hi, and store both into shared memory in the
//     canonical K-major SWIZZLE_128B layout of the tcgen05 shared-memory descriptors (8-row x 128-byte atoms, 16-byte
//     chunk c of row r at chunk position c ^ (r % 8));
//   * weights are split and laid out in exactly that shared-memory image ONCE per call (mlp_pack_weight_kernel): a slice
//     of the weight operand is then one 64 KB bulk copy global -> shared (cp.async.bulk + mbarrier complete_tx, issued
//     by the MMA thread), no thread touches it;
//   * one 96 KB stage per CTA and two CTAs per SM (2 x 256 tensor-memory columns): while one CTA waits for its
//     operands or runs its epilogue the other one keeps the tensor core busy;
//   * one thread issues tcgen05.mma.cta_group::1.kind::tf32 (M = 128, N <= 256, K = 8 per instruction) three times per
//     k-step: hi.hi + lo.hi + hi.lo -- the 3xTF32 scheme, fp32-level accuracy at tensor-core speed -- accumulating in
//     tensor memory; tcgen05.commit on an mbarrier hands the shared-memory stage back to the producers;
//   * after the last k-step the same warps read the accumulator with tcgen05.ld (32 lanes x 32 columns per instruction),
//     apply bias / Softplus(beta=100) / the activation's derivative, and store fp32 rows.
//
// mlp_linear_kernel : c = f(a w^T + bias), tile = 128 rows of a x all N <= 256 output columns, K walked in 32-column slices.
//                     Two more epilogues serve the second derivative (the eikonal term): tangent (z-dot and a-dot =
//                     z-dot * softplus') and adjoint (input gradient * softplus' + the softplus'' term of delta and z-dot).
// mlp_wgrad_kernel  : dw += dz^T a, the contraction runs over the POINTS: the producers transpose 32-point slices of dz
//                     and a on their way into shared memory (lanes <-> points, conflict-free), every CTA owns a point
//                     range and 128 of dz's columns and adds its partial result to dw with red.global.add.f32.
//
// No CPU emulation of this file (tests/emu does not list it): tensor-core instructions have no stand-in there; the
// parity tests of this stage are GPU-only and compare against oracle/mlp_oracle.py (float64).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/d3h_mlp.h"
#include "d3h_internal.cuh"

namespace d3h {
namespace mlp {

constexpr int kTileM = 128;          // rows of the accumulator (tensor-memory lanes)
constexpr int kSliceK = 32;          // fp32 values per shared-memory row: 128 bytes = one swizzle row
constexpr int kProducerWarps = 8;
constexpr int kThreads = (kProducerWarps + 1) * 32;   // + the MMA / tensor-memory warp
constexpr int kCtasPerSm = 2;
constexpr float kBeta = 100.f, kThreshold = 20.f;     // nn.Softplus(beta=100), default threshold (mlp.py:16)

// ---------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// generic-proxy stores to shared memory -> visible to the async proxy (the tensor core reads through it)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bulk copy global -> shared through the async proxy (TMA, no tensor map: one contiguous piece); completion is counted
// in bytes on the mbarrier
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {     // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, one thread
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier once every MMA issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive columns of the accumulator -> 32 registers per thread (lane = row of this warp's quarter)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Shared-memory matrix descriptor of a K-major SWIZZLE_128B tile (rows of 128 bytes, 8-row atoms 1024 bytes apart):
// start address and offsets in 16-byte units; leading byte offset 1 (unused with swizzle), stride byte offset 64,
// version 1 (sm_100), layout type 2 = SWIZZLE_128B.  The tile base must be 1024-byte aligned (base_offset = 0).
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)64 << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor of kind::tf32: fp32 accumulator (bits 4-5 = 1), A and B TF32 (format 2 at bits 7-9 / 10-12),
// both K-major (bits 15, 16 = 0), N / 8 at bits 17-22, M / 16 at bits 24-28.
__device__ __forceinline__ uint32_t instr_desc(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// byte offset of (row r, 16-byte chunk c) inside a swizzled tile
__device__ __forceinline__ uint32_t swz(int r, int c) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// Softplus(beta = 100): torch computes (x*beta > threshold) ? x : log1p(exp(x*beta)) / beta.  Most pre-activations are far
// from zero on the 1/beta scale, so the common cases cost no or one transcendental; the fast intrinsics are accurate to
// ~1e-6 relative for |t| <= 20 and the result is divided by beta (absolute error < 1e-8).
__device__ __forceinline__ float softplus100(float z) {
  const float t = z * kBeta;
  if (t > kThreshold) return z;
  const float e = __expf(t);
  const float l = e < 2.44140625e-4f ? e * (1.f - 0.5f * e) : __logf(1.f + e);     // log1p(e); 2^-12: e^3/3 < 5e-12
  return l * (1.f / kBeta);
}
// d softplus / dz from the OUTPUT y = softplus(z): sigmoid(beta z) = 1 - exp(-beta y)  (exactly 1 - e^-20.. in the linear
// branch, where torch's backward returns 1: the difference is < 2.1e-9)
__device__ __forceinline__ float softplus100_grad_from_output(float y) { return 1.f - __expf(-kBeta * y); }
// softplus''(z) / softplus'(z) = beta (1 - softplus'(z)) = beta exp(-beta y), zero past the threshold as in torch's
// softplus_double_backward: the factor that turns delta = lambda softplus'(z) into lambda softplus''(z)
__device__ __forceinline__ float softplus100_curv_from_output(float y) {
  return kBeta * y <= kThreshold ? kBeta * __expf(-kBeta * y) : 0.f;
}

struct StageBuffers {       // byte offsets inside the dynamic shared memory of one stage
  uint32_t a_hi, a_lo, b_hi, b_lo, bytes;
};
__host__ __device__ inline StageBuffers stage_layout(int rows_b) {
  StageBuffers s;
  s.a_hi = 0;
  s.a_lo = kTileM * 128;
  s.b_hi = 2 * kTileM * 128;
  s.b_lo = s.b_hi + rows_b * 128;
  s.bytes = s.b_lo + rows_b * 128;
  return s;
}

// The 3 x 4 instructions of one 32-wide slice: lo.hi + hi.lo + hi.hi (small terms first), K = 8 per instruction.
__device__ __forceinline__ void issue_slice(uint32_t base, const StageBuffers& sl, uint32_t tmem_d, uint32_t idesc, bool first) {
  const uint64_t dah = smem_desc(base + sl.a_hi), dal = smem_desc(base + sl.a_lo);
  const uint64_t dbh = smem_desc(base + sl.b_hi), dbl = smem_desc(base + sl.b_lo);
#pragma unroll
  for (int ks = 0; ks < kSliceK / 8; ++ks) {
    const uint64_t adv = (uint64_t)(ks * 2);     // 8 TF32 values = 32 bytes = 2 units of the start-address field
    umma_tf32(tmem_d, dal + adv, dbh + adv, idesc, (!first || ks > 0) ? 1u : 0u);
    umma_tf32(tmem_d, dah + adv, dbl + adv, idesc, 1u);
    umma_tf32(tmem_d, dah + adv, dbh + adv, idesc, 1u);
  }
}

// Weight operand in its shared-memory image: for every 32-column slice s of B (n_pad rows x k_pad columns, zero outside
// the valid part) a block of n_pad x 128 bytes of hi values followed by the same of lo values, both swizzled.
//   B[n][k] = transpose ? w[(row0 + k) ldw + col0 + n] : w[(row0 + n) ldw + col0 + k],  n < n_valid, k < k_valid
struct PackArgs {
  const float* w; int64_t ldw;
  float* out;
  int n_valid, k_valid, transpose, row0, col0, n_pad, k_pad;
};
__global__ void __launch_bounds__(256) mlp_pack_weight_kernel(PackArgs g) {
  const int chunks = g.k_pad / 4;                      // 16-byte chunks per row of B
  const int64_t total = (int64_t)g.n_pad * chunks;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i / chunks), ch = (int)(i % chunks);
    float x[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = 4 * ch + u;
      x[u] = 0.f;
      if (n < g.n_valid && k < g.k_valid)
        x[u] = g.transpose ? g.w[(int64_t)(g.row0 + k) * g.ldw + g.col0 + n] : g.w[(int64_t)(g.row0 + n) * g.ldw + g.col0 + k];
    }
    const float4 h = make_float4(tf32_hi(x[0]), tf32_hi(x[1]), tf32_hi(x[2]), tf32_hi(x[3]));
    const float4 l = make_float4(x[0] - h.x, x[1] - h.y, x[2] - h.z, x[3] - h.w);
    const int s = ch / 8, c = ch % 8;
    uint8_t* blk = reinterpret_cast<uint8_t*>(g.out) + (size_t)s * 2 * g.n_pad * 128;
    *reinterpret_cast<float4*>(blk + swz(n, c)) = h;
    *reinterpret_cast<float4*>(blk + (size_t)g.n_pad * 128 + swz(n, c)) = l;
  }
}

struct LinearArgs {
  const float* a; int64_t lda;
  const float* wp;           // packed weight image (mlp_pack_weight_kernel)
  const float* bias;
  const float* y; int64_t ldy;
  float* c; int64_t ldc;
  int64_t m;
  int k, n, mode;
  float* c2; int64_t ldc2;           // kEpiTangent: z-dot
  const float* d; int64_t ldd;       // kEpiAdjoint: delta and z-dot of the layer whose output is y
  const float* zd; int64_t ldzd;
};

// Epilogues of mlp_linear_kernel.  kEpiFirstOrder: `mode` 0 / 1 / 2 of d3h_mlp_linear.  The other two serve the second
// derivative (d3h_mlp_linear_tangent / d3h_mlp_linear_adjoint): tangent c2 = acc, c = acc * softplus'(y); adjoint
// c = acc * softplus'(y) + beta [beta y <= 20] exp(-beta y) * d * zd.
constexpr int kEpiFirstOrder = 0, kEpiTangent = 1, kEpiAdjoint = 2;

// ---------------------------------------------------------------------------------------------- c = f(a w^T + bias)
template <int kEpi>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) mlp_linear_kernel(LinearArgs g) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t s_full, s_empty, s_done;
  __shared__ uint32_t s_tmem;
  const StageBuffers sl = stage_layout(g.n);
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const int64_t row0 = (int64_t)blockIdx.x * kTileM;
  const int n_slices = g.k / kSliceK;
  const uint32_t tmem_cols = g.n <= 64 ? 64u : (g.n <= 128 ? 128u : 256u);

  if (threadIdx.x == 0) {
    mbar_init(&s_full, kProducerWarps * 32 + 1);     // the producers + the thread that announces the bulk copy
    mbar_init(&s_empty, 1);
    mbar_init(&s_done, 1);
    fence_barrier_init();
  }
  if (warp == kProducerWarps) tmem_alloc(&s_tmem, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = s_tmem;

  if (warp < kProducerWarps) {
    // ---- producers: thread t owns 16-byte chunk (t & 7) of rows (t >> 3) + 32 i of the activation slice ----
    const int c = threadIdx.x & 7, r0 = threadIdx.x >> 3;
    const float* src[kTileM / 32];
#pragma unroll
    for (int i = 0; i < kTileM / 32; ++i) {
      const int64_t r = row0 + r0 + 32 * i;
      src[i] = r < g.m ? g.a + r * g.lda + 4 * c : nullptr;
    }
    // two slices of loads in flight: registers va (slice it) and vb (slice it + 1)
    float4 va[kTileM / 32], vb[kTileM / 32];
    auto load = [&](float4 (&v)[kTileM / 32], int slice) {
#pragma unroll
      for (int i = 0; i < kTileM / 32; ++i)
        v[i] = (src[i] && slice < n_slices) ? __ldg(reinterpret_cast<const float4*>(src[i] + slice * kSliceK)) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    auto publish = [&](const float4 (&v)[kTileM / 32], int it) {
      mbar_wait(&s_empty, (uint32_t)((it & 1) ^ 1));      // the MMAs of slice it - 1 have read the stage (fresh: passes)
#pragma unroll
      for (int i = 0; i < kTileM / 32; ++i) {
        const int r = r0 + 32 * i;
        const float4 h = make_float4(tf32_hi(v[i].x), tf32_hi(v[i].y), tf32_hi(v[i].z), tf32_hi(v[i].w));
        const float4 l = make_float4(v[i].x - h.x, v[i].y - h.y, v[i].z - h.z, v[i].w - h.w);
        *reinterpret_cast<float4*>(smem + sl.a_hi + swz(r, c)) = h;
        *reinterpret_cast<float4*>(smem + sl.a_lo + swz(r, c)) = l;
      }
      fence_proxy_async();
      mbar_arrive(&s_full);
    };
    load(va, 0);
    load(vb, 1);
    for (int it = 0; it < n_slices; it += 2) {
      publish(va, it);
      load(va, it + 2);                                   // in flight while the tensor core works on slices it, it + 1
      if (it + 1 < n_slices) {
        publish(vb, it + 1);
        load(vb, it + 3);
      }
    }
    // ---- epilogue: warp w reads lanes [32 (w & 3), +32) = rows of the tile, column half (w >> 2) ----
    mbar_wait(&s_done, 0u);
    tc_fence_after();
    const int q = warp & 3, half = warp >> 2;
    const int64_t r = row0 + 32 * q + lane;
    const int ncol_half = g.n / 2;                      // N % 64 == 0: each half is a whole number of 32-column loads
    for (int c0 = half * ncol_half; c0 < (half + 1) * ncol_half; c0 += 32) {
      float v[32];
      tmem_ld32(tmem_d + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, v);
      if (kEpi != kEpiFirstOrder && r < g.m) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 yy = __ldg(reinterpret_cast<const float4*>(g.y + r * g.ldy + c0 + j));
          const float4 acc = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          float4 o = make_float4(acc.x * softplus100_grad_from_output(yy.x), acc.y * softplus100_grad_from_output(yy.y),
                                 acc.z * softplus100_grad_from_output(yy.z), acc.w * softplus100_grad_from_output(yy.w));
          if (kEpi == kEpiTangent) {
            *reinterpret_cast<float4*>(g.c2 + r * g.ldc2 + c0 + j) = acc;
          } else {
            const float4 dd = __ldg(reinterpret_cast<const float4*>(g.d + r * g.ldd + c0 + j));
            const float4 zz = __ldg(reinterpret_cast<const float4*>(g.zd + r * g.ldzd + c0 + j));
            o.x += softplus100_curv_from_output(yy.x) * dd.x * zz.x; o.y += softplus100_curv_from_output(yy.y) * dd.y * zz.y;
            o.z += softplus100_curv_from_output(yy.z) * dd.z * zz.z; o.w += softplus100_curv_from_output(yy.w) * dd.w * zz.w;
          }
          *reinterpret_cast<float4*>(g.c + r * g.ldc + c0 + j) = o;
        }
      }
      if (kEpi == kEpiFirstOrder && r < g.m) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float o[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float z = v[j + u];
            if (g.bias != nullptr) z += __ldg(g.bias + c0 + j + u);
            o[u] = g.mode == 1 ? softplus100(z) : z;
          }
          if (g.mode == 2) {
            const float4 yy = __ldg(reinterpret_cast<const float4*>(g.y + r * g.ldy + c0 + j));
            o[0] *= softplus100_grad_from_output(yy.x); o[1] *= softplus100_grad_from_output(yy.y);
            o[2] *= softplus100_grad_from_output(yy.z); o[3] *= softplus100_grad_from_output(yy.w);
          }
          *reinterpret_cast<float4*>(g.c + r * g.ldc + c0 + j) = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    tc_fence_before();
  } else {
    // ---- one thread: announces and issues the bulk copy of the weight slice, then the MMAs of the slice ----
    if (lane == 0) {
      const uint32_t idesc = instr_desc(kTileM, g.n);
      const uint32_t wbytes = (uint32_t)(2 * g.n * 128);
      const uint32_t base = smem_u32(smem);
      for (int it = 0; it < n_slices; ++it) {
        mbar_wait(&s_empty, (uint32_t)((it & 1) ^ 1));
        mbar_expect_tx(&s_full, wbytes);
        bulk_copy_g2s(smem + sl.b_hi, reinterpret_cast<const uint8_t*>(g.wp) + (size_t)it * wbytes, wbytes, &s_full);
        mbar_wait(&s_full, (uint32_t)(it & 1));
        tc_fence_after();
        issue_slice(base, sl, tmem_d, idesc, it == 0);
        umma_commit(&s_empty);                        // the stage may be refilled once these have read it
        if (it == n_slices - 1) umma_commit(&s_done); // ... and the accumulator is complete
      }
    }
    __syncwarp();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == kProducerWarps) {
    tc_fence_after();
    tmem_dealloc(tmem_d, tmem_cols);
  }
}

struct WgradArgs {
  const float* dz; int64_t ldz;
  const float* a; int64_t lda;
  float* part;               // (ranges, n, k) partial products, one slab per point range (plain stores, summed afterwards)
  float* part_b;             // (ranges, n) partial column sums of dz, or nullptr
  int64_t m, points_per_cta;
  int n, k;
};

// ---------------------------------------------------------------------------------------------- dw += dz^T a
// grid = (point ranges, N / 128).  Accumulator: 128 columns of dz (lanes) x K columns of a; every CTA stores its partial
// product to its own slab of the workspace (65536 atomics per CTA on one 256 KB matrix were the bottleneck of the first
// version: 60 of 83 ms of the backward pass) and wgrad_reduce_kernel adds the slabs to dw.  Both operands are
// activations: the producers transpose 32-point slices on their way into shared memory -- lane = point of the slice
// (the k index of the MMA), warp w takes the 16-byte column groups w, w + 8, ... of that point's row, and the four values
// of a group go to four tile rows at k = lane (32 lanes -> 32 distinct words of one 128-byte row: no bank conflict).
__global__ void __launch_bounds__(kThreads, kCtasPerSm) mlp_wgrad_kernel(WgradArgs g) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t s_full, s_empty, s_done;
  __shared__ uint32_t s_tmem;
  const StageBuffers sl = stage_layout(g.k);
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const int64_t p_begin = (int64_t)blockIdx.x * g.points_per_cta;
  const int64_t p_end = min(g.m, p_begin + g.points_per_cta);
  const int ch0 = blockIdx.y * kTileM;
  const int64_t n_slices = p_end > p_begin ? (p_end - p_begin + kSliceK - 1) / kSliceK : 0;
  const uint32_t tmem_cols = g.k <= 64 ? 64u : (g.k <= 128 ? 128u : 256u);
  if (n_slices == 0) return;     // (whole CTA)

  if (threadIdx.x == 0) {
    mbar_init(&s_full, kProducerWarps * 32);
    mbar_init(&s_empty, 1);
    mbar_init(&s_done, 1);
    fence_barrier_init();
  }
  if (warp == kProducerWarps) tmem_alloc(&s_tmem, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = s_tmem;

  if (warp < kProducerWarps) {
    float bsum[4][4];              // bias gradient: this thread's share of sum_m dz[m, ch] for its 16 columns of dz
#pragma unroll
    for (int i = 0; i < 4; ++i) bsum[i][0] = bsum[i][1] = bsum[i][2] = bsum[i][3] = 0.f;
    const int kc = (int)lane >> 2, kw = ((int)lane & 3) * 4;       // 16-byte chunk and byte offset of k = lane in a row
    const uint32_t row_base = (uint32_t)((warp >> 1) * 1024);      // 8-row atom of this warp's first column group
    uint32_t off_u[4];                                             // row inside the atom + swizzled chunk + word, per value u
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int r7 = 4 * ((int)warp & 1) + u;
      off_u[u] = (uint32_t)(r7 * 128 + ((kc ^ r7) << 4) + kw);
    }
    const int a_groups = g.k / 4;                                   // 16-byte column groups of a row of a: 16 .. 64
    float4 vz[4], va[8];
    auto load_slice = [&](int64_t it) {
      const int64_t p = p_begin + it * kSliceK + lane;
      const bool live = p < p_end;
#pragma unroll
      for (int i = 0; i < 4; ++i)      // 128 columns of dz = 32 groups of 4: groups warp + 8 i
        vz[i] = live ? __ldg(reinterpret_cast<const float4*>(g.dz + p * g.ldz + ch0 + 4 * ((int)warp + 8 * i)))
                     : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {    // K columns of a: groups warp + 8 i
        const int f = (int)warp + 8 * i;
        va[i] = (live && f < a_groups) ? __ldg(reinterpret_cast<const float4*>(g.a + p * g.lda + 4 * f)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    load_slice(0);
    for (int64_t it = 0; it < n_slices; ++it) {
      mbar_wait(&s_empty, (uint32_t)((it & 1) ^ 1));
      // tile row of value u of column group f = warp + 8 i: r = 4 f + u, so r >> 3 = (warp >> 1) + 4 i and r & 7 = 4 (warp & 1) + u
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if ((int)warp + 8 * i >= a_groups) continue;
        const float x[4] = {va[i].x, va[i].y, va[i].z, va[i].w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float h = tf32_hi(x[u]);
          const uint32_t off = row_base + 4096u * i + off_u[u];
          *reinterpret_cast<float*>(smem + sl.b_hi + off) = h;
          *reinterpret_cast<float*>(smem + sl.b_lo + off) = x[u] - h;
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float x[4] = {vz[i].x, vz[i].y, vz[i].z, vz[i].w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float h = tf32_hi(x[u]);
          const uint32_t off = row_base + 4096u * i + off_u[u];
          *reinterpret_cast<float*>(smem + sl.a_hi + off) = h;
          *reinterpret_cast<float*>(smem + sl.a_lo + off) = x[u] - h;
          bsum[i][u] += x[u];
        }
      }
      fence_proxy_async();
      mbar_arrive(&s_full);
      if (it + 1 < n_slices) load_slice(it + 1);       // in flight while the tensor core works on slice `it`
    }
    if (g.part_b != nullptr) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float v = bsum[i][u];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
          if (lane == 0) g.part_b[(int64_t)blockIdx.x * g.n + ch0 + 4 * ((int)warp + 8 * i) + u] = v;
        }
    }
    // ---- epilogue: lanes of the accumulator = columns of dz, columns = columns of a ----
    mbar_wait(&s_done, 0u);
    tc_fence_after();
    const int q = warp & 3, half = warp >> 2;
    const int row = ch0 + 32 * q + (int)lane;             // row of dw
    const int ncol_half = g.k / 2;
    float* __restrict__ dst = g.part + ((int64_t)blockIdx.x * g.n + row) * g.k;
    for (int c0 = half * ncol_half; c0 < (half + 1) * ncol_half; c0 += 32) {
      float v[32];
      tmem_ld32(tmem_d + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, v);
#pragma unroll
      for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(dst + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    }
    tc_fence_before();
  } else {
    if (lane == 0) {
      const uint32_t idesc = instr_desc(kTileM, g.k);
      const uint32_t base = smem_u32(smem);
      for (int64_t it = 0; it < n_slices; ++it) {
        mbar_wait(&s_full, (uint32_t)(it & 1));
        tc_fence_after();
        issue_slice(base, sl, tmem_d, idesc, it == 0);
        umma_commit(&s_empty);
        if (it == n_slices - 1) umma_commit(&s_done);
      }
    }
    __syncwarp();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == kProducerWarps) {
    tc_fence_after();
    tmem_dealloc(tmem_d, tmem_cols);
  }
}

// dw[r][c] += sum over the point ranges of part[range][r][c]; db likewise.  One thread per output element, the slabs are
// read coalesced.
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ part, const float* __restrict__ part_b,
                                                           int ranges, int n, int k, float* __restrict__ dw, int64_t lddw,
                                                           float* __restrict__ db) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nk = (int64_t)n * k;
  if (i < nk) {
    float s = 0.f;
    for (int r = 0; r < ranges; ++r) s += part[(int64_t)r * nk + i];
    const int row = (int)(i / k), col = (int)(i % k);
    dw[(int64_t)row * lddw + col] += s;
  } else if (db != nullptr && i < nk + n) {
    const int c = (int)(i - nk);
    float s = 0.f;
    for (int r = 0; r < ranges; ++r) s += part_b[(int64_t)r * n + c];
    db[c] += s;
  }
}

// ---------------------------------------------------------------------------------------------- small kernels
__global__ void __launch_bounds__(256) embed_kernel(const float* __restrict__ x, int64_t m, int n_freq, float* __restrict__ out,
                                                    int64_t ld, int n_cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const float p[3] = {x[3 * i], x[3 * i + 1], x[3 * i + 2]};
  float* o = out + i * ld;
  o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
  float f = 1.f;                                   // freq_bands = 2 ** linspace(0, n_freq - 1, n_freq): exact powers of two
  for (int k = 0; k < n_freq; ++k, f *= 2.f) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const float a = f * p[d];
      o[3 + 6 * k + d] = sinf(a);
      o[6 + 6 * k + d] = cosf(a);
    }
  }
  for (int c = 3 * (2 * n_freq + 1); c < n_cols; ++c) o[c] = 0.f;
}

// The same with one thread per (point, group of four output columns): 16-byte stores, 16 lanes cover a 256-byte row.
// Needs n_cols % 4 == 0, ld % 4 == 0 and a 16-byte aligned `out` (the padded operand buffers of the GEMMs).
__global__ void __launch_bounds__(256) embed4_kernel(const float* __restrict__ x, int64_t m, int n_freq, float* __restrict__ out,
                                                     int64_t ld, int n_cols) {
  const int groups = n_cols / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m * groups) return;
  const int64_t pt = i / groups;
  const int g = (int)(i % groups);
  const int e = 3 * (2 * n_freq + 1);
  float o[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int c = 4 * g + u;
    float v = 0.f;
    if (c < 3) {
      v = x[3 * pt + c];
    } else if (c < e) {
      const int k = (c - 3) / 6, r = (c - 3) % 6;
      const float a = (float)(1 << k) * x[3 * pt + (r % 3)];
      v = r < 3 ? sinf(a) : cosf(a);
    }
    o[u] = v;
  }
  *reinterpret_cast<float4*>(out + pt * ld + 4 * g) = make_float4(o[0], o[1], o[2], o[3]);
}

__global__ void __launch_bounds__(256) embed_backward_kernel(const float* __restrict__ x, int64_t m, int n_freq,
                                                             const float* __restrict__ g_emb, int64_t ld,
                                                             float* __restrict__ g_x, int accumulate) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const float* ge = g_emb + i * ld;
  float f = 1.f;
  float acc[3] = {ge[0], ge[1], ge[2]};
  for (int k = 0; k < n_freq; ++k, f *= 2.f) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const float a = f * x[3 * i + d];
      acc[d] += f * (cosf(a) * ge[3 + 6 * k + d] - sinf(a) * ge[6 + 6 * k + d]);
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) g_x[3 * i + d] = accumulate ? g_x[3 * i + d] + acc[d] : acc[d];
}

// out[m, j] = a[m, :] . w[j, :] + bias[j]; one warp per row, d_out <= 8
__global__ void __launch_bounds__(256) head_kernel(const float* __restrict__ a, int64_t lda, int64_t m, int k,
                                                   const float* __restrict__ w, const float* __restrict__ bias, int d_out,
                                                   float* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const unsigned lane = threadIdx.x & 31u;
  if (row >= m) return;
  for (int j = 0; j < d_out; ++j) {
    float s = 0.f;
    for (int c = (int)lane; c < k; c += 32) s = fmaf(a[row * lda + c], __ldg(w + (int64_t)j * k + c), s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[row * d_out + j] = s + (bias ? bias[j] : 0.f);
  }
}

// dz = (g w) * softplus'(a), dw += g^T a, db += sum g in one sweep over a.  Block = 64 x 4 threads: thread (x, y) owns the
// 16-byte column groups x, x + 64, ... of rows y, y + 4, ... of the CTA's row range (coalesced 16-byte loads / stores),
// keeps its share of dw in registers, the four row-threads are summed through shared memory, one atomic per column and CTA.
constexpr int kHeadRows = 128;     // rows per CTA
template <int DOUT>
__global__ void __launch_bounds__(256) head_backward_kernel(const float* __restrict__ a, int64_t lda, int64_t m, int k,
                                                            const float* __restrict__ w, const float* __restrict__ g,
                                                            float* __restrict__ dz, int64_t ldz, float* __restrict__ dw,
                                                            float* __restrict__ db) {
  __shared__ float s_dw[4][DOUT][256];
  __shared__ float s_db[4][DOUT];
  const int x = threadIdx.x & 63, y = threadIdx.x >> 6;
  const int64_t r_begin = (int64_t)blockIdx.x * kHeadRows, r_end = min(m, r_begin + kHeadRows);
  const int groups = k / 4;                       // (k % 4 == 0, k <= 256: one group per thread x)
  float4 wv[DOUT], acc[DOUT];
  float gsum[DOUT];
#pragma unroll
  for (int j = 0; j < DOUT; ++j) {
    wv[j] = x < groups ? __ldg(reinterpret_cast<const float4*>(w + (int64_t)j * k) + x) : make_float4(0.f, 0.f, 0.f, 0.f);
    acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    gsum[j] = 0.f;
  }
  for (int64_t r = r_begin + y; r < r_end; r += 4) {
    float gj[DOUT];
#pragma unroll
    for (int j = 0; j < DOUT; ++j) { gj[j] = __ldg(g + r * DOUT + j); gsum[j] += gj[j]; }
    if (x < groups) {
      const float4 av = __ldg(reinterpret_cast<const float4*>(a + r * lda) + x);
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < DOUT; ++j) {
        t.x = fmaf(gj[j], wv[j].x, t.x); t.y = fmaf(gj[j], wv[j].y, t.y); t.z = fmaf(gj[j], wv[j].z, t.z); t.w = fmaf(gj[j], wv[j].w, t.w);
        acc[j].x = fmaf(gj[j], av.x, acc[j].x); acc[j].y = fmaf(gj[j], av.y, acc[j].y);
        acc[j].z = fmaf(gj[j], av.z, acc[j].z); acc[j].w = fmaf(gj[j], av.w, acc[j].w);
      }
      t.x *= softplus100_grad_from_output(av.x); t.y *= softplus100_grad_from_output(av.y);
      t.z *= softplus100_grad_from_output(av.z); t.w *= softplus100_grad_from_output(av.w);
      *(reinterpret_cast<float4*>(dz + r * ldz) + x) = t;
    }
  }
#pragma unroll
  for (int j = 0; j < DOUT; ++j) {
    s_dw[y][j][4 * x] = acc[j].x; s_dw[y][j][4 * x + 1] = acc[j].y; s_dw[y][j][4 * x + 2] = acc[j].z; s_dw[y][j][4 * x + 3] = acc[j].w;
    if (x == 0) s_db[y][j] = gsum[j];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < DOUT * k; i += 256) {
    const int j = i / k, c = i % k;
    atomicAdd(dw + i, s_dw[0][j][c] + s_dw[1][j][c] + s_dw[2][j][c] + s_dw[3][j][c]);
  }
  if (db != nullptr && threadIdx.x < DOUT) atomicAdd(db + threadIdx.x, s_db[0][threadIdx.x] + s_db[1][threadIdx.x] + s_db[2][threadIdx.x] + s_db[3][threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------- second derivative
// Directional derivative of the encoding along v: out = [v, 2^k cos(2^k x) v, -2^k sin(2^k x) v, ...], zero padding up to
// n_cols.  One thread per point (the GEMMs that read it dominate).
__global__ void __launch_bounds__(256) embed_tangent_kernel(const float* __restrict__ x, const float* __restrict__ v, int64_t m,
                                                            int n_freq, float* __restrict__ out, int64_t ld, int n_cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const float p[3] = {x[3 * i], x[3 * i + 1], x[3 * i + 2]};
  const float t[3] = {v[3 * i], v[3 * i + 1], v[3 * i + 2]};
  float* o = out + i * ld;
  o[0] = t[0]; o[1] = t[1]; o[2] = t[2];
  float f = 1.f;
  for (int k = 0; k < n_freq; ++k, f *= 2.f) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      float s, c;
      sincosf(f * p[d], &s, &c);
      o[3 + 6 * k + d] = f * c * t[d];
      o[6 + 6 * k + d] = -f * s * t[d];
    }
  }
  for (int c = 3 * (2 * n_freq + 1); c < n_cols; ++c) o[c] = 0.f;
}

// g_x = E'(x)^T gbar + E''(x)[v]^T g_emb: the adjoint of the encoding applied to gbar (skipped when gbar is null) plus the
// derivative of the first adjoint E'(x)^T g_emb along v, diagonal per coordinate: sum_k -4^k v (sin(2^k x) g_sin + cos(2^k x) g_cos).
__global__ void __launch_bounds__(256) embed_second_backward_kernel(const float* __restrict__ x, const float* __restrict__ v,
                                                                    int64_t m, int n_freq, const float* __restrict__ gbar,
                                                                    int64_t ldbar, const float* __restrict__ g_emb, int64_t ld,
                                                                    float* __restrict__ g_x) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const float* gb = gbar ? gbar + i * ldbar : nullptr;
  const float* ge = g_emb + i * ld;
  float acc[3] = {0.f, 0.f, 0.f};
  if (gb) { acc[0] = gb[0]; acc[1] = gb[1]; acc[2] = gb[2]; }
  float f = 1.f;
  for (int k = 0; k < n_freq; ++k, f *= 2.f) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      float s, c;
      sincosf(f * x[3 * i + d], &s, &c);
      if (gb) acc[d] += f * (c * gb[3 + 6 * k + d] - s * gb[6 + 6 * k + d]);
      acc[d] -= f * f * v[3 * i + d] * (s * ge[3 + 6 * k + d] + c * ge[6 + 6 * k + d]);
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) g_x[3 * i + d] = acc[d];
}

// Second derivative through the output layer in one sweep, laid out as head_backward_kernel:
//   dw[j, k] += sum_m g[m, j] adot[m, k],   mu[m, k] = beta [beta a <= 20] exp(-beta a) delta zdot   (a, delta, zdot at m, k)
template <int DOUT>
__global__ void __launch_bounds__(256) head_second_backward_kernel(const float* __restrict__ adot, int64_t ldad,
                                                                   const float* __restrict__ a, int64_t lda,
                                                                   const float* __restrict__ delta, int64_t ldd,
                                                                   const float* __restrict__ zdot, int64_t ldzd, int64_t m, int k,
                                                                   const float* __restrict__ g, float* __restrict__ dw,
                                                                   float* __restrict__ mu, int64_t ldmu) {
  __shared__ float s_dw[4][DOUT][256];
  const int x = threadIdx.x & 63, y = threadIdx.x >> 6;
  const int64_t r_begin = (int64_t)blockIdx.x * kHeadRows, r_end = min(m, r_begin + kHeadRows);
  const int groups = k / 4;
  float4 acc[DOUT];
#pragma unroll
  for (int j = 0; j < DOUT; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (x < groups) {
    for (int64_t r = r_begin + y; r < r_end; r += 4) {
      const float4 ad = __ldg(reinterpret_cast<const float4*>(adot + r * ldad) + x);
#pragma unroll
      for (int j = 0; j < DOUT; ++j) {
        const float gj = __ldg(g + r * DOUT + j);
        acc[j].x = fmaf(gj, ad.x, acc[j].x); acc[j].y = fmaf(gj, ad.y, acc[j].y);
        acc[j].z = fmaf(gj, ad.z, acc[j].z); acc[j].w = fmaf(gj, ad.w, acc[j].w);
      }
      const float4 av = __ldg(reinterpret_cast<const float4*>(a + r * lda) + x);
      const float4 dv = __ldg(reinterpret_cast<const float4*>(delta + r * ldd) + x);
      const float4 zv = __ldg(reinterpret_cast<const float4*>(zdot + r * ldzd) + x);
      *(reinterpret_cast<float4*>(mu + r * ldmu) + x) =
          make_float4(softplus100_curv_from_output(av.x) * dv.x * zv.x, softplus100_curv_from_output(av.y) * dv.y * zv.y,
                      softplus100_curv_from_output(av.z) * dv.z * zv.z, softplus100_curv_from_output(av.w) * dv.w * zv.w);
    }
  }
#pragma unroll
  for (int j = 0; j < DOUT; ++j) {
    s_dw[y][j][4 * x] = acc[j].x; s_dw[y][j][4 * x + 1] = acc[j].y; s_dw[y][j][4 * x + 2] = acc[j].z; s_dw[y][j][4 * x + 3] = acc[j].w;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < DOUT * k; i += 256) {
    const int j = i / k, c = i % k;
    atomicAdd(dw + i, s_dw[0][j][c] + s_dw[1][j][c] + s_dw[2][j][c] + s_dw[3][j][c]);
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace mlp
}  // namespace d3h

using namespace d3h;
using namespace d3h::mlp;

static int finish_launch(const char* who) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s: %s", who, cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}

template <int kEpi>
static void launch_linear(const LinearArgs& g, d3h_stream_t stream) {
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(mlp_linear_kernel<kEpi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stage_layout(256).bytes);
    attr = true;
  }
  mlp_linear_kernel<kEpi><<<(unsigned)((g.m + kTileM - 1) / kTileM), kThreads, stage_layout(g.n).bytes, (cudaStream_t)stream>>>(g);
}

extern "C" int d3h_mlp_embed(const float* x, int64_t m, int32_t n_freq, float* out, int64_t ld, int32_t n_cols,
                             d3h_stream_t stream) {
  if (m < 0 || n_freq < 0 || n_freq > 16 || n_cols < 3 * (2 * n_freq + 1) || ld < n_cols || (m > 0 && (!x || !out))) {
    set_error("d3h_mlp_embed: bad argument (n_cols must hold the 3 (2 n_freq + 1) channels, ld >= n_cols)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  if ((n_cols % 4) == 0 && (ld % 4) == 0 && aligned16(out))
    embed4_kernel<<<(unsigned)((m * (n_cols / 4) + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, m, n_freq, out, ld, n_cols);
  else
    embed_kernel<<<(unsigned)((m + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, m, n_freq, out, ld, n_cols);
  return finish_launch("d3h_mlp_embed");
}

extern "C" int d3h_mlp_embed_backward(const float* x, int64_t m, int32_t n_freq, const float* g_emb, int64_t ld,
                                      float* g_x, int32_t accumulate, d3h_stream_t stream) {
  if (m < 0 || n_freq < 0 || n_freq > 16 || ld < 3 * (2 * n_freq + 1) || (m > 0 && (!x || !g_emb || !g_x))) {
    set_error("d3h_mlp_embed_backward: bad argument");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  embed_backward_kernel<<<(unsigned)((m + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, m, n_freq, g_emb, ld, g_x, accumulate);
  return finish_launch("d3h_mlp_embed_backward");
}

extern "C" int64_t d3h_mlp_packed_weight_bytes(int32_t n_pad, int32_t k_pad) { return (int64_t)8 * n_pad * k_pad; }

extern "C" int d3h_mlp_pack_weight(const float* w, int64_t ldw, int32_t n_valid, int32_t k_valid, int32_t transpose,
                                   int32_t row0, int32_t col0, int32_t n_pad, int32_t k_pad, float* packed,
                                   d3h_stream_t stream) {
  if (!w || !packed || n_valid < 0 || k_valid < 0 || n_valid > n_pad || k_valid > k_pad || n_pad < 64 || n_pad > 256 ||
      (n_pad % 64) || k_pad <= 0 || (k_pad % kSliceK) || row0 < 0 || col0 < 0 || ldw <= 0 || !aligned16(packed)) {
    set_error("d3h_mlp_pack_weight: bad argument (n_pad in {64, 128, 192, 256}, k_pad %% 32 == 0, valid sizes within the padded "
              "ones, packed 16-byte aligned)");
    return D3H_E_BADARG;
  }
  PackArgs g{w, ldw, packed, n_valid, k_valid, transpose ? 1 : 0, row0, col0, n_pad, k_pad};
  const int64_t total = (int64_t)n_pad * (k_pad / 4);
  mlp_pack_weight_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(g);
  return finish_launch("d3h_mlp_pack_weight");
}

extern "C" int d3h_mlp_linear(const float* a, int64_t lda, int64_t m, int32_t k, const float* w_packed, int32_t n,
                              const float* bias, int32_t mode, const float* y, int64_t ldy, float* c, int64_t ldc,
                              d3h_stream_t stream) {
  if (m < 0 || k <= 0 || (k % kSliceK) || n < 64 || n > 256 || (n % 64) || mode < 0 || mode > 2 || lda < k ||
      ldc < n || (lda % 4) || (ldc % 4) || !w_packed || (m > 0 && (!a || !c)) || !aligned16(a) || !aligned16(w_packed) ||
      !aligned16(c) || (mode == 2 && (!y || ldy < n || (ldy % 4) || !aligned16(y)))) {
    set_error("d3h_mlp_linear: bad argument (K %% 32 == 0, N in {64, 128, 192, 256}, leading dimensions multiples of 4 "
              "and >= the row length, 16-byte aligned pointers, mode 2 needs y)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  LinearArgs g{a, lda, w_packed, bias, y, ldy, c, ldc, m, k, n, mode};
  launch_linear<kEpiFirstOrder>(g, stream);
  return finish_launch("d3h_mlp_linear");
}

// shape / alignment rules of the tangent and adjoint variants: those of d3h_mlp_linear, with y always required
static bool linear_shape_ok(const float* a, int64_t lda, int64_t m, int32_t k, const float* w_packed, int32_t n,
                            const float* y, int64_t ldy, const float* c, int64_t ldc) {
  return m >= 0 && k > 0 && (k % kSliceK) == 0 && n >= 64 && n <= 256 && (n % 64) == 0 && lda >= k && ldc >= n &&
         (lda % 4) == 0 && (ldc % 4) == 0 && w_packed && (m == 0 || (a && c && y)) && aligned16(a) && aligned16(w_packed) &&
         aligned16(c) && ldy >= n && (ldy % 4) == 0 && aligned16(y);
}
static bool operand_ok(const float* p, int64_t ld, int64_t m, int32_t n) {
  return (m == 0 || p) && ld >= n && (ld % 4) == 0 && aligned16(p);
}

extern "C" int d3h_mlp_linear_tangent(const float* a, int64_t lda, int64_t m, int32_t k, const float* w_packed, int32_t n,
                                      const float* y, int64_t ldy, float* zdot, int64_t ldzd, float* adot, int64_t ldad,
                                      d3h_stream_t stream) {
  if (!linear_shape_ok(a, lda, m, k, w_packed, n, y, ldy, adot, ldad) || !operand_ok(zdot, ldzd, m, n)) {
    set_error("d3h_mlp_linear_tangent: bad argument (K %% 32 == 0, N in {64, 128, 192, 256}, y / zdot / adot of N columns, "
              "leading dimensions multiples of 4, 16-byte aligned pointers)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  LinearArgs g{a, lda, w_packed, nullptr, y, ldy, adot, ldad, m, k, n, 0, zdot, ldzd};
  launch_linear<kEpiTangent>(g, stream);
  return finish_launch("d3h_mlp_linear_tangent");
}

extern "C" int d3h_mlp_linear_adjoint(const float* a, int64_t lda, int64_t m, int32_t k, const float* w_packed, int32_t n,
                                      const float* y, int64_t ldy, const float* delta, int64_t ldd, const float* zdot,
                                      int64_t ldzd, float* c, int64_t ldc, d3h_stream_t stream) {
  if (!linear_shape_ok(a, lda, m, k, w_packed, n, y, ldy, c, ldc) || !operand_ok(delta, ldd, m, n) ||
      !operand_ok(zdot, ldzd, m, n)) {
    set_error("d3h_mlp_linear_adjoint: bad argument (K %% 32 == 0, N in {64, 128, 192, 256}, y / delta / zdot / c of N "
              "columns, leading dimensions multiples of 4, 16-byte aligned pointers)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  LinearArgs g{a, lda, w_packed, nullptr, y, ldy, c, ldc, m, k, n, 0, nullptr, 0, delta, ldd, zdot, ldzd};
  launch_linear<kEpiAdjoint>(g, stream);
  return finish_launch("d3h_mlp_linear_adjoint");
}

extern "C" int d3h_mlp_embed_tangent(const float* x, const float* v, int64_t m, int32_t n_freq, float* out, int64_t ld,
                                     int32_t n_cols, d3h_stream_t stream) {
  if (m < 0 || n_freq < 0 || n_freq > 16 || n_cols < 3 * (2 * n_freq + 1) || ld < n_cols || (m > 0 && (!x || !v || !out))) {
    set_error("d3h_mlp_embed_tangent: bad argument (n_cols must hold the 3 (2 n_freq + 1) channels, ld >= n_cols)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  embed_tangent_kernel<<<(unsigned)((m + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, v, m, n_freq, out, ld, n_cols);
  return finish_launch("d3h_mlp_embed_tangent");
}

extern "C" int d3h_mlp_embed_second_backward(const float* x, const float* v, int64_t m, int32_t n_freq, const float* gbar,
                                             int64_t ldbar, const float* g_emb, int64_t ld, float* g_x, d3h_stream_t stream) {
  const int e = 3 * (2 * n_freq + 1);
  if (m < 0 || n_freq < 0 || n_freq > 16 || ld < e || (gbar && ldbar < e) || (m > 0 && (!x || !v || !g_emb || !g_x))) {
    set_error("d3h_mlp_embed_second_backward: bad argument (g_emb, and gbar if given, hold the 3 (2 n_freq + 1) channels)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  embed_second_backward_kernel<<<(unsigned)((m + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, v, m, n_freq, gbar, ldbar,
                                                                                             g_emb, ld, g_x);
  return finish_launch("d3h_mlp_embed_second_backward");
}

extern "C" int d3h_mlp_head_second_backward(const float* adot, int64_t ldad, const float* a, int64_t lda, const float* delta,
                                            int64_t ldd, const float* zdot, int64_t ldzd, int64_t m, int32_t k,
                                            const float* g, int32_t d_out, float* dw, float* mu, int64_t ldmu,
                                            d3h_stream_t stream) {
  if (m < 0 || k <= 0 || k > 256 || (k % 4) || d_out <= 0 || d_out > 8 || !dw || (m > 0 && !g) ||
      !operand_ok(adot, ldad, m, k) || !operand_ok(a, lda, m, k) || !operand_ok(delta, ldd, m, k) ||
      !operand_ok(zdot, ldzd, m, k) || !operand_ok(mu, ldmu, m, k)) {
    set_error("d3h_mlp_head_second_backward: bad argument (K <= 256 and a multiple of 4, 1 <= d_out <= 8, leading "
              "dimensions multiples of 4, 16-byte aligned adot / a / delta / zdot / mu)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  const unsigned blocks = (unsigned)((m + kHeadRows - 1) / kHeadRows);
  cudaStream_t st = (cudaStream_t)stream;
#define D3H_HEAD2(D) head_second_backward_kernel<D><<<blocks, 256, 0, st>>>(adot, ldad, a, lda, delta, ldd, zdot, ldzd, m, k, g, dw, mu, ldmu)
  switch (d_out) {
    case 1: D3H_HEAD2(1); break;
    case 2: D3H_HEAD2(2); break;
    case 3: D3H_HEAD2(3); break;
    case 4: D3H_HEAD2(4); break;
    case 5: D3H_HEAD2(5); break;
    case 6: D3H_HEAD2(6); break;
    case 7: D3H_HEAD2(7); break;
    default: D3H_HEAD2(8); break;
  }
#undef D3H_HEAD2
  return finish_launch("d3h_mlp_head_second_backward");
}

// point ranges of a wgrad call: two CTAs per SM and column tile, at least 16 slices (512 points) each
static void wgrad_ranges(int64_t m, int n, int64_t* ranges, int64_t* per) {
  int64_t r = (int64_t)kCtasPerSm * 148 / (n / kTileM);
  int64_t p = ((m + r - 1) / r + kSliceK - 1) / kSliceK * kSliceK;
  if (p < 16 * kSliceK) p = 16 * kSliceK;
  *per = p;
  *ranges = (m + p - 1) / p;
}

extern "C" int64_t d3h_mlp_wgrad_workspace_bytes(int64_t m, int32_t n, int32_t k) {
  if (m <= 0 || n <= 0 || (n % kTileM) || k <= 0) return 0;
  int64_t ranges, per;
  wgrad_ranges(m, n, &ranges, &per);
  return ranges * ((int64_t)n * k + n) * 4;
}

extern "C" int d3h_mlp_wgrad(const float* dz, int64_t ldz, const float* a, int64_t lda, int64_t m, int32_t n, int32_t k,
                             float* dw, int64_t lddw, float* db, void* workspace, int64_t workspace_bytes,
                             d3h_stream_t stream) {
  if (m < 0 || n <= 0 || (n % kTileM) || n > 256 || k < 64 || k > 256 || (k % 64) || ldz < n || lda < k || lddw < k ||
      (ldz % 4) || (lda % 4) || !dw || (m > 0 && (!dz || !a)) || !aligned16(dz) || !aligned16(a) || !aligned16(workspace)) {
    set_error("d3h_mlp_wgrad: bad argument (N in {128, 256}, K in {64, 128, 192, 256}, leading dimensions multiples "
              "of 4, 16-byte aligned pointers)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  if (!workspace || workspace_bytes < d3h_mlp_wgrad_workspace_bytes(m, n, k)) {
    set_error("d3h_mlp_wgrad: workspace has %lld bytes, %lld needed", (long long)workspace_bytes,
              (long long)d3h_mlp_wgrad_workspace_bytes(m, n, k));
    return D3H_E_SMALLWS;
  }
  const size_t smem = stage_layout(k).bytes;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(mlp_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stage_layout(256).bytes);
    attr = true;
  }
  int64_t ranges, per;
  wgrad_ranges(m, n, &ranges, &per);
  float* part = reinterpret_cast<float*>(workspace);
  float* part_b = db ? part + ranges * (int64_t)n * k : nullptr;
  WgradArgs g{dz, ldz, a, lda, part, part_b, m, per, n, k};
  mlp_wgrad_kernel<<<dim3((unsigned)ranges, (unsigned)(n / kTileM)), kThreads, smem, (cudaStream_t)stream>>>(g);
  const int64_t total = (int64_t)n * k + (db ? n : 0);
  wgrad_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(part, part_b, (int)ranges, n, k, dw, lddw, db);
  return finish_launch("d3h_mlp_wgrad");
}

extern "C" int d3h_mlp_head(const float* a, int64_t lda, int64_t m, int32_t k, const float* w, const float* bias,
                            int32_t d_out, float* out, d3h_stream_t stream) {
  if (m < 0 || k <= 0 || d_out <= 0 || d_out > 8 || lda < k || !w || (m > 0 && (!a || !out))) {
    set_error("d3h_mlp_head: bad argument (1 <= d_out <= 8)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  head_kernel<<<(unsigned)((m + 7) / 8), 256, 0, (cudaStream_t)stream>>>(a, lda, m, k, w, bias, d_out, out);
  return finish_launch("d3h_mlp_head");
}

extern "C" int d3h_mlp_head_backward(const float* a, int64_t lda, int64_t m, int32_t k, const float* w, int32_t d_out,
                                     const float* g, float* dz, int64_t ldz, float* dw, float* db, d3h_stream_t stream) {
  if (m < 0 || k <= 0 || k > 256 || (k % 4) || d_out <= 0 || d_out > 8 || lda < k || ldz < k || (lda % 4) || (ldz % 4) || !w || !dw ||
      (m > 0 && (!a || !g || !dz)) || !aligned16(a) || !aligned16(dz) || !aligned16(w)) {
    set_error("d3h_mlp_head_backward: bad argument (K <= 256 and a multiple of 4, 1 <= d_out <= 8, leading dimensions multiples of 4, "
              "16-byte aligned a / dz / w)");
    return D3H_E_BADARG;
  }
  if (m == 0) return D3H_OK;
  const unsigned blocks = (unsigned)((m + kHeadRows - 1) / kHeadRows);
  cudaStream_t st = (cudaStream_t)stream;
  switch (d_out) {
    case 1: head_backward_kernel<1><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
    case 2: head_backward_kernel<2><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
    case 3: head_backward_kernel<3><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
    case 4: head_backward_kernel<4><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
    case 5: head_backward_kernel<5><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
    case 6: head_backward_kernel<6><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
    case 7: head_backward_kernel<7><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
    default: head_backward_kernel<8><<<blocks, 256, 0, st>>>(a, lda, m, k, w, g, dz, ldz, dw, db); break;
  }
  return finish_launch("d3h_mlp_head_backward");
}
