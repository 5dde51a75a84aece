// TEST INFRASTRUCTURE ONLY: fibre scheduler of the CPU emulation (see tests/emu/cuda_runtime.h).
#include <stdio.h>
#include <time.h>
#include <ucontext.h>

#include <unordered_map>
#include <vector>

#include "cuda_runtime.h"

// EMU_TSAN (tests/emu/build_emu.py, tsan=True): every emulated CUDA thread is a ThreadSanitizer fibre.  Fibre switches
// carry NO synchronisation; happens-before edges are added exactly where CUDA gives them: __syncthreads (block-wide),
// __syncwarp (the named lanes), kernel boundaries, and device atomics (cuda_runtime.h maps them to seq_cst atomics).
// TSan then reports two emulated threads touching the same shared or global address without such an edge -- the offline
// stand-in for `compute-sanitizer --tool racecheck` (which only sees shared memory).
#ifdef EMU_TSAN
#include <sanitizer/tsan_interface.h>
#define TSAN_ONLY(x) x
#else
#define TSAN_ONLY(x)
#endif

namespace emu {

Idx g_threadIdx, g_blockIdx, g_blockDim, g_gridDim;

namespace {
constexpr size_t kStack = 256 * 1024;
enum State { kRunnable, kAtBarrier, kAtCollective, kAtMbarrier, kDone };
struct Fibre {
  TSAN_ONLY(void* tsan = nullptr;)
  ucontext_t ctx;
  char* stack = nullptr;
  State st = kDone;
  unsigned barrier_gen = 0;
  // pending warp collective
  unsigned coll_mask = 0;
  unsigned long long coll_val = 0;
  unsigned long long coll_out[32];
  // pending mbarrier.try_wait.parity loop: index into BlockState::mbar, parity waited for
  unsigned wait_bar = 0, wait_parity = 0;
};
// mbarrier (PTX ISA, "Parallel synchronization and communication instructions: mbarrier"): a phase completes when its
// pending arrival count AND its transaction count are both zero; the next phase starts with the expected count again
struct Mbar {
  const uint64_t* addr;
  unsigned expected, pending;
  long long tx;        // outstanding transaction bytes (may go negative: complete_tx may precede expect_tx)
  unsigned phase;      // phases completed so far; try_wait.parity(p) succeeds once the phase of parity p completed
};
// one tcgen05.mma.kind::tf32 issued and not yet committed: operands decoded at issue (the snapshot), the D columns
struct PendingMma {
  uint64_t desc_a, desc_b;
  unsigned col, n;
  bool accumulate;
  std::vector<float> a, b;   // 128 x 8 and n x 8, TF32-truncated
};
constexpr unsigned kTmemLanes = 128, kTmemCols = 512;
struct BlockState {
  std::vector<Fibre> f;
  unsigned n = 0, alive = 0, at_barrier = 0, barrier_gen = 0;
  unsigned cur = 0;
  TSAN_ONLY(void* sched_tsan = nullptr;)
  char barrier_obj = 0;      // TSan sync object of __syncthreads
  char warp_obj[32] = {0};   // ... of __syncwarp, one per warp
  ucontext_t sched;
  const std::function<void()>* body = nullptr;
  std::vector<Mbar> mbar;                // the block's initialised mbarriers
  std::vector<float> tmem;               // tensor memory: 128 lanes x 512 columns of 32-bit cells
  unsigned tmem_next = 0, tmem_live = 0; // next free column, columns allocated and not yet freed
  std::vector<PendingMma> mma;           // issued, not yet committed
};
BlockState B;
std::vector<char*> g_stacks;
char g_launch_obj = 0;  // TSan sync objects: scheduler -> threads of the next block ...
char g_done_obj = 0;    // ... and exiting threads -> scheduler (two objects: an exiting thread must not order itself
                        // before a thread of the same block that merely starts later)
unsigned char* g_dyn = nullptr;         // dynamic shared memory of the running launch (one block at a time)
size_t g_dyn_bytes = 0;
// shared-memory window: the static __shared__ section at offset 0, the dynamic buffer at 1024 as on the GPU (static
// variables first, the dynamic buffer behind them at its declared 1024-byte alignment)
constexpr uint32_t kDynBase = 1024;
int g_last_error = 0;
std::unordered_map<const void*, int> g_max_dyn_smem;

[[noreturn]] void fail(const char* what) {
  fprintf(stderr, "emu: %s (block (%u,%u), thread %u)\n", what, g_blockIdx.x, g_blockIdx.y, g_threadIdx.x);
  abort();
}

// D3H_EMU_SHUFFLE=<seed>: blocks run in a random order and every scheduler sweep starts at a random thread, in a random
// direction.  Results must not depend on either (on the GPU both are arbitrary): a shared variable read without the
// barrier that orders it after its writer, or an assumption that lower block indices ran first, shows up as a parity
// failure under some seed.  0 / unset = blocks and threads in index order.
unsigned long long g_rng = 0;
bool g_shuffle = false, g_shuffle_init = false;
unsigned rnd(unsigned n) {  // xorshift64*, uniform enough for shuffling
  g_rng ^= g_rng >> 12; g_rng ^= g_rng << 25; g_rng ^= g_rng >> 27;
  return (unsigned)(((g_rng * 2685821657736338717ull) >> 33) % (n ? n : 1));
}
void init_shuffle() {
  if (g_shuffle_init) return;
  g_shuffle_init = true;
  const char* e = getenv("D3H_EMU_SHUFFLE");
  if (e && atoll(e) != 0) { g_shuffle = true; g_rng = 0x9E3779B97F4A7C15ull ^ (unsigned long long)atoll(e); }
}

void fibre_entry() {
  TSAN_ONLY(__tsan_acquire(&g_launch_obj);)   // everything before the launch happened before this thread
  (*B.body)();
  TSAN_ONLY(__tsan_release(&g_done_obj);)     // ... and this thread happens before whatever follows the block
  B.f[B.cur].st = kDone;
  --B.alive;
  // a thread that exits never reaches the barrier the others wait at: release them if it was the last one missing
  if (B.alive > 0 && B.at_barrier == B.alive) { B.at_barrier = 0; ++B.barrier_gen; }
  TSAN_ONLY(__tsan_switch_to_fiber(B.sched_tsan, __tsan_switch_to_fiber_no_sync);)
  swapcontext(&B.f[B.cur].ctx, &B.sched);
}

void yield_to_scheduler() {
  TSAN_ONLY(__tsan_switch_to_fiber(B.sched_tsan, __tsan_switch_to_fiber_no_sync);)
  swapcontext(&B.f[B.cur].ctx, &B.sched);
}

// completes every collective of warp `w` whose participants have all arrived
void try_complete_collectives(unsigned w) {
  const unsigned base = w * 32;
  const unsigned lanes = (B.n - base) < 32u ? (B.n - base) : 32u;
  for (unsigned l = 0; l < lanes; ++l) {
    Fibre& a = B.f[base + l];
    if (a.st != kAtCollective) continue;
    const unsigned mask = a.coll_mask;
    bool ready = true;
    for (unsigned j = 0; j < 32 && ready; ++j) {
      if (!((mask >> j) & 1u)) continue;
      if (j >= lanes) continue;                       // lanes beyond the block do not exist
      const Fibre& p = B.f[base + j];
      if (p.st == kDone) continue;                    // exited lanes cannot arrive (result for them is undefined)
      if (p.st != kAtCollective || p.coll_mask != mask) ready = false;
    }
    if (!ready) continue;
    unsigned long long vals[32];
    for (unsigned j = 0; j < 32; ++j) {
      const bool in = ((mask >> j) & 1u) && j < lanes && B.f[base + j].st == kAtCollective;
      vals[j] = in ? B.f[base + j].coll_val : 0ull;
    }
    for (unsigned j = 0; j < lanes; ++j) {
      Fibre& p = B.f[base + j];
      if (((mask >> j) & 1u) && p.st == kAtCollective && p.coll_mask == mask) {
        memcpy(p.coll_out, vals, sizeof(vals));
        p.st = kRunnable;
      }
    }
  }
}
}  // namespace

void set_shuffle(unsigned long long seed) {
  g_shuffle_init = true;
  g_shuffle = seed != 0;
  g_rng = 0x9E3779B97F4A7C15ull ^ seed;
}

void block_barrier() {
  Fibre& me = B.f[B.cur];
  me.st = kAtBarrier;
  me.barrier_gen = B.barrier_gen;
  TSAN_ONLY(__tsan_release(&B.barrier_obj);)
  if (++B.at_barrier == B.alive) { B.at_barrier = 0; ++B.barrier_gen; }
  yield_to_scheduler();
  TSAN_ONLY(__tsan_acquire(&B.barrier_obj);)  // every thread of the block released before anybody got here
}

// __syncwarp: memory ordering among the lanes of `mask` (the rendezvous itself is a warp_exchange)
void warp_sync_release() { TSAN_ONLY(__tsan_release(&B.warp_obj[(B.cur >> 5) & 31u]);) }
void warp_sync_acquire() { TSAN_ONLY(__tsan_acquire(&B.warp_obj[(B.cur >> 5) & 31u]);) }

void warp_exchange(unsigned mask, unsigned long long v, unsigned long long out[32]) {
  Fibre& me = B.f[B.cur];
  const unsigned lane = B.cur & 31u;
  if (!((mask >> lane) & 1u)) {
    fprintf(stderr, "emu: lane %u calls a warp collective whose mask %08x does not name it\n", lane, mask);
    abort();
  }
  me.coll_mask = mask;
  me.coll_val = v;
  me.st = kAtCollective;
  try_complete_collectives(B.cur >> 5);
  if (me.st != kRunnable) yield_to_scheduler();
  memcpy(out, me.coll_out, sizeof(me.coll_out));
}

unsigned long long now_ns() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (unsigned long long)ts.tv_sec * 1000000000ull + (unsigned long long)ts.tv_nsec;
}

extern "C" char __start_emu_shared[] __attribute__((weak));
extern "C" char __stop_emu_shared[] __attribute__((weak));

static void run_block(const std::function<void()>& body, unsigned nthreads) {
  // shared memory of a fresh CTA holds arbitrary data on the GPU: never zeros by contract
  if (__start_emu_shared != nullptr && __stop_emu_shared > __start_emu_shared) {
    memset(__start_emu_shared, 0xCB, (size_t)(__stop_emu_shared - __start_emu_shared));
  }
  if (g_dyn != nullptr) memset(g_dyn, 0xCB, g_dyn_bytes);   // the dynamic part likewise
  // Every block has its OWN shared memory, but the emulation re-uses one set of static variables: blocks are therefore
  // ordered one after the other for ThreadSanitizer (block k -> scheduler -> block k+1).  This hides races between
  // DIFFERENT blocks on global memory; races inside a block -- what a missing __syncthreads / __syncwarp causes -- are
  // what this build is for.
  TSAN_ONLY(__tsan_release(&g_launch_obj);)
  if (B.f.size() < nthreads) B.f.resize(nthreads);
  while (g_stacks.size() < nthreads) g_stacks.push_back((char*)malloc(kStack));
  B.n = B.alive = nthreads;
  B.at_barrier = 0;
  B.barrier_gen = 0;
  B.body = &body;
  B.mbar.clear();
  B.mma.clear();
  // tensor memory: the second CTA on an SM finds the first one's 256 columns taken -- odd blocks start at column 256
  const unsigned long long linear = g_blockIdx.x + (unsigned long long)g_gridDim.x * (g_blockIdx.y + (unsigned long long)g_gridDim.y * g_blockIdx.z);
  B.tmem_next = (linear & 1u) ? kTmemCols / 2 : 0u;
  B.tmem_live = 0;
  TSAN_ONLY(B.sched_tsan = __tsan_get_current_fiber();)
  for (unsigned t = 0; t < nthreads; ++t) {
    Fibre& f = B.f[t];
    TSAN_ONLY(if (f.tsan == nullptr) f.tsan = __tsan_create_fiber(0);)
    f.stack = g_stacks[t];
    f.st = kRunnable;
    getcontext(&f.ctx);
    f.ctx.uc_stack.ss_sp = f.stack;
    f.ctx.uc_stack.ss_size = kStack;
    f.ctx.uc_link = nullptr;
    makecontext(&f.ctx, fibre_entry, 0);
  }
  while (B.alive > 0) {
    bool progressed = false;
    const unsigned off = g_shuffle ? rnd(nthreads) : 0u;
    const bool back = g_shuffle && (rnd(2) == 1u);
    for (unsigned k = 0; k < nthreads; ++k) {
      const unsigned t = back ? (off + nthreads - k) % nthreads : (off + k) % nthreads;
      Fibre& f = B.f[t];
      if (f.st == kAtBarrier && f.barrier_gen != B.barrier_gen) f.st = kRunnable;
      if (f.st == kAtCollective) try_complete_collectives(t >> 5);
      if (f.st == kAtMbarrier && (B.mbar[f.wait_bar].phase & 1u) != f.wait_parity) f.st = kRunnable;
      if (f.st != kRunnable) continue;
      B.cur = t;
      g_threadIdx = Idx{t, 0, 0};
      progressed = true;
      TSAN_ONLY(__tsan_switch_to_fiber(f.tsan, __tsan_switch_to_fiber_no_sync);)
      swapcontext(&B.sched, &f.ctx);
    }
    if (!progressed && B.alive > 0) {
      unsigned at_mbar = 0;
      for (unsigned t = 0; t < nthreads; ++t) at_mbar += B.f[t].st == kAtMbarrier;
      fprintf(stderr, "emu: deadlock in block (%u,%u): %u threads alive, %u at the barrier, %u waiting on an mbarrier\n",
              g_blockIdx.x, g_blockIdx.y, B.alive, B.at_barrier, at_mbar);
      abort();
    }
  }
  TSAN_ONLY(__tsan_acquire(&g_done_obj);)
  if (!B.mma.empty()) fail("tcgen05.mma issued but never committed at block exit");
  if (B.tmem_live != 0) fail("tensor memory still allocated at block exit (missing tcgen05.dealloc)");
}

void run_grid(dim3 grid, dim3 block, const std::function<void()>& body, size_t dyn_smem_bytes) {
  if (block.y != 1 || block.z != 1) { fprintf(stderr, "emu: only 1-D blocks are supported\n"); abort(); }
  struct DynSmem {   // one buffer per launch (the blocks run one after the other), exactly the launch's size
    explicit DynSmem(size_t n) {
      g_dyn = nullptr;
      g_dyn_bytes = n;
      if (n > 0 && posix_memalign(reinterpret_cast<void**>(&g_dyn), 1024, n) != 0) fail("out of memory");
    }
    ~DynSmem() { free(g_dyn); g_dyn = nullptr; g_dyn_bytes = 0; }
  } dyn(dyn_smem_bytes);
  g_gridDim = Idx{grid.x, grid.y, grid.z};
  g_blockDim = Idx{block.x, block.y, block.z};
  init_shuffle();
  TSAN_ONLY(__tsan_release(&g_launch_obj);)
  struct AcquireAtExit { ~AcquireAtExit() { TSAN_ONLY(__tsan_acquire(&g_done_obj);) } } acquire_at_exit;
  if (g_shuffle) {
    const unsigned long long total = (unsigned long long)grid.x * grid.y * grid.z;
    std::vector<unsigned> order(total);
    for (unsigned long long i = 0; i < total; ++i) order[i] = (unsigned)i;
    for (unsigned long long i = total; i > 1; --i) std::swap(order[i - 1], order[rnd((unsigned)i)]);
    for (unsigned long long i = 0; i < total; ++i) {
      const unsigned b = order[i];
      g_blockIdx = Idx{b % grid.x, (b / grid.x) % grid.y, b / (grid.x * grid.y)};
      run_block(body, block.x);
    }
    return;
  }
  for (unsigned bz = 0; bz < grid.z; ++bz)
    for (unsigned by = 0; by < grid.y; ++by)
      for (unsigned bx = 0; bx < grid.x; ++bx) {
        g_blockIdx = Idx{bx, by, bz};
        run_block(body, block.x);
      }
}

// ---- launches ----------------------------------------------------------------------------------------------------------
int take_last_error() { const int e = g_last_error; g_last_error = 0; return e; }
void set_last_error(int e) { g_last_error = e; }
int func_max_dynamic_smem(const void* f) {
  const auto it = g_max_dyn_smem.find(f);
  return it == g_max_dyn_smem.end() ? 48 * 1024 : it->second;
}
void set_func_max_dynamic_smem(const void* f, int bytes) { g_max_dyn_smem[f] = bytes; }

// ---- shared memory -----------------------------------------------------------------------------------------------------
unsigned char* dyn_smem() {
  if (g_dyn == nullptr) fail("extern __shared__ used by a kernel launched without dynamic shared memory");
  return g_dyn;
}
size_t dyn_smem_bytes() { return g_dyn_bytes; }
size_t cvta_generic_to_shared(const void* p) {
  const unsigned char* c = static_cast<const unsigned char*>(p);
  if (g_dyn != nullptr && c >= g_dyn && c < g_dyn + g_dyn_bytes) return kDynBase + (size_t)(c - g_dyn);
  const char* s = static_cast<const char*>(p);
  if (__start_emu_shared != nullptr && s >= __start_emu_shared && s < __stop_emu_shared && (size_t)(s - __start_emu_shared) < kDynBase)
    return (size_t)(s - __start_emu_shared);
  fail("__cvta_generic_to_shared of an address outside the shared window");
}
// shared address -> host pointer of `bytes` bytes inside the dynamic buffer (operands of the async proxy live there)
static unsigned char* dyn_at(uint64_t saddr, size_t bytes, const char* who) {
  if (saddr < kDynBase || saddr - kDynBase + bytes > g_dyn_bytes) {
    fprintf(stderr, "emu: %s: shared address 0x%llx + %zu bytes outside the dynamic shared memory (%zu bytes at 0x%x)\n", who,
            (unsigned long long)saddr, bytes, g_dyn_bytes, kDynBase);
    fail("shared-memory operand out of range");
  }
  return g_dyn + (saddr - kDynBase);
}

// ---- mbarrier ----------------------------------------------------------------------------------------------------------
static unsigned mbar_index(const uint64_t* bar) {
  for (unsigned i = 0; i < B.mbar.size(); ++i)
    if (B.mbar[i].addr == bar) return i;
  fail("mbarrier operation on an address that mbarrier.init has not initialised in this block");
}
static void mbar_complete_if_done(Mbar& m) {
  if (m.pending == 0 && m.tx == 0) { ++m.phase; m.pending = m.expected; }
}
void mbar_init(uint64_t* bar, unsigned count) {
  if (count == 0 || count >= (1u << 20)) fail("mbarrier.init: count outside [1, 2^20)");
  if ((reinterpret_cast<uintptr_t>(bar) & 7u) != 0) fail("mbarrier.init: address not 8-byte aligned");
  for (Mbar& m : B.mbar)
    if (m.addr == bar) { m = Mbar{bar, count, count, 0, 0}; return; }
  B.mbar.push_back(Mbar{bar, count, count, 0, 0});
}
static void mbar_arrive_one(uint64_t* bar, long long tx) {
  Mbar& m = B.mbar[mbar_index(bar)];
  if (m.pending == 0) fail("mbarrier: more arrivals than the phase expects");
  TSAN_ONLY(__tsan_release(bar);)      // arrive has release semantics
  m.tx += tx;
  --m.pending;
  mbar_complete_if_done(m);
}
void mbar_arrive(uint64_t* bar) { mbar_arrive_one(bar, 0); }
void mbar_arrive_expect_tx(uint64_t* bar, unsigned bytes) { mbar_arrive_one(bar, (long long)bytes); }
static void mbar_complete_tx(uint64_t* bar, unsigned bytes) {
  Mbar& m = B.mbar[mbar_index(bar)];
  TSAN_ONLY(__tsan_release(bar);)
  m.tx -= (long long)bytes;
  mbar_complete_if_done(m);
}
// the try_wait.parity loop of the kernel: parked (not spinning) until the phase of parity `parity` has completed, so that
// a protocol error ends in the scheduler's deadlock report
void mbar_wait(uint64_t* bar, unsigned parity) {
  const unsigned i = mbar_index(bar);
  if ((B.mbar[i].phase & 1u) == (parity & 1u)) {
    Fibre& me = B.f[B.cur];
    me.wait_bar = i;
    me.wait_parity = parity & 1u;
    me.st = kAtMbarrier;
    yield_to_scheduler();
  }
  TSAN_ONLY(__tsan_acquire(bar);)      // a successful wait acquires
}

// ---- cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes ----------------------------------------------------
void bulk_copy_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  if (bytes == 0 || bytes % 16 != 0) fail("cp.async.bulk: size not a positive multiple of 16");
  if ((reinterpret_cast<uintptr_t>(dst) & 15u) || (reinterpret_cast<uintptr_t>(src) & 15u)) fail("cp.async.bulk: address not 16-byte aligned");
  unsigned char* d = static_cast<unsigned char*>(dst);
  if (g_dyn == nullptr || d < g_dyn || d + bytes > g_dyn + g_dyn_bytes) fail("cp.async.bulk: destination outside the dynamic shared memory");
  memcpy(d, src, bytes);
  mbar_complete_tx(bar, bytes);
}

// ---- tensor memory -------------------------------------------------------------------------------------------------------
void tmem_alloc(uint32_t* dst, unsigned cols) {
  if (cols < 32 || cols > kTmemCols || (cols & (cols - 1)) != 0) fail("tcgen05.alloc: column count not a power of two in [32, 512]");
  if (B.tmem_next + cols > kTmemCols) fail("tcgen05.alloc: more than the 512 columns of tensor memory");
  if (B.tmem.empty()) B.tmem.resize((size_t)kTmemLanes * kTmemCols);
  for (unsigned l = 0; l < kTmemLanes; ++l)   // fresh tensor memory holds arbitrary data
    memset(&B.tmem[(size_t)l * kTmemCols + B.tmem_next], 0xCB, cols * 4);
  *dst = B.tmem_next;                         // lane 0, column base
  B.tmem_next += cols;
  B.tmem_live += cols;
}
void tmem_dealloc(uint32_t taddr, unsigned cols) {
  if ((taddr >> 16) != 0 || cols > B.tmem_live) fail("tcgen05.dealloc of columns that are not allocated");
  B.tmem_live -= cols;
}
static void tmem_range_check(unsigned col, unsigned n, const char* who) {
  const unsigned first = B.tmem_next - B.tmem_live;
  if (B.tmem_live == 0 || col < first || col + n > B.tmem_next) {
    fprintf(stderr, "emu: %s: columns [%u, %u) outside the allocation [%u, %u)\n", who, col, col + n, first, B.tmem_next);
    fail("tensor-memory access outside the allocated columns");
  }
}

// ---- tcgen05.mma.cta_group::1.kind::tf32 ----------------------------------------------------------------------------------
// Shared-memory matrix descriptor (PTX ISA, tcgen05 "Shared memory descriptor"): bits 0-13 start address >> 4, 16-29
// leading-dimension byte offset >> 4, 32-45 stride-dimension byte offset >> 4, 46-48 fixed 0b001, 49-51 base offset,
// 52 leading-dimension stride mode, 61-63 swizzle mode (2 = 128-byte swizzle).  K-major 128-byte swizzle: row r of the
// operand at start + (r / 8) SBO + (r % 8) 128 bytes, its K elements contiguous; the swizzle then XORs address bits [4:6]
// with bits [7:9] of the resulting address.
static void gather(uint64_t desc, unsigned rows, std::vector<float>& out) {
  const uint64_t start = (desc & 0x3fffu) << 4, sbo = ((desc >> 32) & 0x3fffu) << 4;
  const unsigned version = (unsigned)((desc >> 46) & 7u), base_off = (unsigned)((desc >> 49) & 7u);
  const unsigned lbo_mode = (unsigned)((desc >> 52) & 1u), layout = (unsigned)((desc >> 61) & 7u);
  if (version != 1 || base_off != 0 || lbo_mode != 0 || layout != 2)
    fail("tcgen05.mma: shared-memory descriptor is not version 1, SWIZZLE_128B, base offset 0");
  out.resize((size_t)rows * 8);
  for (unsigned r = 0; r < rows; ++r)
    for (unsigned k = 0; k < 8; ++k) {
      const uint64_t addr = start + (uint64_t)(r / 8) * sbo + (r % 8) * 128 + 4 * k;
      const uint64_t phys = addr ^ (((addr >> 7) & 7u) << 4);
      uint32_t bits;
      memcpy(&bits, dyn_at(phys, 4, "tcgen05.mma operand"), 4);
      bits &= 0xffffe000u;                  // TF32: the low 13 mantissa bits are not read
      memcpy(&out[(size_t)r * 8 + k], &bits, 4);
    }
}
// Instruction descriptor of .kind::tf32 (PTX ISA, "Instruction descriptor"): bits 0-2 sparsity, 3 saturate, 4-5 D type
// (1 = F32), 7-9 A type and 10-12 B type (2 = TF32), 13 / 14 negate A / B, 15 / 16 transpose A / B (0 = K-major), 17-22
// N >> 3, 24-28 M >> 4, 30-31 max shift.
void mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, unsigned accumulate) {
  const unsigned dtype = (idesc >> 4) & 3u, atype = (idesc >> 7) & 7u, btype = (idesc >> 10) & 7u;
  const unsigned n = ((idesc >> 17) & 63u) << 3, m = ((idesc >> 24) & 31u) << 4;
  if ((idesc & 0xfu) || dtype != 1 || atype != 2 || btype != 2 || ((idesc >> 13) & 0xfu) || (idesc >> 29))
    fail("tcgen05.mma: instruction descriptor is not dense TF32 x TF32 -> F32 with K-major A and B");
  if (m != 128 || n < 16 || n > 256 || n % 16) fail("tcgen05.mma: shape is not M = 128, N in [16, 256] with N % 16 == 0");
  if ((tmem_d >> 16) != 0) fail("tcgen05.mma: D does not start at lane 0 (M = 128 spans all lanes)");
  tmem_range_check(tmem_d & 0xffffu, n, "tcgen05.mma D");
  PendingMma p;
  p.desc_a = desc_a;
  p.desc_b = desc_b;
  p.col = tmem_d & 0xffffu;
  p.n = n;
  p.accumulate = accumulate != 0;
  gather(desc_a, 128, p.a);   // the snapshot of the operands as they are at issue
  gather(desc_b, n, p.b);
  B.mma.push_back(std::move(p));
}
// The MMAs run here, the latest moment the hardware may read their operands: operands that changed since issue were
// overwritten while the MMA was in flight (a stage refilled before the commit that frees it).
void mma_commit(uint64_t* bar) {
  std::vector<float> a, b;
  for (PendingMma& p : B.mma) {
    gather(p.desc_a, 128, a);
    gather(p.desc_b, p.n, b);
    if (memcmp(a.data(), p.a.data(), a.size() * 4) || memcmp(b.data(), p.b.data(), b.size() * 4))
      fail("tcgen05.mma: operand overwritten while the MMA was in flight");
    for (unsigned r = 0; r < 128; ++r) {
      float* d = &B.tmem[(size_t)r * kTmemCols + p.col];
      const float* ar = &p.a[(size_t)r * 8];
      for (unsigned j = 0; j < p.n; ++j) {
        const float* br = &p.b[(size_t)j * 8];
        float s = p.accumulate ? d[j] : 0.f;
        for (unsigned k = 0; k < 8; ++k) s += ar[k] * br[k];   // TF32 x TF32 is exact in fp32; fp32 accumulation
        d[j] = s;
      }
    }
  }
  B.mma.clear();
  mbar_arrive_one(bar, 0);   // .mbarrier::arrive::one, release
}
// tcgen05.ld.32x32b.x32: lane l of the warp reads 32 consecutive columns of tensor-memory lane (taddr.lane + l).  Warp w
// may only access lanes 32 (w % 4) .. + 31.
void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  const unsigned warp = B.cur >> 5, lane = B.cur & 31u, lane0 = taddr >> 16, col = taddr & 0xffffu;
  if (lane0 != 32 * (warp % 4)) {
    fprintf(stderr, "emu: tcgen05.ld: warp %u reads lanes [%u, %u), its quarter is [%u, %u)\n", warp, lane0, lane0 + 32,
            32 * (warp % 4), 32 * (warp % 4) + 32);
    fail("tcgen05.ld outside the warp's lane quarter");
  }
  tmem_range_check(col, 32, "tcgen05.ld");
  for (const PendingMma& p : B.mma)
    if (col < p.col + p.n && p.col < col + 32) fail("tcgen05.ld of columns whose MMAs are not committed");
  memcpy(r, &B.tmem[(size_t)(lane0 + lane) * kTmemCols + col], sizeof(r));
}

}  // namespace emu

// tests/test_emu_shuffle.py: switch the shuffled schedule on (seed != 0) or off from Python
extern "C" void d3h_emu_set_shuffle(unsigned long long seed) { emu::set_shuffle(seed); }

// tests/test_emu_mlp.py: a launch with `bytes` of dynamic shared memory and no attribute -> 1 if the runtime refused it
static void launch_probe_kernel() { emu::dyn_smem()[threadIdx.x] = 1; }
extern "C" int d3h_emu_launch_probe(unsigned long long bytes) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(1);
  cfg.blockDim = dim3(32);
  cfg.dynamicSmemBytes = bytes;
  cudaLaunchKernelEx(&cfg, launch_probe_kernel);
  return cudaGetLastError() != cudaSuccess ? 1 : 0;
}
