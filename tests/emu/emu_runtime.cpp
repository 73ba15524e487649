// TEST INFRASTRUCTURE -- runtime of the host warp emulator (see tests/emu/cuda_runtime.h).
//
// Every CUDA thread of a block is a fiber with its own stack; the fibers of one block are scheduled
// round-robin on one OS thread and give up the processor only at synchronisation points.  Blocks
// of a grid are distributed over a pool of OS threads (global atomics are real atomics).  Kernel
// launches are synchronous, so stream order is trivially respected.
#include <cuda_runtime.h>

#include <execinfo.h>
#include <signal.h>
#include <ucontext.h>
#include <sys/mman.h>
#include <unistd.h>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <string>
#include <algorithm>
#include <thread>
#include <vector>

#if !defined(__x86_64__)
#error "the host warp emulator switches fibers with x86-64 assembly"
#endif

thread_local uint3 threadIdx, blockIdx;
thread_local dim3 blockDim, gridDim;

// the dynamic shared memory of the kernels: `extern __shared__ double sm[]` / `srec[]` inside
// namespace gwi name these objects (one block at a time per OS thread)
namespace gwi {
constexpr size_t EMU_SMEM_DOUBLES = 232448 / 8;
alignas(16) thread_local double sm[EMU_SMEM_DOUBLES];
alignas(16) thread_local double srec[EMU_SMEM_DOUBLES];
}  // namespace gwi

// void gwi_emu_switch(void** save_sp, void* load_sp): save the callee-saved registers on the current
// stack, store the stack pointer, continue on the other stack
extern "C" void gwi_emu_switch(void** save_sp, void* load_sp);
asm(R"(
.pushsection .text
.globl gwi_emu_switch
.type gwi_emu_switch,@function
gwi_emu_switch:
  pushq %rbp
  pushq %rbx
  pushq %r12
  pushq %r13
  pushq %r14
  pushq %r15
  movq %rsp, (%rdi)
  movq %rsi, %rsp
  popq %r15
  popq %r14
  popq %r13
  popq %r12
  popq %rbx
  popq %rbp
  ret
.size gwi_emu_switch,.-gwi_emu_switch
.popsection
)");

namespace gwi_emu {

constexpr size_t STACK_BYTES = 256 * 1024;

// A completed barrier is published to the waiting fibers only at the start of the scheduler's next
// sweep (gen = gen_next), and the fiber that completed it waits like the others: between two
// synchronisation points the lanes of a warp therefore always run in lane order 0..31, whatever the
// warp did before -- the emulation is deterministic even when blocks race for work items.
struct PartialBarrier {  // __syncwarp(mask) with a proper subset of the lanes
  unsigned mask = 0;
  uint64_t gen = 0, gen_next = 0;
  unsigned arrived = 0;
};
struct Warp {
  uint64_t gen = 0, gen_next = 0;
  int arrived = 0, alive = 0;
  unsigned alive_mask = 0;
  PartialBarrier partial[4];
  uint64_t xbuf[2][32];
  unsigned ballot[4] = {0, 0, 0, 0};
};

struct Fiber {
  void* sp = nullptr;
  char* stack = nullptr;
  uint3 tid{0, 0, 0};
  bool done = true;
  const uint64_t* wait_ptr = nullptr;  // blocked while *wait_ptr == wait_val
  uint64_t wait_val = 0;
  unsigned xchg_count = 0;
  Warp* warp = nullptr;
};

struct NamedBarrier {  // bar.sync id, n
  uint64_t gen = 0, gen_next = 0;
  int arrived = 0;
};
struct Block {
  std::vector<Fiber> fibers;
  std::vector<Warp> warps;
  NamedBarrier named[16];
  uint64_t gen = 0, gen_next = 0;
  int arrived = 0, alive = 0;
  void* sched_sp = nullptr;
  Fiber* current = nullptr;
  Body* body = nullptr;
};

static thread_local Block* t_block = nullptr;

static void release_warp_if_complete(Warp& w) {
  if (w.alive > 0 && w.arrived == w.alive) {
    w.arrived = 0;
    ++w.gen_next;
  }
}
static void release_block_if_complete(Block& b) {
  if (b.alive > 0 && b.arrived == b.alive) {
    b.arrived = 0;
    ++b.gen_next;
  }
}

static void yield_to_scheduler() {
  Block& b = *t_block;
  Fiber* f = b.current;
  gwi_emu_switch(&f->sp, b.sched_sp);
}

void warp_barrier() {
  Block& b = *t_block;
  Fiber* f = b.current;
  Warp& w = *f->warp;
  if (++w.arrived == w.alive) {
    w.arrived = 0;
    ++w.gen_next;
  }
  f->wait_ptr = &w.gen;
  f->wait_val = w.gen;
  yield_to_scheduler();
}

void warp_yield() { yield_to_scheduler(); }  // stays runnable: resumed on the next sweep

unsigned warp_alive_mask() { return t_block->current->warp->alive_mask; }

void warp_barrier_mask(unsigned mask) {
  Block& b = *t_block;
  Fiber* f = b.current;
  Warp& w = *f->warp;
  mask &= w.alive_mask;
  PartialBarrier* pb = nullptr;
  for (auto& c : w.partial)
    if (c.mask == mask && c.arrived != 0) pb = &c;  // a barrier of this lane set is already forming
  if (!pb)
    for (auto& c : w.partial)
      if (c.arrived == 0 && c.gen == c.gen_next) {
        pb = &c;
        pb->mask = mask;
        break;
      }
  if (!pb) {
    std::fprintf(stderr, "gwi_emu: more than 4 concurrent partial-mask __syncwarp barriers in one warp\n");
    std::abort();
  }
  pb->arrived |= 1u << (f->tid.x & 31u);
  if (pb->arrived == mask) {
    pb->arrived = 0;
    ++pb->gen_next;
  }
  f->wait_ptr = &pb->gen;
  f->wait_val = pb->gen;
  yield_to_scheduler();
}

void named_barrier(int id, int n_threads) {
  Block& b = *t_block;
  Fiber* f = b.current;
  if (id < 0 || id > 15 || n_threads <= 0) {
    std::fprintf(stderr, "gwi_emu: bad named barrier (%d, %d)\n", id, n_threads);
    std::abort();
  }
  NamedBarrier& nb = b.named[id];
  if (++nb.arrived == n_threads) {
    nb.arrived = 0;
    ++nb.gen_next;
  }
  f->wait_ptr = &nb.gen;
  f->wait_val = nb.gen;
  yield_to_scheduler();
}

void block_barrier() {
  Block& b = *t_block;
  Fiber* f = b.current;
  if (++b.arrived == b.alive) {
    b.arrived = 0;
    ++b.gen_next;
  }
  f->wait_ptr = &b.gen;
  f->wait_val = b.gen;
  yield_to_scheduler();
}

// double-buffered: the buffer written by exchange k is read before any lane can pass the barrier of
// exchange k+1, so exchange k+2 may overwrite it
uint64_t warp_exchange(uint64_t mine, int from) {
  Fiber* f = t_block->current;
  Warp& w = *f->warp;
  const unsigned k = f->xchg_count++;
  const unsigned par = k & 1u;
  w.xbuf[par][f->tid.x & 31u] = mine;
  warp_barrier();
  w.ballot[(k + 2u) & 3u] = 0;  // see warp_ballot: every exchange operation keeps the ballot slots clean
  return w.xbuf[par][from];
}

// Exchange operation k of a warp (shuffle or ballot) owns ballot[k & 3].  A lane that has passed
// barrier k knows that every lane has finished operation k-1, and none can be past barrier k+1, so
// slot (k+2) & 3 is free to be cleared for its next use.  Lanes that have exited contribute 0.
unsigned warp_ballot(bool pred) {
  Fiber* f = t_block->current;
  Warp& w = *f->warp;
  const unsigned k = f->xchg_count++;
  if (pred) w.ballot[k & 3u] |= 1u << (f->tid.x & 31u);
  warp_barrier();
  const unsigned r = w.ballot[k & 3u];
  w.ballot[(k + 2u) & 3u] = 0;
  return r;
}

extern "C" void gwi_emu_fiber_main() {
  Block& b = *t_block;
  Fiber* f = b.current;
  b.body->run();
  f->done = true;
  // a finished thread no longer takes part in barriers
  Warp& w = *f->warp;
  --w.alive;
  w.alive_mask &= ~(1u << (f->tid.x & 31u));
  release_warp_if_complete(w);
  --b.alive;
  release_block_if_complete(b);
  gwi_emu_switch(&f->sp, b.sched_sp);
  std::fprintf(stderr, "gwi_emu: finished fiber resumed\n");
  std::abort();
}

static void prepare_fiber(Fiber& f) {
  // stack image popped by gwi_emu_switch: r15 r14 r13 r12 rbx rbp | return address | (alignment)
  uintptr_t top = (uintptr_t)(f.stack + STACK_BYTES) & ~(uintptr_t)15;
  uint64_t* s = reinterpret_cast<uint64_t*>(top);
  *--s = 0;                                   // fake return address of gwi_emu_fiber_main: rsp % 16 == 8 at its entry
  *--s = (uint64_t)(uintptr_t)&gwi_emu_fiber_main;
  for (int i = 0; i < 6; ++i) *--s = 0;
  f.sp = s;
}

// fiber stacks are recycled between launches (a fresh mapping would page-fault on every first touch)
static std::mutex g_stack_mutex;
static std::vector<char*> g_free_stacks;

static bool lane_order_reversed() {
  static const bool r = [] {
    const char* e = std::getenv("GWI_EMU_LANE_ORDER");
    return e && std::string(e) == "reverse";
  }();
  return r;
}

struct Worker {
  Block block;
  std::vector<char*> stacks;
  ~Worker() {
    std::lock_guard<std::mutex> lock(g_stack_mutex);
    for (char* s : stacks) g_free_stacks.push_back(s);
  }
  void run_block(dim3 grid, dim3 bdim, uint3 bidx, Body& body) {
    const int n = (int)(bdim.x * bdim.y * bdim.z);
    Block& b = block;
    if ((int)stacks.size() < n) {
      std::lock_guard<std::mutex> lock(g_stack_mutex);
      while ((int)stacks.size() < n && !g_free_stacks.empty()) {
        stacks.push_back(g_free_stacks.back());
        g_free_stacks.pop_back();
      }
    }
    while ((int)stacks.size() < n) {
      void* p = mmap(nullptr, STACK_BYTES, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
      if (p == MAP_FAILED) {
        std::fprintf(stderr, "gwi_emu: cannot allocate a fiber stack\n");
        std::abort();
      }
      stacks.push_back((char*)p);
    }
    b.fibers.assign(n, Fiber());
    b.warps.assign((n + 31) / 32, Warp());
    b.gen = b.gen_next = 0;
    for (auto& nb : b.named) nb = NamedBarrier();
    b.arrived = 0;
    b.alive = n;
    b.body = &body;
    for (int i = 0; i < n; ++i) {
      Fiber& f = b.fibers[i];
      f.stack = stacks[i];
      f.tid = uint3{(unsigned)i % bdim.x, ((unsigned)i / bdim.x) % bdim.y, (unsigned)i / (bdim.x * bdim.y)};
      f.done = false;
      f.warp = &b.warps[i / 32];
      f.warp->alive++;
      f.warp->alive_mask |= 1u << (i & 31);
      prepare_fiber(f);
    }
    for (auto& w : b.warps) std::memset(w.xbuf, 0, sizeof(w.xbuf));
    t_block = &b;
    blockIdx = bidx;
    blockDim = bdim;
    gridDim = grid;
    int remaining = n;
    while (remaining > 0) {
      bool progress = b.gen != b.gen_next;
      b.gen = b.gen_next;
      for (auto& w : b.warps) {
        progress = progress || w.gen != w.gen_next;
        w.gen = w.gen_next;
        for (auto& c : w.partial) {
          progress = progress || c.gen != c.gen_next;
          c.gen = c.gen_next;
        }
      }
      for (auto& nb : b.named) {
        progress = progress || nb.gen != nb.gen_next;
        nb.gen = nb.gen_next;
      }
      for (int ii = 0; ii < n; ++ii) {
        // GWI_EMU_LANE_ORDER=reverse: lanes of a warp run 31..0 between synchronisation points (a result
        // that depends on the lane order beyond atomic-add rounding points at a missing barrier)
        const int i = lane_order_reversed() ? (ii & ~31) + std::min(31, n - 1 - (ii & ~31)) - (ii & 31) : ii;
        if (i < 0 || i >= n) continue;
        Fiber& f = b.fibers[i];
        if (f.done) continue;
        if (f.wait_ptr) {
          if (*f.wait_ptr == f.wait_val) continue;
          f.wait_ptr = nullptr;
        }
        b.current = &f;
        threadIdx = f.tid;
        gwi_emu_switch(&b.sched_sp, f.sp);
        progress = true;
        if (f.done) --remaining;
      }
      if (!progress) {
        std::fprintf(stderr, "gwi_emu: deadlock in block (%u,%u,%u): %d threads wait at a barrier the others never reach\n", bidx.x, bidx.y, bidx.z, remaining);
        std::abort();
      }
    }
    t_block = nullptr;
  }
};

static int pool_size() {
  static const int n = [] {
    const char* e = std::getenv("GWI_EMU_THREADS");
    int v = e ? std::atoi(e) : (int)std::thread::hardware_concurrency();
    return v < 1 ? 1 : (v > 64 ? 64 : v);
  }();
  return n;
}

}  // namespace gwi_emu

// a captured stream: the recorded operations, replayed in order by cudaGraphLaunch
struct gwi_emu_graph {
  std::vector<std::function<void()>> ops;
};
static thread_local gwi_emu_graph* t_capture = nullptr;

namespace gwi_emu {

static void run_grid_now(dim3 grid, dim3 block, size_t dyn_smem, Body& body);

void run_grid(dim3 grid, dim3 block, size_t dyn_smem, std::shared_ptr<Body> body) {
  if (t_capture) {
    t_capture->ops.push_back([=]() { run_grid_now(grid, block, dyn_smem, *body); });
    return;
  }
  run_grid_now(grid, block, dyn_smem, *body);
}

static void run_grid_now(dim3 grid, dim3 block, size_t dyn_smem, Body& body) {
  if (dyn_smem > gwi::EMU_SMEM_DOUBLES * 8) {
    std::fprintf(stderr, "gwi_emu: %zu bytes of dynamic shared memory requested\n", dyn_smem);
    std::abort();
  }
  const long total = (long)grid.x * grid.y * grid.z;
  static const bool trace = std::getenv("GWI_EMU_TRACE") != nullptr;
  if (trace) std::fprintf(stderr, "gwi_emu: launch grid (%u,%u,%u) block (%u,%u,%u) dynamic shared %zu B\n", grid.x, grid.y, grid.z, block.x, block.y, block.z, dyn_smem);
  if (total <= 0) return;
  std::atomic<long> next{0};
  auto work = [&]() {
    Worker w;
    for (;;) {
      const long i = next.fetch_add(1);
      if (i >= total) break;
      const uint3 bidx{(unsigned)(i % grid.x), (unsigned)((i / grid.x) % grid.y), (unsigned)(i / ((long)grid.x * grid.y))};
      w.run_block(grid, block, bidx, body);
    }
  };
  const int nthreads = (int)std::min<long>(pool_size(), total);
  if (nthreads <= 1) {
    work();
    return;
  }
  std::vector<std::thread> th;
  for (int t = 0; t < nthreads; ++t) th.emplace_back(work);
  for (auto& t : th) t.join();
}

}  // namespace gwi_emu

// ---- the runtime API -----------------------------------------------------------------------------
struct gwi_emu_stream {
  int dummy;
};
struct gwi_emu_event {
  std::chrono::steady_clock::time_point t;
};

// GWI_EMU_DEBUG=1: print a native backtrace on SIGSEGV (fibers run on their own stacks, so the
// handler gets an alternate stack)
static void segv_handler(int sig, siginfo_t* info, void* ucv) {
  ucontext_t* uc = (ucontext_t*)ucv;
  void* frames[64];
  frames[0] = (void*)uc->uc_mcontext.gregs[REG_RIP];
  char msg[160];
  const int len = std::snprintf(msg, sizeof(msg), "gwi_emu: fatal signal %d, fault address %p, rsp %p, instruction:\n", sig, info->si_addr,
                                (void*)uc->uc_mcontext.gregs[REG_RSP]);
  if (write(2, msg, len) < 0) _exit(3);
  backtrace_symbols_fd(frames, 1, 2);
  // words on top of the faulting stack (return addresses among them)
  void** sp = (void**)uc->uc_mcontext.gregs[REG_RSP];
  backtrace_symbols_fd(sp, 24, 2);
  _exit(128 + sig);
}
static void install_debug_handler() {
  static bool done = false;
  if (done || !std::getenv("GWI_EMU_DEBUG")) return;
  done = true;
  static char alt[1 << 16];
  stack_t ss{};
  ss.ss_sp = alt;
  ss.ss_size = sizeof(alt);
  sigaltstack(&ss, nullptr);
  struct sigaction sa{};
  sa.sa_sigaction = segv_handler;
  sa.sa_flags = SA_ONSTACK | SA_SIGINFO;
  sigaction(SIGSEGV, &sa, nullptr);
  sigaction(SIGBUS, &sa, nullptr);
}

extern "C" {

int gwi_emu_marker(void) {
  install_debug_handler();
  return 1;
}

cudaError_t cudaGetDeviceCount(int* n) {
  *n = 1;
  return cudaSuccess;
}
cudaError_t cudaSetDevice(int d) { return d == 0 ? cudaSuccess : cudaErrorInvalidValue; }
cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) {
  std::memset(p, 0, sizeof(*p));
  std::snprintf(p->name, sizeof(p->name), "gwi host warp emulator");
  const char* e = std::getenv("GWI_EMU_SMS");
  p->multiProcessorCount = e ? std::max(1, std::atoi(e)) : 4;
  p->sharedMemPerBlockOptin = 232448;
  return cudaSuccess;
}
cudaError_t cudaMalloc(void** p, size_t bytes) {
  void* q = nullptr;
  if (posix_memalign(&q, 256, bytes ? bytes : 1) != 0) return cudaErrorMemoryAllocation;
  *p = q;
  return cudaSuccess;
}
cudaError_t cudaFree(void* p) {
  std::free(p);
  return cudaSuccess;
}
cudaError_t cudaMallocHost(void** p, size_t bytes) { return cudaMalloc(p, bytes); }
cudaError_t cudaFreeHost(void* p) { return cudaFree(p); }
cudaError_t cudaMemcpy(void* dst, const void* src, size_t bytes, int) {
  std::memmove(dst, src, bytes);
  return cudaSuccess;
}
cudaError_t cudaMemcpyAsync(void* dst, const void* src, size_t bytes, int kind, cudaStream_t) {
  if (t_capture) {
    t_capture->ops.push_back([=]() { std::memmove(dst, src, bytes); });
    return cudaSuccess;
  }
  return cudaMemcpy(dst, src, bytes, kind);
}
cudaError_t cudaStreamBeginCapture(cudaStream_t, int) {
  if (t_capture) return cudaErrorInvalidValue;
  t_capture = new gwi_emu_graph();
  return cudaSuccess;
}
cudaError_t cudaStreamEndCapture(cudaStream_t, cudaGraph_t* graph) {
  if (!t_capture) return cudaErrorInvalidValue;
  *graph = t_capture;
  t_capture = nullptr;
  return cudaSuccess;
}
cudaError_t cudaGraphInstantiate(cudaGraphExec_t* exec, cudaGraph_t graph, unsigned long long) {
  *exec = new gwi_emu_graph(*graph);
  return cudaSuccess;
}
cudaError_t cudaGraphLaunch(cudaGraphExec_t exec, cudaStream_t) {
  for (auto& op : exec->ops) op();
  return cudaSuccess;
}
cudaError_t cudaGraphDestroy(cudaGraph_t graph) {
  delete graph;
  return cudaSuccess;
}
cudaError_t cudaGraphExecDestroy(cudaGraphExec_t exec) {
  delete exec;
  return cudaSuccess;
}
cudaError_t cudaMemset(void* p, int v, size_t bytes) {
  std::memset(p, v, bytes);
  return cudaSuccess;
}
cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) {
  *s = new gwi_emu_stream{0};
  return cudaSuccess;
}
cudaError_t cudaStreamDestroy(cudaStream_t s) {
  delete s;
  return cudaSuccess;
}
cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
cudaError_t cudaEventCreate(cudaEvent_t* e) {
  *e = new gwi_emu_event{std::chrono::steady_clock::now()};
  return cudaSuccess;
}
cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { return cudaEventCreate(e); }
cudaError_t cudaEventDestroy(cudaEvent_t e) {
  delete e;
  return cudaSuccess;
}
cudaError_t cudaEventRecord(cudaEvent_t e, cudaStream_t) {
  e->t = std::chrono::steady_clock::now();
  return cudaSuccess;
}
cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t a, cudaEvent_t b) {
  *ms = std::chrono::duration<float, std::milli>(b->t - a->t).count();
  return cudaSuccess;
}
cudaError_t cudaDeviceSynchronize(void) { return cudaSuccess; }
cudaError_t cudaGetLastError(void) { return cudaSuccess; }
cudaError_t cudaFuncSetAttribute(const void*, int, int) { return cudaSuccess; }
const char* cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : "emulated CUDA runtime error"; }

}  // extern "C"
