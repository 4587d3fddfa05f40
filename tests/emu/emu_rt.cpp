// Host-thread emulation runtime for the kernels in sopht_mpi_b200/csrc
// (TEST INFRASTRUCTURE ONLY; see sb200_rt.h).  Blocks run one after another;
// "coop" launches give every CUDA thread an OS thread so that __syncthreads and
// warp shuffles work; plain launches run the threads of a block sequentially.
// The OS threads of coop launches come from a pool that lives as long as the process: creating
// and destroying one thread per CUDA thread per block cost more than the kernels themselves.
// Every launch also records the kernel's address, so that a test can list which of the compiled
// kernel instantiations the process has run (sb200_emu_launched_kernels).
#define SB200_EMU 1
#include "sb200_rt.h"

#include <atomic>
#include <mutex>
#include <semaphore>
#include <set>

namespace sbemu {
thread_local uint3 t_threadIdx, t_blockIdx;
thread_local dim3 t_blockDim, t_gridDim;
thread_local BlockCtx* t_ctx = nullptr;
thread_local unsigned t_linear_tid = 0;

static std::mutex g_launched_mu;
static std::set<const void*> g_launched;

// Runs job(tid) for tid < n on n pool threads at once and returns when all have finished.  Each thread
// waits on a semaphore of its own, so a block wakes only the threads it uses.
class ThreadPool {
 public:
  void run(unsigned n, const std::function<void(unsigned)>& job) {
    std::lock_guard<std::mutex> lk(mu_);
    while (go_.size() < n) {
      go_.push_back(std::make_unique<std::binary_semaphore>(0));
      std::thread(&ThreadPool::worker, this, go_.back().get(), (unsigned)go_.size() - 1).detach();  // parked
    }
    job_ = &job;
    pending_.store(n);
    for (unsigned i = 0; i < n; ++i) go_[i]->release();
    done_.acquire();
  }

 private:
  void worker(std::binary_semaphore* go, unsigned id) {
    for (;;) {
      go->acquire();
      (*job_)(id);
      if (pending_.fetch_sub(1) == 1) done_.release();
    }
  }
  std::mutex mu_;  // one launch at a time
  std::vector<std::unique_ptr<std::binary_semaphore>> go_;
  const std::function<void(unsigned)>* job_ = nullptr;
  std::atomic<unsigned> pending_{0};
  std::binary_semaphore done_{0};
};

void note_launch(const void* kernel) {
  std::lock_guard<std::mutex> lk(g_launched_mu);
  g_launched.insert(kernel);
}

void launch(dim3 grid, dim3 block, size_t smem, bool coop, const std::function<void()>& body) {
  const unsigned nthreads = block.x * block.y * block.z;
  BlockCtx ctx;
  ctx.dyn_smem.resize(smem + 16);
  ctx.xchg.resize(nthreads);
  if (coop) {
    ctx.block_bar = std::make_unique<std::barrier<>>(nthreads);
    for (unsigned w = 0; w < (nthreads + 31) / 32; ++w) {
      unsigned cnt = std::min(32u, nthreads - w * 32);
      ctx.warp_bar.push_back(std::make_unique<std::barrier<>>(cnt));
    }
  }
  auto run_thread = [&](unsigned bx, unsigned by, unsigned bz, unsigned tid) {
    t_ctx = &ctx;
    t_linear_tid = tid;
    t_blockDim = block;
    t_gridDim = grid;
    t_blockIdx = uint3{bx, by, bz};
    t_threadIdx = uint3{tid % block.x, (tid / block.x) % block.y, tid / (block.x * block.y)};
    body();
  };
  static ThreadPool* pool = new ThreadPool();  // never destroyed: its threads are parked, not joined
  for (unsigned bz = 0; bz < grid.z; ++bz)
    for (unsigned by = 0; by < grid.y; ++by)
      for (unsigned bx = 0; bx < grid.x; ++bx) {
        if (!coop) {
          for (unsigned tid = 0; tid < nthreads; ++tid) run_thread(bx, by, bz, tid);
        } else {
          pool->run(nthreads, [&](unsigned tid) { run_thread(bx, by, bz, tid); });
        }
      }
}
}  // namespace sbemu

// Distinct kernel addresses launched so far in this process: writes up to `cap` of them to `out` and
// returns how many there are.
extern "C" int sb200_emu_launched_kernels(const void** out, int cap) {
  std::lock_guard<std::mutex> lk(sbemu::g_launched_mu);
  int i = 0;
  for (const void* k : sbemu::g_launched) {
    if (i < cap && out) out[i] = k;
    ++i;
  }
  return i;
}
