// SIMT-on-CPU shim: compiles the warp-synchronous CUDA kernels of this directory (mlp_persistent.cu + mlp_v2.inc) with
// g++ and runs them with one OS thread per CUDA thread, so that the CPU test-suite executes the *same source* the GPU
// runs — the flagship persistent-MLP kernel included (tests only; never used to train).
//
//   thread block      one block at a time; blockDim.x*y*z std::threads per launch walk the blocks together
//   __syncthreads()   std::barrier over the live threads of the block (a thread that returns from the kernel drops out,
//                     like an exited CUDA thread)
//   __shfl_*_sync()   per-warp exchange slots between two warp barriers (all 32 lanes of a warp must take part, which
//                     is also what the kernels assume on the device)
//   __shared__        function-local static (blocks run one after the other; contents are as undefined between blocks
//                     as real shared memory); dynamic shared memory: COLEARN_DYN_SMEM -> a per-block heap buffer
//   ld.acquire / st.release .sys   __atomic builtins
//   thread-block cluster   launch_cluster: the blocks of one cluster run concurrently; cluster barrier, peer shared memory and
//                     the st.async + mbarrier transaction count (mlp_generic.cu) — see the section above launch_cluster
//   kernel<<<g, b, s, stream>>>(args)   COLEARN_LAUNCH(kernel, g, b, s, stream, args) -> colearn_shim::launch(...)
//
// Include this header BEFORE the kernel source and define COLEARN_HOST_SHIM.
#pragma once
#include <cuda_runtime.h>   // under g++ the CUDA qualifiers (__device__, __global__, __forceinline__, ...) are harmless

#include <math.h>
#include <stdint.h>
#include <string.h>

#include <barrier>
#include <chrono>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#undef __shared__
#define __shared__ static
#ifndef __launch_bounds__
#define __launch_bounds__(...)
#endif

namespace colearn_shim {

struct Dim3 {
  unsigned x = 1, y = 1, z = 1;
  Dim3() = default;
  Dim3(unsigned x_, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
  Dim3(const dim3& d) : x(d.x), y(d.y), z(d.z) {}       // NOLINT: launch sites pass dim3 or plain ints
  unsigned count() const { return x * y * z; }
};

struct Block {
  explicit Block(int n, size_t smem_bytes) : nthreads(n), bar(n), dyn((smem_bytes + 63) / 4 + 16, 0.f) {
    for (int w = 0; w < (n + 31) / 32; ++w) {
      const int lanes = (w * 32 + 32 <= n) ? 32 : n - w * 32;
      warp_bar.emplace_back(std::make_unique<std::barrier<>>(lanes));
    }
    slots.assign((size_t)((n + 31) / 32) * 32, 0ull);
  }
  int nthreads;
  Dim3 block_idx, block_dim, grid_dim;
  std::barrier<> bar;
  std::vector<std::unique_ptr<std::barrier<>>> warp_bar;
  std::vector<unsigned long long> slots;   // one 8-byte exchange slot per lane
  std::vector<float> dyn;                  // dynamic shared memory (16-byte aligned start, see dyn_smem())
  // per-block scratch outside shared memory (the tcgen05 model keeps the CTA's tensor memory here)
  float* scratch(size_t n) {
    std::call_once(scratch_once, [&] { scratch_buf.assign(n, 0.f); });
    return scratch_buf.data();
  }
  std::once_flag scratch_once;
  std::vector<float> scratch_buf;
};

inline thread_local Dim3 t_threadIdx;
inline thread_local unsigned t_linear = 0;               // threadIdx.x + threadIdx.y * blockDim.x + ...: warps are formed from it
inline thread_local Block* t_block = nullptr;

inline float* dyn_smem() {
  uintptr_t p = reinterpret_cast<uintptr_t>(t_block->dyn.data());
  return reinterpret_cast<float*>((p + 15) & ~(uintptr_t)15);
}

inline void syncthreads() { t_block->bar.arrive_and_wait(); }
inline void syncwarp() { t_block->warp_bar[t_linear / 32]->arrive_and_wait(); }

template <class T>
inline T shfl_from(T v, int src_lane) {
  static_assert(sizeof(T) <= 8, "shuffle payload");
  Block* b = t_block;
  const int w = t_linear / 32, l = t_linear % 32;
  unsigned long long bits = 0;
  memcpy(&bits, &v, sizeof(T));
  b->slots[(size_t)w * 32 + l] = bits;
  b->warp_bar[w]->arrive_and_wait();
  const unsigned long long got = b->slots[(size_t)w * 32 + (src_lane & 31)];
  b->warp_bar[w]->arrive_and_wait();
  T r;
  memcpy(&r, &got, sizeof(T));
  return r;
}

// all 32 lanes' values of one warp (for the reductions that have no shuffle form)
template <class T>
inline void warp_gather(T v, T (&out)[32]) {
  Block* b = t_block;
  const int w = t_linear / 32, l = t_linear % 32;
  unsigned long long bits = 0;
  memcpy(&bits, &v, sizeof(T));
  b->slots[(size_t)w * 32 + l] = bits;
  b->warp_bar[w]->arrive_and_wait();
  const int lanes = (w * 32 + 32 <= b->nthreads) ? 32 : b->nthreads - w * 32;
  for (int i = 0; i < 32; ++i) {
    T r{};
    if (i < lanes) memcpy(&r, &b->slots[(size_t)w * 32 + i], sizeof(T));
    out[i] = r;
  }
  b->warp_bar[w]->arrive_and_wait();
}

// Runs `body()` once per CUDA thread, block after block (x fastest, like the hardware's linear block order).  The OS
// threads are created once per launch and walk the blocks together: between two blocks they meet at `next`, whose
// completion step replaces the Block object (fresh barriers: threads that exited early in one block take part again).
template <class F>
inline void launch(Dim3 grid, Dim3 block, size_t smem_bytes, F&& body) {
  const unsigned nthreads = block.count();
  const unsigned long long nblocks = (unsigned long long)grid.x * grid.y * grid.z;
  if (nthreads == 0 || nblocks == 0) return;
  std::unique_ptr<Block> cur;
  unsigned long long next_b = 0;
  auto advance = [&]() noexcept {
    if (next_b < nblocks) {
      cur = std::make_unique<Block>((int)nthreads, smem_bytes);
      cur->block_idx = Dim3{(unsigned)(next_b % grid.x), (unsigned)((next_b / grid.x) % grid.y), (unsigned)(next_b / ((unsigned long long)grid.x * grid.y))};
      cur->block_dim = block;
      cur->grid_dim = grid;
    } else {
      cur.reset();
    }
    ++next_b;
  };
  advance();
  std::barrier next((std::ptrdiff_t)nthreads, advance);
  std::vector<std::thread> threads;
  threads.reserve(nthreads);
  for (unsigned t = 0; t < nthreads; ++t)
    threads.emplace_back([&, t] {
      t_linear = t;
      t_threadIdx = Dim3{t % block.x, (t / block.x) % block.y, t / (block.x * block.y)};
      for (;;) {
        Block* blk = cur.get();
        if (blk == nullptr) break;
        t_block = blk;
        body();
        // an exited thread no longer takes part in this block's barriers (CUDA semantics)
        blk->bar.arrive_and_drop();
        blk->warp_bar[t / 32]->arrive_and_drop();
        next.arrive_and_wait();
      }
    });
  for (auto& th : threads) th.join();
}

// ---- thread-block clusters (mlp_generic.cu) ------------------------------------------------------------------------------------
// launch_cluster runs the `cluster` blocks of one cluster CONCURRENTLY (cluster x blockDim OS threads; clusters one after the
// other), so that blocks can wait for each other.  Distributed shared memory: the same offset in the peer block's `dyn` buffer.
// mbarrier (transaction-count form): the 8-byte word holds {int32 count, uint32 phase}; count starts at ARRIVE (one pending
// arrival), expect_tx / complete_tx add and subtract bytes, and the operation that brings it to zero re-arms it and flips the
// phase (release), which try_wait.parity observes (acquire).
struct Cluster {
  std::vector<std::unique_ptr<Block>> blocks;
  std::unique_ptr<std::barrier<>> bar;
};
inline thread_local Cluster* t_cluster = nullptr;
inline thread_local int t_cluster_rank = 0;
constexpr int32_t kMbarArrive = 1 << 24;

inline int cluster_rank() { return t_cluster_rank; }
inline void cluster_sync() { t_cluster->bar->arrive_and_wait(); }
inline float* dyn_base(Block* b) {
  uintptr_t p = reinterpret_cast<uintptr_t>(b->dyn.data());
  return reinterpret_cast<float*>((p + 15) & ~(uintptr_t)15);
}
template <class T>
inline T* peer_ptr(T* local, int peer) {
  const ptrdiff_t off = reinterpret_cast<char*>(local) - reinterpret_cast<char*>(dyn_smem());
  return reinterpret_cast<T*>(reinterpret_cast<char*>(dyn_base(t_cluster->blocks[(size_t)peer].get())) + off);
}
inline void mbar_init(uint64_t* bar) {
  int32_t* w = reinterpret_cast<int32_t*>(bar);
  __atomic_store_n(w, kMbarArrive, __ATOMIC_RELAXED);
  __atomic_store_n(reinterpret_cast<uint32_t*>(w + 1), 0u, __ATOMIC_RELEASE);
}
inline void mbar_add(uint64_t* bar, int32_t delta) {
  int32_t* w = reinterpret_cast<int32_t*>(bar);
  if (__atomic_add_fetch(w, delta, __ATOMIC_SEQ_CST) == 0) {
    __atomic_store_n(w, kMbarArrive, __ATOMIC_RELAXED);
    __atomic_fetch_xor(reinterpret_cast<uint32_t*>(w + 1), 1u, __ATOMIC_RELEASE);
  }
}
// st.async of one float into the peer's copy of `local` + complete_tx(4) on the peer's copy of `bar`
inline void push_to_peer(float* local, float v, int peer, uint64_t* bar) {
  *peer_ptr(local, peer) = v;
  mbar_add(peer_ptr(bar, peer), -4);
}
inline void mbar_wait(uint64_t* bar, uint32_t parity, uint32_t bytes, bool arrive) {
  if (arrive) mbar_add(bar, (int32_t)bytes - kMbarArrive);
  const uint32_t* phase = reinterpret_cast<const uint32_t*>(bar) + 1;
  while ((__atomic_load_n(phase, __ATOMIC_ACQUIRE) & 1u) == (parity & 1u)) std::this_thread::yield();
}

template <class F>
inline void launch_cluster(Dim3 grid, unsigned cluster, Dim3 block, size_t smem_bytes, F&& body) {
  const unsigned nthreads = block.count();
  if (nthreads == 0 || grid.x == 0 || cluster == 0) return;
  for (unsigned c0 = 0; c0 < grid.x; c0 += cluster) {
    Cluster cl;
    for (unsigned r = 0; r < cluster; ++r) {
      cl.blocks.emplace_back(std::make_unique<Block>((int)nthreads, smem_bytes));
      Block& b = *cl.blocks.back();
      b.block_idx = Dim3{c0 + r};
      b.block_dim = block;
      b.grid_dim = grid;
    }
    cl.bar = std::make_unique<std::barrier<>>((std::ptrdiff_t)(nthreads * cluster));
    std::vector<std::thread> threads;
    threads.reserve(nthreads * cluster);
    for (unsigned r = 0; r < cluster; ++r)
      for (unsigned t = 0; t < nthreads; ++t)
        threads.emplace_back([&, r, t] {
          t_linear = t;
          t_threadIdx = Dim3{t % block.x, (t / block.x) % block.y, t / (block.x * block.y)};
          t_block = cl.blocks[r].get();
          t_cluster = &cl;
          t_cluster_rank = (int)r;
          body();
          t_block->bar.arrive_and_drop();
          t_block->warp_bar[t / 32]->arrive_and_drop();
          cl.bar->arrive_and_drop();
          t_cluster = nullptr;
        });
    for (auto& th : threads) th.join();
  }
}

}  // namespace colearn_shim

#define threadIdx (::colearn_shim::t_threadIdx)
#define blockIdx (::colearn_shim::t_block->block_idx)
#define blockDim (::colearn_shim::t_block->block_dim)
#define gridDim (::colearn_shim::t_block->grid_dim)

inline void __syncthreads() { ::colearn_shim::syncthreads(); }
inline void __syncwarp(unsigned = 0xffffffffu) { ::colearn_shim::syncwarp(); }
template <class T>
inline T __shfl_xor_sync(unsigned, T v, int lane_mask, int = 32) {
  return ::colearn_shim::shfl_from(v, (int)(::colearn_shim::t_linear % 32) ^ lane_mask);
}
template <class T>
inline T __shfl_sync(unsigned, T v, int src_lane, int = 32) {
  return ::colearn_shim::shfl_from(v, src_lane);
}
template <class T>
inline T __shfl_down_sync(unsigned, T v, unsigned delta, int = 32) {
  const int l = (int)(::colearn_shim::t_linear % 32);
  return ::colearn_shim::shfl_from(v, l + (int)delta < 32 ? l + (int)delta : l);
}
inline int __reduce_add_sync(unsigned, int v) {
  int all[32];
  ::colearn_shim::warp_gather(v, all);
  int s = 0;
  for (int i = 0; i < 32; ++i) s += all[i];
  return s;
}
template <class T>
inline T __ldcs(const T* p) { return *p; }
inline float __uint_as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }
inline unsigned __float_as_uint(float f) { unsigned u; memcpy(&u, &f, 4); return u; }
// atomics (threads of a block are real OS threads here)
inline float atomicAdd(float* p, float v) {
  unsigned* up = reinterpret_cast<unsigned*>(p);
  unsigned old = __atomic_load_n(up, __ATOMIC_RELAXED), want;
  do { want = __float_as_uint(__uint_as_float(old) + v); } while (!__atomic_compare_exchange_n(up, &old, want, false, __ATOMIC_SEQ_CST, __ATOMIC_RELAXED));
  return __uint_as_float(old);
}
inline int atomicAdd(int* p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline unsigned atomicAdd(unsigned* p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline unsigned atomicExch(unsigned* p, unsigned v) { return __atomic_exchange_n(p, v, __ATOMIC_SEQ_CST); }
inline unsigned atomicOr(unsigned* p, unsigned v) { return __atomic_fetch_or(p, v, __ATOMIC_SEQ_CST); }
inline int __popc(unsigned v) { return __builtin_popcount(v); }
template <class T>
inline T __ldg(const T* p) { return *p; }
template <class T>
inline T __ldcg(const T* p) { return *p; }
inline float __expf(float x) { return expf(x); }
inline float __logf(float x) { return logf(x); }
inline float __frcp_rn(float x) { return 1.0f / x; }
inline float __fdividef(float a, float b) { return a / b; }
inline void __nanosleep(unsigned) { std::this_thread::yield(); }
inline void __threadfence() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
inline void __threadfence_system() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
inline void __threadfence_block() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }

// runtime calls the launchers make: nothing to configure on the host
#define cudaFuncSetAttribute(...) cudaSuccess
#define cudaGetDevice(p) (*(p) = 0, cudaSuccess)
#define cudaDeviceGetAttribute(p, attr, dev) (*(p) = 4, cudaSuccess)   /* "4 SMs": persistent kernels walk several tiles per CTA */
#define cudaGetLastError() cudaSuccess
#define cudaMemsetAsync(ptr, value, bytes, stream) (memset((ptr), (value), (bytes)), cudaSuccess)
#define cudaMemset(ptr, value, bytes) (memset((ptr), (value), (bytes)), cudaSuccess)

#undef COLEARN_NOINLINE
#define COLEARN_NOINLINE
#define COLEARN_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(::colearn_shim::dyn_smem())
#define COLEARN_DYN_SMEM_UNALIGNED(type, name) COLEARN_DYN_SMEM(type, name)
#define COLEARN_LAUNCH(kernel, grid, block, smem, stream, ...) \
  ::colearn_shim::launch(::colearn_shim::Dim3(grid), ::colearn_shim::Dim3(block), (size_t)(smem), [&] { kernel(__VA_ARGS__); })
#define COLEARN_KERNEL_NAME(...) __VA_ARGS__
