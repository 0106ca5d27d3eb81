// cuda_host_emu.h — TEST INFRASTRUCTURE: a warp-level CUDA execution model on the CPU, so that the product's kernel
// sources (openea_b200/csrc/*.cu, compiled unchanged with -DOEA_HOST_EMU by g++) can be checked against the oracle
// where no GPU exists.  Not a fallback: nothing under openea_b200/ ever loads a library built with it.
//
// Model: one OS thread per CUDA thread (a worker pool reused from block to block).  All warps of a block run concurrently; the 32 lanes of a warp meet at every
// warp collective (__shfl*_sync, __ballot_sync, __match_any_sync, __syncwarp) on a per-mask rendezvous of their warp —
// exactly where real lanes exchange registers — and nowhere else (lanes are free-running, so code that silently relies
// on a converged warp staying in step is caught); __syncthreads() is a real barrier; the blocks of a grid run one after
// another, so static __shared__ storage is per block as on the device; a kernel with a grid barrier
// (cooperative_groups::this_grid().sync()) is launched as ONE block, whose barrier then is the grid's.
// "Device" pointers are host pointers; atomics and red adds are real atomics (std::atomic_ref).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

// stream-ordered runtime calls the entry points make between launches: "device" memory is host memory and launches are
// synchronous, so they are plain memset / memcpy
#define cudaMemsetAsync(P, V, N, ST) (memset((P), (V), (N)), cudaSuccess)
#define cudaMemcpyAsync(D, S, N, KIND, ST) (memcpy((D), (S), (N)), cudaSuccess)
#define cudaStreamSynchronize(ST) (cudaSuccess)
#define cudaFuncSetAttribute(...) (cudaSuccess)
// An emulated kernel is a host function the real runtime does not know.  Asking the real runtime about it fails, and on
// a machine with a GPU that failure would stay as the last error of the CUDA runtime the process shares with torch.
// Answer with the one resident block per SM the grid sizing falls back to.
#define cudaOccupancyMaxActiveBlocksPerMultiprocessor(N, ...) (*(N) = 1, cudaSuccess)
/* launches and copies are synchronous and in program order: stream / event ordering is already satisfied */
#define cudaStreamWaitEvent(...) (cudaSuccess)
#define cudaEventRecord(...) (cudaSuccess)
#define cudaEventSynchronize(...) (cudaSuccess)

#undef __shared__
#define __shared__ static
#undef __launch_bounds__
#define __launch_bounds__(...)

struct EmuDim3 { unsigned x = 0, y = 0, z = 0; };
inline thread_local EmuDim3 threadIdx, blockIdx;
inline EmuDim3 gridDim, blockDim;

#define _COOPERATIVE_GROUPS_H_          /* keep <cooperative_groups.h> out: it needs nvcc */
namespace cooperative_groups {
struct grid_group { void sync() const; };      // OEA_LAUNCH_COOPERATIVE runs such kernels as ONE block: its barrier is the grid's
inline grid_group this_grid() { return {}; }
}  // namespace cooperative_groups

namespace emu {

struct Rendezvous {
    std::atomic<int> arrived{0};
    std::atomic<unsigned> generation{0};
};
// collective state of ONE warp: a rendezvous per participation mask and the 32 exchange slots
struct WarpState {
    std::mutex map_mutex;
    std::map<unsigned, Rendezvous> rendezvous;
    uint64_t slot[32];
};
// __syncthreads() of a block
struct BlockBarrier {
    int expected = 0;
    std::atomic<int> arrived{0};
    std::atomic<unsigned> generation{0};
    void wait() {
        const unsigned gen = generation.load();
        if (arrived.fetch_add(1) + 1 == expected) {
            arrived.store(0);
            generation.fetch_add(1);
        } else {
            while (generation.load() == gen) std::this_thread::yield();
        }
    }
};
inline thread_local WarpState* t_warp = nullptr;           // set by launch() for every thread of the grid
inline thread_local BlockBarrier* t_block = nullptr;
inline thread_local int t_lane = 0;

inline Rendezvous& rendezvous_of(unsigned mask) {
    std::lock_guard<std::mutex> lk(t_warp->map_mutex);
    return t_warp->rendezvous[mask];
}
// all lanes named in `mask` meet here
inline void sync(unsigned mask) {
    Rendezvous& r = rendezvous_of(mask);
    const int expected = __builtin_popcount(mask);
    const unsigned gen = r.generation.load();
    if (r.arrived.fetch_add(1) + 1 == expected) {
        r.arrived.store(0);
        r.generation.fetch_add(1);
    } else {
        while (r.generation.load() == gen) std::this_thread::yield();
    }
}
template <typename T>
inline void publish(T v) {
    static_assert(sizeof(T) <= 8, "exchange slot is 64 bits");
    uint64_t bits = 0;
    memcpy(&bits, &v, sizeof(T));
    t_warp->slot[t_lane] = bits;
}
template <typename T>
inline T peek(int lane) {
    T v;
    memcpy(&v, &t_warp->slot[lane], sizeof(T));
    return v;
}

template <typename Body>
inline void launch_row(int grid, int threads, Body body);

// run `body` as a (1- or 2-dimensional) grid of blocks of block.x threads (a multiple of 32)
template <typename Body>
inline void launch(dim3 grid, dim3 block, Body body) {
    gridDim.y = grid.y;
    for (unsigned y = 0; y < grid.y; ++y) {
        blockIdx.y = y;
        launch_row((int)grid.x, (int)block.x, [&, y] { blockIdx.y = y; body(); });
    }
}

// The CUDA threads of a block run on a pool of worker threads that lives for the process: one block at a time, all of its
// threads concurrently (they meet at barriers), workers reused by the next block and the next launch.
class BlockPool {
public:
    template <typename Job>
    void run(int n, Job&& job) {
        std::lock_guard<std::mutex> serial(run_mutex_);
        {
            std::unique_lock<std::mutex> lk(m_);
            while ((int)workers_ < n) {
                const int id = workers_++;
                std::thread([this, id] { work(id); }).detach();
            }
            job_ = job;
            active_ = n;
            done_ = 0;
            ++generation_;
        }
        start_.notify_all();
        std::unique_lock<std::mutex> lk(m_);
        finished_.wait(lk, [&] { return done_ == active_; });
    }

private:
    void work(int id) {
        uint64_t seen = 0;
        for (;;) {
            std::function<void(int)> job;
            {
                std::unique_lock<std::mutex> lk(m_);
                start_.wait(lk, [&] { return generation_ != seen; });
                seen = generation_;
                if (id >= active_) continue;
                job = job_;
            }
            job(id);
            std::lock_guard<std::mutex> lk(m_);
            if (++done_ == active_) finished_.notify_all();
        }
    }
    std::mutex m_, run_mutex_;
    std::condition_variable start_, finished_;
    std::function<void(int)> job_;
    uint64_t generation_ = 0;
    int workers_ = 0, active_ = 0, done_ = 0;
};
inline BlockPool& block_pool() {
    static BlockPool* pool = new BlockPool();       // never destroyed: its detached workers outlive static destruction
    return *pool;
}

template <typename Body>
inline void launch_row(int grid, int threads, Body body) {
    gridDim.x = (unsigned)grid;
    blockDim.x = (unsigned)threads;
    const int warps = threads / 32;
    const unsigned by = blockIdx.y;                        // the launching thread's value: workers have their own copy
    for (int b = 0; b < grid; ++b) {
        std::vector<WarpState> ws(warps);
        BlockBarrier bar;
        bar.expected = threads;
        block_pool().run(threads, [&](int t) {
            t_lane = t & 31;
            t_warp = &ws[t >> 5];
            t_block = &bar;
            threadIdx.x = (unsigned)t;
            blockIdx.x = (unsigned)b;
            blockIdx.y = by;
            body();
        });
    }
}

}  // namespace emu

// ---- warp collectives ------------------------------------------------------------------------------------------------
template <typename T>
inline T __shfl_xor_sync(unsigned mask, T v, int lane_mask) {
    emu::publish(v);
    emu::sync(mask);
    const T r = emu::peek<T>((emu::t_lane ^ lane_mask) & 31);
    emu::sync(mask);
    return r;
}
template <typename T>
inline T __shfl_sync(unsigned mask, T v, int src) {
    emu::publish(v);
    emu::sync(mask);
    const T r = emu::peek<T>(src & 31);
    emu::sync(mask);
    return r;
}
template <typename T>
inline T __shfl_up_sync(unsigned mask, T v, unsigned delta) {
    emu::publish(v);
    emu::sync(mask);
    const int src = emu::t_lane - (int)delta;
    const T r = src >= 0 ? emu::peek<T>(src) : v;         // lanes below delta keep their own value
    emu::sync(mask);
    return r;
}
template <typename T>
inline T __shfl_down_sync(unsigned mask, T v, unsigned delta) {
    emu::publish(v);
    emu::sync(mask);
    const int src = emu::t_lane + (int)delta;
    const T r = src < 32 ? emu::peek<T>(src) : v;
    emu::sync(mask);
    return r;
}
inline unsigned __ballot_sync(unsigned mask, bool pred) {
    emu::publish<unsigned>(pred ? 1u : 0u);
    emu::sync(mask);
    unsigned out = 0;
    for (int l = 0; l < 32; ++l)
        if (((mask >> l) & 1u) && emu::peek<unsigned>(l)) out |= 1u << l;
    emu::sync(mask);
    return out;
}
template <typename T>
inline unsigned __match_any_sync(unsigned mask, T v) {
    emu::publish(v);
    emu::sync(mask);
    unsigned out = 0;
    for (int l = 0; l < 32; ++l)
        if (((mask >> l) & 1u) && emu::peek<T>(l) == v) out |= 1u << l;
    emu::sync(mask);
    return out;
}
inline void __syncthreads() { emu::t_block->wait(); }
inline void cooperative_groups::grid_group::sync() const { __syncthreads(); }
inline void __syncwarp(unsigned mask = 0xffffffffu) { emu::sync(mask); }     // lanes are threads: a real rendezvous

// ---- loads, atomics, intrinsics ----------------------------------------------------------------------------------------
template <typename T>
inline T __ldg(const T* p) { return *p; }
template <typename T>
inline T emu_atomic_rmw(T* p, T (*op)(T, T), T v) {
    std::atomic_ref<T> a(*p);
    T old = a.load(std::memory_order_relaxed);
    while (!a.compare_exchange_weak(old, op(old, v), std::memory_order_relaxed)) {}
    return old;
}
inline double atomicAdd(double* p, double v) { return emu_atomic_rmw<double>(p, [](double a, double b) { return a + b; }, v); }
inline unsigned atomicAdd(unsigned* p, unsigned v) { return std::atomic_ref<unsigned>(*p).fetch_add(v); }
inline int atomicAdd(int* p, int v) { return std::atomic_ref<int>(*p).fetch_add(v); }
inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { return std::atomic_ref<unsigned long long>(*p).fetch_add(v); }
inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) {
    return emu_atomic_rmw<unsigned long long>(p, [](unsigned long long a, unsigned long long b) { return a > b ? a : b; }, v);
}
inline unsigned atomicMax(unsigned* p, unsigned v) { return emu_atomic_rmw<unsigned>(p, [](unsigned a, unsigned b) { return a > b ? a : b; }, v); }
inline int atomicMax(int* p, int v) { return emu_atomic_rmw<int>(p, [](int a, int b) { return a > b ? a : b; }, v); }
inline float atomicAdd(float* p, float v) {          // lanes of one warp may hit the same word (scatter-adds): really atomic
    std::atomic_ref<float> a(*p);
    float old = a.load(std::memory_order_relaxed);
    while (!a.compare_exchange_weak(old, old + v, std::memory_order_relaxed)) {}
    return old;
}
inline unsigned long long atomicCAS(unsigned long long* p, unsigned long long expected, unsigned long long desired) {
    std::atomic_ref<unsigned long long> a(*p);
    a.compare_exchange_strong(expected, desired);
    return expected;                                  // the value found at *p, as CUDA's atomicCAS returns
}
using std::min;
using std::max;
inline int __ffs(int x) { return __builtin_ffs(x); }
inline int __popc(unsigned x) { return __builtin_popcount(x); }
inline int __clz(int x) { return x == 0 ? 32 : __builtin_clz((unsigned)x); }
inline unsigned __float_as_uint(float f) { unsigned u; memcpy(&u, &f, 4); return u; }
inline float __uint_as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }
inline int __float_as_int(float f) { int i; memcpy(&i, &f, 4); return i; }
inline float __int_as_float(int i) { float f; memcpy(&f, &i, 4); return f; }
inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((uint64_t)a * (uint64_t)b) >> 32); }
inline float rsqrtf(float x) { return 1.0f / sqrtf(x); }
inline float emu_expf(float x) { return expf(x); }
#define __expf emu_expf
