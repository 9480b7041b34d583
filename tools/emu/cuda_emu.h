// CPU warp emulation for the warp-synchronous kernels of epnn_b200 (test infrastructure, CPU only).
//
// A kernel source compiled with -DEPNN_CPU_EMU includes this header instead of epnn_internal.cuh.  Every lane of a warp
// is a host thread running the UNMODIFIED kernel body; the warp-level primitives the kernels use (__shfl_sync,
// __all_sync, __syncwarp) are implemented with a per-warp barrier, shared memory is a per-CTA host buffer, atomicAdd is
// a GCC atomic.  Inline PTX has to be replaced by the kernel source itself (#ifdef EPNN_CPU_EMU around its asm helpers).
// This checks indexing, control flow, shared-memory layout and the order of the arithmetic -- not performance.
#pragma once
#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdint>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "../../epnn_b200/csrc/epnn_consts.h"

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __grid_constant__
#define __align__(n)
#define __constant__
#define __shared__ static            /* statically sized shared arrays: one CTA runs at a time, its threads share the static */

struct alignas(16) float4 { float x, y, z, w; };
struct alignas(16) int4 { int x, y, z, w; };
struct alignas(8) float2 { float x, y; };
inline unsigned __float_as_uint(float f) { unsigned u; std::memcpy(&u, &f, 4); return u; }
inline float __uint_as_float(unsigned u) { float f; std::memcpy(&f, &u, 4); return f; }
struct alignas(16) ulonglong2 { unsigned long long x, y; };
struct int2 { int x, y; };
inline float4 make_float4(float x, float y, float z, float w) { float4 r; r.x = x; r.y = y; r.z = z; r.w = w; return r; }
inline int2 make_int2(int x, int y) { int2 r; r.x = x; r.y = y; return r; }
struct EmuDim3 { unsigned x = 0, y = 0, z = 0; };

struct EmuBarrier {                       // reusable barrier: the 32 lanes of a warp, or all threads of a CTA
    std::mutex m; std::condition_variable cv; int count = 0, gen = 0, parties = 32;
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        const int g = gen;
        if (++count == parties) { count = 0; ++gen; cv.notify_all(); }
        else cv.wait(lk, [&] { return gen != g; });
    }
};
struct EmuWarp { EmuBarrier bar; uint32_t xbuf[32]; };

inline thread_local EmuDim3 threadIdx, blockIdx, gridDim, blockDim;
inline thread_local EmuWarp* emu_warp = nullptr;
inline thread_local EmuBarrier* emu_cta_bar = nullptr;
inline thread_local float* emu_smem = nullptr;
#define EPNN_EMU_LANE ((int)(threadIdx.x & 31))

template <typename T> inline T __shfl_sync(unsigned, T v, int src) {
    static_assert(sizeof(T) == 4 || sizeof(T) == 8, "emulated shuffles move 32- or 64-bit values");
    T r;
    for (size_t h = 0; h < sizeof(T) / 4; ++h) {
        std::memcpy(&emu_warp->xbuf[EPNN_EMU_LANE], reinterpret_cast<const char*>(&v) + 4 * h, 4);
        emu_warp->bar.wait();
        std::memcpy(reinterpret_cast<char*>(&r) + 4 * h, &emu_warp->xbuf[src & 31], 4);
        emu_warp->bar.wait();
    }
    return r;
}
template <typename T> inline T __shfl_xor_sync(unsigned m, T v, int x) { return __shfl_sync(m, v, EPNN_EMU_LANE ^ x); }
// lanes whose source falls outside the warp keep their own value (CUDA semantics for width 32)
template <typename T> inline T __shfl_up_sync(unsigned m, T v, unsigned d) { const int src = EPNN_EMU_LANE - (int)d; return __shfl_sync(m, v, src >= 0 ? src : EPNN_EMU_LANE); }
template <typename T> inline T __shfl_down_sync(unsigned m, T v, unsigned d) { const int src = EPNN_EMU_LANE + (int)d; return __shfl_sync(m, v, src < 32 ? src : EPNN_EMU_LANE); }
inline int __all_sync(unsigned, int pred) {
    emu_warp->xbuf[EPNN_EMU_LANE] = pred ? 1u : 0u;
    emu_warp->bar.wait();
    int r = 1;
    for (int l = 0; l < 32; ++l) r &= (int)emu_warp->xbuf[l];
    emu_warp->bar.wait();
    return r;
}
inline unsigned __match_any_sync(unsigned, int key) {          // lanes holding the same key
    emu_warp->xbuf[EPNN_EMU_LANE] = (uint32_t)key;
    emu_warp->bar.wait();
    unsigned m = 0;
    for (int l = 0; l < 32; ++l) m |= (emu_warp->xbuf[l] == (uint32_t)key ? 1u : 0u) << l;
    emu_warp->bar.wait();
    return m;
}
inline unsigned __ballot_sync(unsigned, int pred) {
    emu_warp->xbuf[EPNN_EMU_LANE] = pred ? 1u : 0u;
    emu_warp->bar.wait();
    unsigned m = 0;
    for (int l = 0; l < 32; ++l) m |= emu_warp->xbuf[l] << l;
    emu_warp->bar.wait();
    return m;
}
inline void emu_allgather32(unsigned v, unsigned (&out)[32]) {     // every lane's 32-bit value, seen by every lane
    emu_warp->xbuf[EPNN_EMU_LANE] = v;
    emu_warp->bar.wait();
    for (int l = 0; l < 32; ++l) out[l] = emu_warp->xbuf[l];
    emu_warp->bar.wait();
}
// mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 (D = A B + D) with the PTX fragment layout: g = lane >> 2, t = lane & 3,
// a0 (g, t) a1 (g + 8, t) a2 (g, t + 4) a3 (g + 8, t + 4); b0 (k = t, n = g) b1 (k = t + 4, n = g);
// d0 (g, 2t) d1 (g, 2t + 1) d2 (g + 8, 2t) d3 (g + 8, 2t + 1).  TF32 inputs: the low 13 mantissa bits are ignored.
inline void emu_mma_m16n8k8_tf32(float (&d)[4], const unsigned (&a)[4], const unsigned (&b)[2]) {
    unsigned A[4][32], B[2][32];
    for (int r = 0; r < 4; ++r) emu_allgather32(a[r] & 0xFFFFE000u, A[r]);
    for (int r = 0; r < 2; ++r) emu_allgather32(b[r] & 0xFFFFE000u, B[r]);
    const int g = EPNN_EMU_LANE >> 2, t = EPNN_EMU_LANE & 3;
    for (int i = 0; i < 4; ++i) {
        const int row = g + 8 * (i >> 1), col = 2 * t + (i & 1);
        float acc = d[i];
        for (int k = 0; k < 8; ++k) {
            float av, bv;
            std::memcpy(&av, &A[(row >= 8) + 2 * (k >= 4)][4 * (row & 7) + (k & 3)], 4);
            std::memcpy(&bv, &B[k >= 4][4 * col + (k & 3)], 4);
            acc = std::fmaf(av, bv, acc);
        }
        d[i] = acc;
    }
}
inline int __ffs(unsigned x) { return __builtin_ffs((int)x); }
inline int __popc(unsigned x) { return __builtin_popcount(x); }
inline int __any_sync(unsigned m, int pred) { return __ballot_sync(m, pred) != 0u; }
inline void __syncwarp() { emu_warp->bar.wait(); }
inline void __syncthreads() { emu_cta_bar->wait(); }
inline int atomicAdd(int* p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline int atomicMin(int* p, int v) {
    int old = __atomic_load_n(p, __ATOMIC_SEQ_CST);
    while (v < old && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) {}
    return old;
}
template <typename T> inline T __ldg(const T* p) { return *p; }
using std::max;
using std::min;
// round-to-nearest arithmetic intrinsics (compile the emulation with -ffp-contract=off: no fused contraction either)
inline double __dadd_rn(double a, double b) { return a + b; }
inline double __dsub_rn(double a, double b) { return a - b; }
inline double __dmul_rn(double a, double b) { return a * b; }
inline double __ddiv_rn(double a, double b) { return a / b; }
inline double __dsqrt_rn(double a) { return std::sqrt(a); }
inline double rsqrt(double a) { return 1.0 / std::sqrt(a); }     // the device's FP64 rsqrt is within 1 ulp of this
inline float __fdiv_rn(float a, float b) { return a / b; }
inline float __double2float_rn(double a) { return (float)a; }

// Runs a kernel WITHOUT warp-level primitives or shared memory (the one-thread-per-item prep kernels): every thread of
// the grid is executed sequentially on the calling host thread.
template <typename F> inline void emu_launch_simple(int grid, int block, F kernel) {
    gridDim.x = (unsigned)grid; blockDim.x = (unsigned)block;
    for (int b = 0; b < grid; ++b)
        for (int t = 0; t < block; ++t) { blockIdx.x = (unsigned)b; threadIdx.x = (unsigned)t; kernel(); }
}

// Runs `kernel(args...)` for one CTA of `n_warps` warps (all warps concurrently, 32 host threads each).
// emu_launch_grid runs the CTAs of a grid one after the other.
template <typename F> inline void emu_launch_cta(int n_warps, size_t smem_floats, F kernel, int block = 0, int grid = 1) {
    std::vector<float> smem(smem_floats, 0.f);
    std::vector<EmuWarp> warps(n_warps);
    EmuBarrier cta;
    cta.parties = n_warps * 32;
    std::vector<std::thread> th;
    for (int t = 0; t < n_warps * 32; ++t)
        th.emplace_back([&, t] {
            threadIdx.x = (unsigned)t; blockIdx.x = (unsigned)block; gridDim.x = (unsigned)grid; blockDim.x = (unsigned)(n_warps * 32);
            emu_warp = &warps[t >> 5];
            emu_cta_bar = &cta;
            emu_smem = smem.data();
            kernel();
        });
    for (auto& x : th) x.join();
}
template <typename F> inline void emu_launch_grid(int grid, int n_warps, size_t smem_floats, F kernel) {
    for (int b = 0; b < grid; ++b) emu_launch_cta(n_warps, smem_floats, kernel, b, grid);
}
