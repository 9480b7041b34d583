// Electrostatics of a packed batch of point charges (epnn_electrostatics, include/epnn_b200.h): potential phi_i at every atom,
// E_s = 1/2 sum_i q_i phi_i and the dipole mu_s = sum_i q_i (x_i - c_s) of every system, all in FP64 after the float32
// coordinates are loaded.  A pair (i, j) of one system is included when r_ij > 0 (this also drops i == j) and, with
// fragment labels, when the labels differ.  Without labels the target label is -1 and every source label 0, so the label
// test always passes and there is a single code path.
//
// Every ordered pair is evaluated once from each side and no result is accumulated with atomics: every sum has a fixed
// order, so the outputs are bitwise repeatable and a system's outputs do not depend on the other systems of the call.
//   - systems of at most ELST_SMALL_MAX atoms: one warp per system; lane l owns the targets l and l + 32, the sources are
//     read from shared memory in index order; E and mu are xor-butterfly warp sums (every lane ends with the same bits).
//   - larger systems: a pair CTA owns a tile of ELST_TILE targets (one per thread) and streams a range of sources through
//     shared memory in tiles of ELST_TILE.  A system with too few target tiles to fill the GPU has its source range split
//     into parts (elst_parts: a function of n and the SM count); each part writes its partial potentials to a workspace
//     row.  One reduction CTA per system then adds the parts in order and forms E and mu with a fixed-order block sum.
#ifdef EPNN_CPU_EMU
#include "../../tools/emu/cuda_emu.h"      // CPU warp emulation (tests/test_emu_elst.py): same kernel bodies, lanes = host threads
#else
#include "epnn_internal.cuh"
#endif
#include "epnn_elst.cuh"

struct alignas(16) ElstSrc { double x, y, z, q; };

// phi contribution of m sources held in shared memory to the target (xi, yi, zi) with label fi, in source order.
__device__ __forceinline__ double elst_sum(double xi, double yi, double zi, int fi, const ElstSrc* src, const int* lab, int m,
                                           double acc) {
#pragma unroll 4
    for (int j = 0; j < m; ++j) {
        const ElstSrc s = src[j];
        const double dx = xi - s.x, dy = yi - s.y, dz = zi - s.z;
        const double r2 = dx * dx + dy * dy + dz * dz;
        const bool in = r2 > 0.0 && fi != lab[j];                 // selects instead of a branch: the unrolled pairs interleave
        acc += (in ? s.q : 0.0) * rsqrt(in ? r2 : 1.0);
    }
    return acc;
}

__device__ __forceinline__ double elst_warp_sum(double v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(ELST_WARPS * 32) elst_small_kernel(const ElstArgs a) {
    __shared__ ElstSrc src[ELST_WARPS][ELST_SMALL_MAX];
    __shared__ int lab[ELST_WARPS][ELST_SMALL_MAX];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * ELST_WARPS + w;
    if (s >= a.n_sys) return;
    const int a0 = a.off[s] - a.base, n = a.off[s + 1] - a.off[s];
    if (n > ELST_SMALL_MAX) return;                              // warp-uniform: large systems take the pair kernel
    ElstSrc* S = src[w];
    int* L = lab[w];
    for (int k = lane; k < n; k += 32) {
        const int i = a0 + k;
        S[k] = ElstSrc{(double)a.xyz[3 * i], (double)a.xyz[3 * i + 1], (double)a.xyz[3 * i + 2], a.q[i]};
        L[k] = a.frag ? a.frag[i] : 0;
    }
    __syncwarp();
    double e = 0.0, cx = 0.0, cy = 0.0, cz = 0.0;
    for (int k = lane; k < n; k += 32) {
        const ElstSrc t = S[k];
        const double phi = elst_sum(t.x, t.y, t.z, a.frag ? L[k] : -1, S, L, n, 0.0);
        if (a.phi) a.phi[a0 + k] = phi;
        e += t.q * phi;
        cx += t.x; cy += t.y; cz += t.z;
    }
    e = elst_warp_sum(e);
    cx = elst_warp_sum(cx) / n; cy = elst_warp_sum(cy) / n; cz = elst_warp_sum(cz) / n;
    double mx = 0.0, my = 0.0, mz = 0.0;
    for (int k = lane; k < n; k += 32) {
        const ElstSrc t = S[k];
        mx += t.q * (t.x - cx); my += t.q * (t.y - cy); mz += t.q * (t.z - cz);
    }
    mx = elst_warp_sum(mx); my = elst_warp_sum(my); mz = elst_warp_sum(mz);
    if (lane == 0) {
        if (a.energy) a.energy[s] = 0.5 * e;
        if (a.dipole) { a.dipole[3 * s] = mx; a.dipole[3 * s + 1] = my; a.dipole[3 * s + 2] = mz; }
    }
}

__global__ void __launch_bounds__(ELST_TILE) elst_pair_kernel(const ElstArgs a) {
    __shared__ ElstSrc src[ELST_TILE];
    __shared__ int lab[ELST_TILE];
    const ElstItem it = a.items[blockIdx.x];
    const int t = it.t0 + (int)threadIdx.x;
    const int ti = it.a0 + (t < it.n ? t : it.n - 1);            // threads past the end compute a copy and write nothing
    const double xi = a.xyz[3 * ti], yi = a.xyz[3 * ti + 1], zi = a.xyz[3 * ti + 2];
    const int fi = a.frag ? a.frag[ti] : -1;
    double acc = 0.0;
    for (int j0 = it.s0; j0 < it.s1; j0 += ELST_TILE) {
        const int m = it.s1 - j0 < ELST_TILE ? it.s1 - j0 : ELST_TILE;
        __syncthreads();                                          // the previous tile has been read by every thread
        if ((int)threadIdx.x < m) {
            const int j = it.a0 + j0 + (int)threadIdx.x;
            src[threadIdx.x] = ElstSrc{(double)a.xyz[3 * j], (double)a.xyz[3 * j + 1], (double)a.xyz[3 * j + 2], a.q[j]};
            lab[threadIdx.x] = a.frag ? a.frag[j] : 0;
        }
        __syncthreads();
        acc = elst_sum(xi, yi, zi, fi, src, lab, m, acc);
    }
    if (t < it.n) a.partial[it.pw + t] = acc;
}

// Sum over the CTA of four values in a fixed order (butterfly in each warp, then the warp totals in warp order); every
// thread returns the totals.
__device__ __forceinline__ void elst_block_sum(double (&v)[4], double (*red)[4]) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int k = 0; k < 4; ++k) v[k] = elst_warp_sum(v[k]);
    if (lane == 0)
        for (int k = 0; k < 4; ++k) red[w][k] = v[k];
    __syncthreads();
    for (int k = 0; k < 4; ++k) {
        double s = 0.0;
        for (int u = 0; u < ELST_RED / 32; ++u) s += red[u][k];
        v[k] = s;
    }
    __syncthreads();                                              // red is reused by the next call
}

__global__ void __launch_bounds__(ELST_RED) elst_reduce_kernel(const ElstArgs a) {
    __shared__ double red[ELST_RED / 32][4];
    const ElstSys S = a.sys[blockIdx.x];
    double v[4] = {0.0, 0.0, 0.0, 0.0};                           // sum q phi, sum x, sum y, sum z
    for (int k = threadIdx.x; k < S.n; k += ELST_RED) {
        double phi = 0.0;
        for (int p = 0; p < S.parts; ++p) phi += a.partial[S.pofs + (long long)p * S.n + k];
        const int i = S.a0 + k;
        if (a.phi) a.phi[i] = phi;
        v[0] += a.q[i] * phi;
        v[1] += (double)a.xyz[3 * i]; v[2] += (double)a.xyz[3 * i + 1]; v[3] += (double)a.xyz[3 * i + 2];
    }
    elst_block_sum(v, red);
    const double e = 0.5 * v[0], cx = v[1] / S.n, cy = v[2] / S.n, cz = v[3] / S.n;
    double m[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k = threadIdx.x; k < S.n; k += ELST_RED) {
        const int i = S.a0 + k;
        const double qi = a.q[i];
        m[0] += qi * ((double)a.xyz[3 * i] - cx); m[1] += qi * ((double)a.xyz[3 * i + 1] - cy); m[2] += qi * ((double)a.xyz[3 * i + 2] - cz);
    }
    elst_block_sum(m, red);
    if (threadIdx.x == 0) {
        if (a.energy) a.energy[S.s] = e;
        if (a.dipole) { a.dipole[3 * S.s] = m[0]; a.dipole[3 * S.s + 1] = m[1]; a.dipole[3 * S.s + 2] = m[2]; }
    }
}

// ---- potential (and field) at given points (epnn_potential_points) ---------------------------------------------------
// A CTA owns up to ELST_PT_TILE points of one system (one per thread) and streams one source part of that system's atoms
// through shared memory in tiles of ELST_PT_TILE, in index order.  The parts are fixed slices of ELST_PT_PART atoms, so a
// point's sums depend only on the point, its system's atoms and charges: not on the other points, the chunking or the GPU.
// FIELD adds E = sum_j q_j (p - x_j) / r^3; phi-only calls do not carry its accumulators.
template <bool FIELD>
__global__ void __launch_bounds__(ELST_PT_TILE) elst_point_kernel(const ElstPtArgs a) {
    __shared__ ElstSrc src[ELST_PT_TILE];
    const ElstPtItem it = a.items[blockIdx.x];
    const int t = (int)threadIdx.x;
    const long long pi = it.p0 + (t < it.np ? t : it.np - 1);    // threads past the end compute a copy and write nothing
    const double px = a.pts[3 * pi], py = a.pts[3 * pi + 1], pz = a.pts[3 * pi + 2];
    double phi = 0.0, ex = 0.0, ey = 0.0, ez = 0.0;
    for (int j0 = it.s0; j0 < it.s1; j0 += ELST_PT_TILE) {
        const int m = it.s1 - j0 < ELST_PT_TILE ? it.s1 - j0 : ELST_PT_TILE;
        __syncthreads();                                          // the previous tile has been read by every thread
        if (t < m) {
            const int j = it.a0 + j0 + t;
            src[t] = ElstSrc{(double)a.xyz[3 * j], (double)a.xyz[3 * j + 1], (double)a.xyz[3 * j + 2], a.q[j]};
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < m; ++k) {
            const ElstSrc s = src[k];
            const double dx = px - s.x, dy = py - s.y, dz = pz - s.z;
            const double r2 = dx * dx + dy * dy + dz * dz;
            const bool in = r2 > 0.0;                             // selects instead of a branch, as in elst_sum
            const double rinv = rsqrt(in ? r2 : 1.0), qr = (in ? s.q : 0.0) * rinv;
            phi += qr;
            if (FIELD) {
                const double w = qr * rinv * rinv;
                ex += w * dx; ey += w * dy; ez += w * dz;
            }
        }
    }
    if (t >= it.np) return;
    const long long i = it.p0 + t;
    if (it.pw < 0) {
        if (a.phi) a.phi[i] = phi;
        if (FIELD) { a.field[3 * i] = ex; a.field[3 * i + 1] = ey; a.field[3 * i + 2] = ez; }
    } else if (FIELD) {
        double* w = a.partial + 4 * (it.pw + t);
        w[0] = phi; w[1] = ex; w[2] = ey; w[3] = ez;
    } else {
        a.partial[it.pw + t] = phi;
    }
}

// Adds the parts of the points of a split system in part order.
template <bool FIELD>
__global__ void __launch_bounds__(ELST_PT_TILE) elst_point_reduce_kernel(const ElstPtArgs a) {
    const ElstPtRed r = a.red[blockIdx.x];
    const int t = (int)threadIdx.x;
    if (t >= r.np) return;
    constexpr int W = FIELD ? 4 : 1;
    double v[W];
    for (int k = 0; k < W; ++k) v[k] = 0.0;
    for (int p = 0; p < r.parts; ++p) {
        const double* w = a.partial + W * (r.pw + (long long)p * r.stride + t);
        for (int k = 0; k < W; ++k) v[k] += w[k];
    }
    const long long i = r.p0 + t;
    if (a.phi) a.phi[i] = v[0];
    if (FIELD) { a.field[3 * i] = v[1 % W]; a.field[3 * i + 1] = v[2 % W]; a.field[3 * i + 2] = v[3 % W]; }
}

#ifndef EPNN_CPU_EMU
cudaError_t launch_elst(const ElstArgs& a, int n_items, int n_large, cudaStream_t st) {
    if (a.n_sys > 0) elst_small_kernel<<<div_up(a.n_sys, ELST_WARPS), ELST_WARPS * 32, 0, st>>>(a);
    if (n_items > 0) elst_pair_kernel<<<n_items, ELST_TILE, 0, st>>>(a);
    if (n_large > 0) elst_reduce_kernel<<<n_large, ELST_RED, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_elst_points(const ElstPtArgs& a, int n_items, int n_red, cudaStream_t st) {
    if (a.field) {
        if (n_items > 0) elst_point_kernel<true><<<n_items, ELST_PT_TILE, 0, st>>>(a);
        if (n_red > 0) elst_point_reduce_kernel<true><<<n_red, ELST_PT_TILE, 0, st>>>(a);
    } else {
        if (n_items > 0) elst_point_kernel<false><<<n_items, ELST_PT_TILE, 0, st>>>(a);
        if (n_red > 0) elst_point_reduce_kernel<false><<<n_red, ELST_PT_TILE, 0, st>>>(a);
    }
    return cudaGetLastError();
}
#endif   // !EPNN_CPU_EMU
