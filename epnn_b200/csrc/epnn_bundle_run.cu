// GNN bundle kernel, "row-run" mapping (FP32 default since round 2; option "pair_const" = 2).
//
// Message passing for SMALL systems (n <= SMALL_MAX), replaces reference charge_gn.py:62-70 (GNN_layer.call, one step):
//     S_i = sum over ALL columns j of i's system (near, far, self, + the weighted pad pseudo-column) of
//           relu(W2^T relu(u_i + v_j [+ C^T e_ij]) + b2)
// Same arithmetic per slot as the other bundle kernels; what changes is how the slots map onto the warp and how the
// row sums are formed (round-1 ncu: the warp-tile kernel is bound by the shared-memory operand traffic of tile_gemm,
// 44 % FMA pipe; the pair-per-thread "const" kernel by its 32 x 33 transpose + serial add chain at 8 warps/SM, 25 %):
//   * the slots of a bundle form two row-sorted lists: the CSR entries (ordered near pairs: col / pid / local row) and
//     the far list (ordered e == 0 columns or one weighted slot per species, + the pad slot);
//   * a list of L slots is cut into 32 CONTIGUOUS runs of J = ceil(L / 32) slots, ONE RUN PER LANE.  A lane walks its run
//     slot by slot; u_i stays in registers while the row does not change, the slot's 32 outputs are added into the lane's
//     own 32 row-sum accumulators -- no transpose, no shuffles, no per-slot shared-memory write;
//   * the weights are a __grid_constant__ parameter: every lane needs the same weight at the same time, ptxas turns them
//     into uniform-register operands of FFMA2 (no shared-memory operand traffic);
//   * row sums reach the warp's S rows (shared memory) in a fixed order without atomics: a row that ENDS inside a lane's
//     run is flushed by that lane at the slot where it ends (at most one such lane per row); the run's last row, which may
//     continue in the next lanes, is flushed after the loop in rounds -- lanes holding the same row go one after the other
//     in lane order (__match_any_sync).  Every addition has a fixed position -> bitwise reproducible.
// Shared memory per warp: v rows (+ the pad row b1) 7.1 KB, S rows 6.1 KB, pad weights: 13.4 KB -> 16 warps per SM.
// The second layer runs as two halves of 16 outputs so that u (32) + z (32) + row sums (32) + 16 accumulators fit 128
// registers.
#ifdef EPNN_CPU_EMU
#include "../../tools/emu/cuda_emu.h"      // CPU warp emulation (tests/test_emu_bundle_run.py): same kernel body, lanes = host threads
#else
#include "epnn_internal.cuh"
#endif

#ifndef RUN_NW
#define RUN_NW 8                        // warps per CTA
#endif
#ifndef RUN_UNROLL
#define RUN_UNROLL 1
#endif
constexpr int kRunUnroll = RUN_UNROLL;     // unroll factor of the slot loop (2 makes ptxas rotate 8 uniform quads instead of 2, but spills 4 KB: stays 1)
#ifndef RUN_CTAS
#define RUN_CTAS 2                      // CTAs per SM (16 warps per SM: 128 registers per thread)
#endif
#ifndef RUN_FULL
#define RUN_HALVES 1                    // second layer as two halves of 16 outputs (fits 128 registers; ptxas then also rotates two uniform quads)
#endif
#define VST 36                          // row stride of the staged v rows: 32 + 4 floats (rows start in different bank groups)
#define RUN_PAD_ROW BUNDLE_ATOMS

struct alignas(16) RunW { float W2[HID * HID]; };      // the ONLY constants the slot loop walks: exactly 4 KB (see bundle_run_kernel)

struct RunArgs {
    int n_bundles; const int2* bundle; int* work_counter;
    const int* rowptr; const int* col; const int* pid; const unsigned char* rowl; const float* e;
    const int* ustart;
    const int* far_off; const unsigned short* far_list;
    const int* far0_off; const unsigned short* far0_list; const unsigned char* far0_w; const int* rep; int dedup;
    const int* atom_sys; const int* sys_off; const int* npad;
    const float* u; const float* v;
    const float* Cw; const float* b2; const float* b1;      // device pointers into the packed weights (staged into shared memory)
    unsigned long long* slot_counter;                       // statistics (may be NULL): [0] near slots, [1] far slots evaluated
    float* S;
};

typedef unsigned long long r2_t;
#ifdef EPNN_CPU_EMU      // inline PTX replaced by its definition: two IEEE fma.rn on the packed halves; prefetches are hints
__device__ __forceinline__ r2_t rpack2(float lo, float hi) { unsigned a, b; memcpy(&a, &lo, 4); memcpy(&b, &hi, 4); return (r2_t)a | ((r2_t)b << 32); }
__device__ __forceinline__ void runpack2(r2_t v, float& lo, float& hi) { const unsigned a = (unsigned)v, b = (unsigned)(v >> 32); memcpy(&lo, &a, 4); memcpy(&hi, &b, 4); }
__device__ __forceinline__ void rfma2(r2_t& d, r2_t wpair, float a) {
    float d0, d1, w0, w1;
    runpack2(d, d0, d1); runpack2(wpair, w0, w1);
    d = rpack2(fmaf(w0, a, d0), fmaf(w1, a, d1));
}
__device__ __forceinline__ void rprefetch_l2(const void*) {}
__device__ __forceinline__ void rprefetch_l1(const void*) {}
#else
__device__ __forceinline__ r2_t rpack2(float lo, float hi) { r2_t r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void runpack2(r2_t v, float& lo, float& hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void rfma2(r2_t& d, r2_t wpair, float a) {
    const r2_t aa = rpack2(a, a);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(wpair), "l"(aa));
}
__device__ __forceinline__ void rprefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void rprefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
#endif

struct RunSmem {
    static constexpr int PW = (BUNDLE_ATOMS + 1) * VST + BUNDLE_ATOMS * HID + BUNDLE_ATOMS;     // floats per warp
    static size_t bytes() { return sizeof(float) * ((size_t)RUN_NW * PW + EDR * HID + HID); }
};

// S[row][0..31] += acc (one lane, 8 x 16-byte read-modify-write)
__device__ __forceinline__ void flush_row(float* __restrict__ S, int row, const r2_t (&sacc)[HID / 2]) {
    float4* p = reinterpret_cast<float4*>(S + row * HID);
    // 16-byte chunk c of row r lives at chunk c ^ (r & 7): lanes whose rows end at the same slot flush in one (divergent)
    // instruction, and with a row stride of 128 B they would all hit the same four banks (ncu: 7.4 wavefronts per flush
    // access, a third of the kernel's shared-memory wavefronts; A/B call81: 27.50 -> 26.25 ms)
    const int sw = row & 7;
#pragma unroll
    for (int cc = 0; cc < HID / 4; ++cc) {
        const int c = cc ^ sw;
        float4 s = p[c];
        float a0, a1, a2, a3;
        runpack2(sacc[2 * cc], a0, a1); runpack2(sacc[2 * cc + 1], a2, a3);
        s.x += a0; s.y += a1; s.z += a2; s.w += a3;
        p[c] = s;
    }
}

// second layer, outputs 16 * HALF .. 16 * HALF + 15 (RUN_HALVES: two passes of 8 FFMA2 chains, 16 registers less)
template <int HALF>
__device__ __forceinline__ void second_half(const RunW& W, const float* __restrict__ sb2, const float (&z)[HID], float wgt, r2_t (&sacc)[HID / 2]) {
    r2_t acc[8];
#pragma unroll
    for (int o = 0; o < 8; o += 2) {
        const ulonglong2 b = *reinterpret_cast<const ulonglong2*>(sb2 + 16 * HALF + 2 * o);
        acc[o] = b.x; acc[o + 1] = b.y;
    }
#pragma unroll
    for (int k = 0; k < HID; ++k)
#pragma unroll
        for (int o = 0; o < 8; ++o) rfma2(acc[o], *reinterpret_cast<const r2_t*>(&W.W2[k * HID + 16 * HALF + 2 * o]), z[k]);
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        float x, y;
        runpack2(acc[o], x, y);
        rfma2(sacc[8 * HALF + o], rpack2(fmaxf(x, 0.f), fmaxf(y, 0.f)), wgt);
    }
}

// second layer:  sacc += wgt * relu(b2 + W2^T z)   (16 independent FFMA2 chains)
__device__ __forceinline__ void second_layer(const RunW& W, const float* __restrict__ sb2, const float (&z)[HID], float wgt, r2_t (&sacc)[HID / 2]) {
    r2_t acc[HID / 2];
#pragma unroll
    for (int o = 0; o < HID / 2; o += 2) {
        const ulonglong2 b = *reinterpret_cast<const ulonglong2*>(sb2 + 2 * o);
        acc[o] = b.x; acc[o + 1] = b.y;
    }
#pragma unroll
    for (int k = 0; k < HID; ++k)
#pragma unroll
        for (int o = 0; o < HID / 2; ++o) rfma2(acc[o], *reinterpret_cast<const r2_t*>(&W.W2[k * HID + 2 * o]), z[k]);
#pragma unroll
    for (int o = 0; o < HID / 2; ++o) {
        float x, y;
        runpack2(acc[o], x, y);
        rfma2(sacc[o], rpack2(fmaxf(x, 0.f), fmaxf(y, 0.f)), wgt);
    }
}

__global__ void __launch_bounds__(RUN_NW * 32, RUN_CTAS) bundle_run_kernel(const __grid_constant__ RunW W, const RunArgs* __restrict__ ap) {
    // The arguments come through global memory on purpose: as kernel parameters ptxas re-reads them from the constant bank
    // inside the slot loop, and those extra lines push the loop's constant footprint (W2 = exactly 4 KB) over the level-0
    // constant cache -- every LDCU of a weight quad then misses.
    const RunArgs a = *ap;
#ifdef EPNN_CPU_EMU
    float* rsm = emu_smem;
#else
    extern __shared__ __align__(16) float rsm[];
#endif
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // The uniform-operand path is only fast while the constants a loop walks fit the 4 KB level-0 constant cache
    // (tools/ubench_uniform.cu: 64.7 TFLOP/s at 4 KB, 41 at >= 5 KB): W2 is exactly that, so the C rows of the near slots'
    // first product and the biases are served from shared memory (2.2 KB per CTA, broadcast LDS.128) instead.
    float* sCw = rsm;                                                // [EDR][32]
    float* sb2 = rsm + EDR * HID;                                    // [32]
    for (int t = threadIdx.x; t < EDR * HID; t += blockDim.x) sCw[t] = a.Cw[t];
    if (threadIdx.x < HID) sb2[threadIdx.x] = a.b2[threadIdx.x];
    __syncthreads();
    float* vS = rsm + EDR * HID + HID + warp * RunSmem::PW;          // [BUNDLE_ATOMS + 1][VST]
    float* S = vS + (BUNDLE_ATOMS + 1) * VST;                        // [BUNDLE_ATOMS][32]
    float* padw = S + BUNDLE_ATOMS * HID;                            // [BUNDLE_ATOMS]
    vS[RUN_PAD_ROW * VST + lane] = a.b1[lane];                       // v of the pad pseudo-atom (a_j = 0, e = 0)
    const unsigned full = 0xffffffffu;

    auto grab = [&]() {
        int x = 0;
        if (lane == 0) x = atomicAdd(a.work_counter, 1);
        return __shfl_sync(full, x, 0);
    };
    int b = grab();
    int b_next = grab();
    for (; b < a.n_bundles; b = b_next, b_next = grab()) {
        const int2 bd = a.bundle[b];
        const int atom0 = bd.x, nat = bd.y;
        if (b_next < a.n_bundles) {                                  // next bundle: u / v rows and descriptor rows -> L2
            const int2 nd = a.bundle[b_next];
            const int nbytes = nd.y * HID * (int)sizeof(float);
            for (int o = lane * 128; o < nbytes; o += 32 * 128) {
                rprefetch_l2(reinterpret_cast<const char*>(a.u + (int64_t)nd.x * HID) + o);
                rprefetch_l2(reinterpret_cast<const char*>(a.v + (int64_t)nd.x * HID) + o);
            }
            const int q0 = a.ustart[nd.x], q1 = a.ustart[nd.x + nd.y];
            for (int64_t o = (int64_t)q0 * EDR * 4 + lane * 128; o < (int64_t)q1 * EDR * 4; o += 32 * 128)
                rprefetch_l2(reinterpret_cast<const char*>(a.e) + o);
        }
        __syncwarp();
        // stage v (coalesced 16-byte loads, six in flight per lane instead of one load per loop trip), zero S
        for (int f0 = 0; f0 < nat * 8; f0 += 6 * 32) {
            float4 x[6];
#pragma unroll
            for (int q = 0; q < 6; ++q) {
                const int f = f0 + q * 32 + lane;
                x[q] = __ldg(reinterpret_cast<const float4*>(a.v + (int64_t)atom0 * HID) + (f < nat * 8 ? f : nat * 8 - 1));
            }
#pragma unroll
            for (int q = 0; q < 6; ++q) {
                const int f = f0 + q * 32 + lane;
                if (f < nat * 8) {
                    *reinterpret_cast<float4*>(vS + (f >> 3) * VST + (f & 7) * 4) = x[q];
                    *reinterpret_cast<float4*>(S + f * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
        for (int r = lane; r < nat; r += 32) {
            const int sys = a.atom_sys[atom0 + r];
            padw[r] = (float)(a.npad[sys] - (a.sys_off[sys + 1] - a.sys_off[sys]));
        }
        __syncwarp();
        // far columns: can they be collapsed to one weighted slot per species?  (v rows equal species by species; exact)
        bool use0 = a.dedup != 0;
        if (use0) {
            bool same = true;
            for (int r = lane; r < nat; r += 32) {
                const int rp = a.rep[atom0 + r] - atom0;
                if (rp != r) {
#pragma unroll
                    for (int c = 0; c < HID / 4; ++c) {
                        const float4 x = *reinterpret_cast<const float4*>(vS + r * VST + c * 4);
                        const float4 y = *reinterpret_cast<const float4*>(vS + rp * VST + c * 4);
                        same = same && x.x == y.x && x.y == y.y && x.z == y.z && x.w == y.w;
                    }
                }
            }
            use0 = __all_sync(full, same);
        }

#pragma unroll 1
        for (int phase = 0; phase < 2; ++phase) {                    // 0: near (CSR entries), 1: far list
            const bool near = phase == 0;
            const unsigned short* flist = use0 ? a.far0_list : a.far_list;
            int s0, s1;
            if (near) { s0 = a.rowptr[atom0]; s1 = a.rowptr[atom0 + nat]; }
            else { s0 = use0 ? a.far0_off[atom0] : a.far_off[atom0]; s1 = use0 ? a.far0_off[atom0 + nat] : a.far_off[atom0 + nat]; }
            const int len = s1 - s0;
            if (len <= 0) continue;
            if (a.slot_counter && lane == 0) atomicAdd(a.slot_counter + phase, (unsigned long long)len);
            const int J = (len + 31) >> 5;
            const int k0 = s0 + lane * J;
            int cur = -1;
            float uu[HID];
            r2_t sacc[HID / 2];
#pragma unroll
            for (int o = 0; o < HID / 2; ++o) sacc[o] = 0ull;
#pragma unroll
            for (int c = 0; c < HID; ++c) uu[c] = 0.f;
            // slot codes are fetched one slot ahead (three registers); the next slot's descriptor row and the next row's u
            // are pulled into L1 while the current slot computes
            int n_a = 0, n_b = 0, n_c = 0;
            auto fetch = [&](int k) {
                if (k < s1) {
                    if (near) {
                        n_a = a.rowl[k]; n_b = a.col[k]; n_c = a.pid[k];       // (fetching the pair index a second slot ahead costs a register: +12 %, call81)
                        rprefetch_l1(a.e + (int64_t)n_c * EDR);
                    } else {
                        n_a = flist[k]; n_b = use0 ? (int)a.far0_w[k] : 1;
                    }
                }
            };
            fetch(k0);
#pragma unroll kRunUnroll
            for (int it = 0; it < J; ++it) {
                const int k = k0 + it;
                const bool ok = k < s1;
                int li = cur < 0 ? 0 : cur, lj = 0;
                float wgt = 0.f;
                const float* erow = a.e;
                if (ok) {
                    if (near) {
                        li = n_a; lj = n_b - atom0; wgt = 1.f;
                        erow = a.e + (int64_t)n_c * EDR;
                    } else {
                        li = n_a >> 8; lj = n_a & 0xFF;
                        if (lj == 0xFF) { lj = RUN_PAD_ROW; wgt = padw[li]; }
                        else wgt = (float)n_b;
                    }
                }
                fetch(k + 1);
                if (ok && li != cur) {                               // row change (divergent, rare): flush the finished row, fetch u
                    if (cur >= 0) {
                        flush_row(S, cur, sacc);
#pragma unroll
                        for (int o = 0; o < HID / 2; ++o) sacc[o] = 0ull;
                    }
                    cur = li;
                    if (li + 1 < nat) rprefetch_l1(a.u + (int64_t)(atom0 + li + 1) * HID);      // the run's next row
#pragma unroll
                    for (int c = 0; c < HID / 4; ++c) {
                        const float4 x = __ldg(reinterpret_cast<const float4*>(a.u + (int64_t)(atom0 + li) * HID) + c);
                        uu[4 * c] = x.x; uu[4 * c + 1] = x.y; uu[4 * c + 2] = x.z; uu[4 * c + 3] = x.w;
                    }
                }
                float z[HID];
                if (near) {                                          // z = u + C^T c  (c = descriptor coefficients of the pair)
                    r2_t t2[HID / 2];
#pragma unroll
                    for (int o = 0; o < HID / 2; ++o) t2[o] = rpack2(uu[2 * o], uu[2 * o + 1]);
                    float cf[EDR];
#pragma unroll
                    for (int q = 0; q < EDR / 4; ++q) {
                        const float4 x = __ldg(reinterpret_cast<const float4*>(erow) + q);
                        cf[4 * q] = x.x; cf[4 * q + 1] = x.y; cf[4 * q + 2] = x.z; cf[4 * q + 3] = x.w;
                    }
#pragma unroll
                    for (int r = 0; r < EDR; ++r)
#pragma unroll
                        for (int o = 0; o < HID / 2; o += 2) {           // C rows come from shared memory (broadcast), see header
                            const ulonglong2 w4 = *reinterpret_cast<const ulonglong2*>(sCw + r * HID + 2 * o);
                            rfma2(t2[o], w4.x, cf[r]); rfma2(t2[o + 1], w4.y, cf[r]);
                        }
#pragma unroll
                    for (int o = 0; o < HID / 2; ++o) runpack2(t2[o], z[2 * o], z[2 * o + 1]);
                } else {
#pragma unroll
                    for (int c = 0; c < HID; ++c) z[c] = uu[c];
                }
                const float* vrow = vS + lj * VST;
#pragma unroll
                for (int c = 0; c < HID / 4; ++c) {
                    const float4 x = *reinterpret_cast<const float4*>(vrow + 4 * c);
                    z[4 * c] = fmaxf(z[4 * c] + x.x, 0.f); z[4 * c + 1] = fmaxf(z[4 * c + 1] + x.y, 0.f);
                    z[4 * c + 2] = fmaxf(z[4 * c + 2] + x.z, 0.f); z[4 * c + 3] = fmaxf(z[4 * c + 3] + x.w, 0.f);
                }
#ifdef RUN_HALVES
                second_half<0>(W, sb2, z, wgt, sacc);
                second_half<1>(W, sb2, z, wgt, sacc);
#else
                second_layer(W, sb2, z, wgt, sacc);
#endif
            }
            // the run's last row may continue in the following lanes: lanes holding the same row flush one after the other
            const unsigned grp = __match_any_sync(full, cur);
            const int rank = __popc(grp & ((1u << lane) - 1u));
            for (int r = 0; __any_sync(full, cur >= 0 && rank >= r); ++r) {
                if (cur >= 0 && rank == r) flush_row(S, cur, sacc);
                __syncwarp();
            }
        }
        // ---- S -> global (plane 0 of the partial-sum planes the per-atom kernel reads)
        for (int f = lane; f < nat * (HID / 4); f += 32)
            *reinterpret_cast<float4*>(a.S + (int64_t)atom0 * HID + f * 4) = *reinterpret_cast<const float4*>(S + (f ^ ((f >> 3) & 7)) * 4);   // undo flush_row's chunk swizzle
        __syncwarp();
    }
}

// local row (atom - first atom of its bundle) of every CSR entry of the small systems; built once per chunk
__global__ void csr_rowl_kernel(int n_atoms, const int* __restrict__ atom_sys, const int* __restrict__ sys_off,
                                const int* __restrict__ rowptr, const int* __restrict__ atom_b0, unsigned char* __restrict__ rowl) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const int s = atom_sys[i];
    if (sys_off[s + 1] - sys_off[s] > SMALL_MAX) return;
    const unsigned char r = (unsigned char)(i - atom_b0[i]);
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) rowl[k] = r;
}

#ifndef EPNN_CPU_EMU
cudaError_t launch_csr_rowl(const Workspace& w, const int* atom_b0, cudaStream_t st, int* nl) {
    if (w.n_atoms == 0 || w.n_bundles == 0 || w.nnz == 0) return cudaSuccess;
    csr_rowl_kernel<<<div_up(w.n_atoms, 256), 256, 0, st>>>(w.n_atoms, w.atom_sys, w.sys_off, w.rowptr, atom_b0, w.rowl);
    ++*nl;
    return cudaGetLastError();
}

cudaError_t launch_gnn_bundle_run(const Workspace& w, const StepW<float>& sw, cudaStream_t st, int* nl) {
    if (w.n_bundles == 0) return cudaSuccess;
    if (!w.wf_host || !w.wf_dev) return cudaErrorInvalidValue;
    RunW W;
    auto host = [&](const float* dev) { return w.wf_host + (dev - w.wf_dev); };
    memcpy(W.W2, host(sw.W2), sizeof(W.W2));
    RunArgs ra;
    ra.n_bundles = w.n_bundles; ra.bundle = w.bundle; ra.work_counter = w.work_counter;
    cudaError_t e = cudaMemsetAsync(w.work_counter, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    ra.rowptr = w.rowptr; ra.col = w.col; ra.pid = w.pid; ra.rowl = w.rowl; ra.e = w.e; ra.ustart = w.ustart;
    ra.far_off = w.far_off; ra.far_list = w.far_list;
    ra.far0_off = w.far0_off; ra.far0_list = w.far0_list; ra.far0_w = w.far0_w; ra.rep = w.rep; ra.dedup = w.dedup_far;
    ra.atom_sys = w.atom_sys; ra.sys_off = w.sys_off; ra.npad = w.npad;
    ra.u = (const float*)w.u; ra.v = (const float*)w.v; ra.S = (float*)w.S;
    ra.Cw = sw.Cw; ra.b2 = sw.b2; ra.b1 = sw.b1; ra.slot_counter = w.slot_counter;
    const size_t smem = RunSmem::bytes();
    e = cudaFuncSetAttribute(bundle_run_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int grid = div_up(w.n_bundles, RUN_NW);
    if (grid > w.sm_count * RUN_CTAS) grid = w.sm_count * RUN_CTAS;
    e = cudaMemcpyAsync(w.args_dev, &ra, sizeof(ra), cudaMemcpyHostToDevice, st);      // pageable source: staged before the call returns
    if (e != cudaSuccess) return e;
    bundle_run_kernel<<<grid, RUN_NW * 32, smem, st>>>(W, (const RunArgs*)w.args_dev);
    ++*nl;
    return cudaGetLastError();
}
#endif   // !EPNN_CPU_EMU
