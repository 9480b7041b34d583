// Internal declarations shared by the translation units of libepnn_b200.so (not installed).
#pragma once

#ifdef EPNN_CPU_EMU
#include "../../tools/emu/cuda_emu.h"      // CPU warp emulation of the kernels (tests/test_emu_*.py): lanes = host threads
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/epnn_b200.h"

#include "epnn_consts.h"
#include "epnn_plan.h"

// ------------------------------------------------------------------------------------------------
// Vector of 4 reals: one LDS.128 / LDG.128 for float, two for double.
template <typename R> struct alignas(4 * sizeof(R)) Vec4 { R x, y, z, w; };
// Width of the per-pair descriptor row the pair kernels consume: the FP32 path stores the EDR coefficients of e_ij in
// an orthonormal basis of the (numerically rank-16) family of radial descriptors, the FP64 verification path the 48
// float32-rounded values themselves.
template <typename R> struct EKof { static constexpr int v = sizeof(R) == 4 ? EDR : ED; };

template <typename R> __device__ __forceinline__ Vec4<R> vzero() { Vec4<R> v; v.x = v.y = v.z = v.w = R(0); return v; }
template <typename R> __device__ __forceinline__ Vec4<R> vadd(Vec4<R> a, Vec4<R> b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; return a; }
#ifndef EPNN_CPU_EMU
// FP32: two packed adds (Blackwell add.rn.f32x2, bit-identical to four scalar FADDs, half the FMA-pipe slots)
template <> __device__ __forceinline__ Vec4<float> vadd<float>(Vec4<float> a, Vec4<float> b) {
    unsigned long long a0, a1, b0, b1;
    asm("mov.b64 %0, {%1,%2};" : "=l"(a0) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1,%2};" : "=l"(a1) : "f"(a.z), "f"(a.w));
    asm("mov.b64 %0, {%1,%2};" : "=l"(b0) : "f"(b.x), "f"(b.y));
    asm("mov.b64 %0, {%1,%2};" : "=l"(b1) : "f"(b.z), "f"(b.w));
    asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a0) : "l"(b0));
    asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a1) : "l"(b1));
    Vec4<float> r;
    asm("mov.b64 {%0,%1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(a0));
    asm("mov.b64 {%0,%1}, %2;" : "=f"(r.z), "=f"(r.w) : "l"(a1));
    return r;
}
#endif
template <typename R> __device__ __forceinline__ Vec4<R> vscale(Vec4<R> a, R s) { a.x *= s; a.y *= s; a.z *= s; a.w *= s; return a; }
#ifndef EPNN_CPU_EMU
template <> __device__ __forceinline__ Vec4<float> vscale<float>(Vec4<float> a, float s) {
    unsigned long long a0, a1, ss;
    asm("mov.b64 %0, {%1,%2};" : "=l"(a0) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1,%2};" : "=l"(a1) : "f"(a.z), "f"(a.w));
    asm("mov.b64 %0, {%1,%1};" : "=l"(ss) : "f"(s));
    asm("mul.rn.f32x2 %0, %0, %1;" : "+l"(a0) : "l"(ss));
    asm("mul.rn.f32x2 %0, %0, %1;" : "+l"(a1) : "l"(ss));
    Vec4<float> r;
    asm("mov.b64 {%0,%1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(a0));
    asm("mov.b64 {%0,%1}, %2;" : "=f"(r.z), "=f"(r.w) : "l"(a1));
    return r;
}
#endif
template <typename R> __device__ __forceinline__ Vec4<R> vrelu(Vec4<R> a) {
    a.x = a.x > R(0) ? a.x : R(0); a.y = a.y > R(0) ? a.y : R(0);
    a.z = a.z > R(0) ? a.z : R(0); a.w = a.w > R(0) ? a.w : R(0); return a;
}
template <typename R> __device__ __forceinline__ R relu(R a) { return a > R(0) ? a : R(0); }
template <typename R> __device__ __forceinline__ Vec4<R> ldv(const R* p) { return *reinterpret_cast<const Vec4<R>*>(p); }
template <typename R> __device__ __forceinline__ void stv(R* p, Vec4<R> v) { *reinterpret_cast<Vec4<R>*>(p) = v; }
template <typename R> __device__ __forceinline__ Vec4<R> cvt4(float4 f) { Vec4<R> v; v.x = R(f.x); v.y = R(f.y); v.z = R(f.z); v.w = R(f.w); return v; }

// ------------------------------------------------------------------------------------------------
// Warp-tile GEMM core used by every MLP kernel.
//
// One warp multiplies a tile of 32 rows ("slots": pairs or atoms) by a K x 32 weight block:
//     acc[s][c] += sum_k  A[pg*8+s][k] * W[k][wcol+c]          s = 0..7, c = 0..3
// Thread (pg = lane>>3, og = lane&7) owns rows pg*8..pg*8+7 and output columns wcol..wcol+3
// (wcol = column base + og*4): an 8x4 register tile, 128 FMA per 12 LDS.128.
//
// The A tile lives in shared memory slot-major, row stride K, with the 4-float chunk index XOR-ed by
// the row's pg (= row>>3): chunk' = chunk ^ (row>>3).  With that swizzle the four pg groups of a warp
// read four different 16-byte bank groups (conflict-free), and the producers' 128-bit stores (8 lanes
// of one pg covering 8 consecutive chunks of one row) are conflict-free as well.
template <typename R, int K, int WLD>
__device__ __forceinline__ void tile_gemm(const R* __restrict__ at, const R* __restrict__ W, int wcol,
                                          R (&acc)[8][4], int pg) {
    const R* arow = at + pg * 8 * K;
#pragma unroll 2
    for (int kc = 0; kc < K / 4; ++kc) {
        const Vec4<R> w0 = ldv(W + (kc * 4 + 0) * WLD + wcol);
        const Vec4<R> w1 = ldv(W + (kc * 4 + 1) * WLD + wcol);
        const Vec4<R> w2 = ldv(W + (kc * 4 + 2) * WLD + wcol);
        const Vec4<R> w3 = ldv(W + (kc * 4 + 3) * WLD + wcol);
        const int kcs = (kc ^ pg) * 4;
#pragma unroll
        for (int s = 0; s < 8; ++s) {
            const Vec4<R> a = ldv(arow + s * K + kcs);
            acc[s][0] = fma(a.x, w0.x, acc[s][0]); acc[s][1] = fma(a.x, w0.y, acc[s][1]);
            acc[s][2] = fma(a.x, w0.z, acc[s][2]); acc[s][3] = fma(a.x, w0.w, acc[s][3]);
            acc[s][0] = fma(a.y, w1.x, acc[s][0]); acc[s][1] = fma(a.y, w1.y, acc[s][1]);
            acc[s][2] = fma(a.y, w1.z, acc[s][2]); acc[s][3] = fma(a.y, w1.w, acc[s][3]);
            acc[s][0] = fma(a.z, w2.x, acc[s][0]); acc[s][1] = fma(a.z, w2.y, acc[s][1]);
            acc[s][2] = fma(a.z, w2.z, acc[s][2]); acc[s][3] = fma(a.z, w2.w, acc[s][3]);
            acc[s][0] = fma(a.w, w3.x, acc[s][0]); acc[s][1] = fma(a.w, w3.y, acc[s][1]);
            acc[s][2] = fma(a.w, w3.z, acc[s][2]); acc[s][3] = fma(a.w, w3.w, acc[s][3]);
        }
    }
}

// FP32 specialisation on Blackwell's packed FFMA2 (PTX fma.rn.f32x2, sm_100+): one instruction does two
// IEEE fma.rn -- bit-identical to two scalar FFMAs -- so the k-loop needs half the issue slots, and the
// 3-distinct-register scalar FFMA's register-bank limit (measured: 35 of 67 TFLOP/s for acc += a*w, tools/ubench.cu)
// goes away.  The pair operand is the weight pair (w[c], w[c+1]); the activation is the scalar that ptxas
// folds into FFMA2's broadcast ".F32" operand form (no MOV is emitted for the duplicated pair).
typedef unsigned long long f32x2_t;
#ifdef EPNN_CPU_EMU      // the packed instructions replaced by their definition: two IEEE fma.rn on the halves
__device__ __forceinline__ f32x2_t pack2(float lo, float hi) { unsigned a, b; memcpy(&a, &lo, 4); memcpy(&b, &hi, 4); return (f32x2_t)a | ((f32x2_t)b << 32); }
__device__ __forceinline__ void unpack2(f32x2_t v, float& lo, float& hi) { const unsigned a = (unsigned)v, b = (unsigned)(v >> 32); memcpy(&lo, &a, 4); memcpy(&hi, &b, 4); }
__device__ __forceinline__ void fma2(f32x2_t& d, f32x2_t wpair, float a) {
    float d0, d1, w0, w1;
    unpack2(d, d0, d1); unpack2(wpair, w0, w1);
    d = pack2(fmaf(w0, a, d0), fmaf(w1, a, d1));
}
#else
__device__ __forceinline__ f32x2_t pack2(float lo, float hi) { f32x2_t r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f32x2_t v, float& lo, float& hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void fma2(f32x2_t& d, f32x2_t wpair, float a) {
    const f32x2_t aa = pack2(a, a);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(wpair), "l"(aa));
}
#endif
template <int K, int WLD, int UNR = 2>
__device__ __forceinline__ void tile_gemm_f32x2(const float* __restrict__ at, const float* __restrict__ W, int wcol,
                                                float (&acc)[8][4], int pg) {
    const float* arow = at + pg * 8 * K;
    f32x2_t c[8][2];
#pragma unroll
    for (int s = 0; s < 8; ++s) { c[s][0] = pack2(acc[s][0], acc[s][1]); c[s][1] = pack2(acc[s][2], acc[s][3]); }
#pragma unroll UNR
    for (int kc = 0; kc < K / 4; ++kc) {
        f32x2_t w[4][2];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const ulonglong2 t = *reinterpret_cast<const ulonglong2*>(W + (kc * 4 + k) * WLD + wcol);
            w[k][0] = t.x; w[k][1] = t.y;
        }
        const int kcs = (kc ^ pg) * 4;
#pragma unroll
        for (int s = 0; s < 8; ++s) {
            const float4 a = *reinterpret_cast<const float4*>(arow + s * K + kcs);
            fma2(c[s][0], w[0][0], a.x); fma2(c[s][1], w[0][1], a.x);
            fma2(c[s][0], w[1][0], a.y); fma2(c[s][1], w[1][1], a.y);
            fma2(c[s][0], w[2][0], a.z); fma2(c[s][1], w[2][1], a.z);
            fma2(c[s][0], w[3][0], a.w); fma2(c[s][1], w[3][1], a.w);
        }
    }
#pragma unroll
    for (int s = 0; s < 8; ++s) { unpack2(c[s][0], acc[s][0], acc[s][1]); unpack2(c[s][1], acc[s][2], acc[s][3]); }
}
template <> __device__ __forceinline__ void tile_gemm<float, EDR, HID>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<EDR, HID>(at, W, wcol, acc, pg); }
template <> __device__ __forceinline__ void tile_gemm<float, ED, HID>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<ED, HID>(at, W, wcol, acc, pg); }
template <> __device__ __forceinline__ void tile_gemm<float, HID, HID>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<HID, HID>(at, W, wcol, acc, pg); }
template <> __device__ __forceinline__ void tile_gemm<float, UPD_IN, HID>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<UPD_IN, HID>(at, W, wcol, acc, pg); }
template <> __device__ __forceinline__ void tile_gemm<float, HID, HD>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<HID, HD>(at, W, wcol, acc, pg); }
template <> __device__ __forceinline__ void tile_gemm<float, 64, HID>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<64, HID>(at, W, wcol, acc, pg); }
template <> __device__ __forceinline__ void tile_gemm<float, HID, 64>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<HID, 64>(at, W, wcol, acc, pg); }
template <> __device__ __forceinline__ void tile_gemm<float, HD, 64>(const float* __restrict__ at, const float* __restrict__ W, int wcol, float (&acc)[8][4], int pg) { tile_gemm_f32x2<HD, 64>(at, W, wcol, acc, pg); }

// Same product with an explicit unroll factor of the k loop (FP32 only; the FP64 verification path keeps the generic core).
// Measured (tools/gpu_ab_unroll.sh): the EPN bundle kernel gains 8 % from a fully unrolled loop, the (larger) GNN bundle
// kernel and the per-atom kernel lose 6..25 % -- hence a per-call-site choice, default 2.
template <typename R, int K, int WLD, int UNR>
__device__ __forceinline__ void tile_gemm_unr(const R* __restrict__ at, const R* __restrict__ W, int wcol, R (&acc)[8][4], int pg) {
    if constexpr (sizeof(R) == 4) tile_gemm_f32x2<K, WLD, UNR>(at, W, wcol, acc, pg);
    else tile_gemm<R, K, WLD>(at, W, wcol, acc, pg);
}

template <typename R> __device__ __forceinline__ void zero_acc(R (&acc)[8][4]) {
#pragma unroll
    for (int s = 0; s < 8; ++s) { acc[s][0] = acc[s][1] = acc[s][2] = acc[s][3] = R(0); }
}

// Address (in elements) of chunk `ch` of row `row` in a swizzled tile with row stride K.
__device__ __forceinline__ int tile_off(int row, int ch, int K) { return row * K + ((ch ^ (row >> 3)) << 2); }

// ------------------------------------------------------------------------------------------------
// Device weight views (all row-major, precision R).  Built once in epnn_create.
template <typename R> struct StepW {      // one message or pass MLP, first layer split per SURVEY 7.2
    const R* Ah64;   // [48][64]  h-rows of the first layer:  cols 0..31 = a_i block (u), 32..63 = a_j block (v)
    const R* Aq64;   // [64]      q-row
    const R* Ax64;   // [MAX_SPECIES][64]  per-species x contribution, b1 folded into the v half
    const R* Cw;     // [EK][32]  e-rows: EK = 48 (FP64: C itself) or 16 (FP32: B^T C, B = reduced basis of the descriptors)
    const R* b1;     // [32]      (v of a padded atom: a_j = 0, e = 0)
    const R* W2;     // [32][32]
    const R* b2;     // [32]
    const R* W3;     // [32][32] (message) or [32] (pass)
    const R* b3;     // [32] or [1]
    // per-atom kernel, linear layers folded on the host (exact algebra, float64):
    const R* Pf;     // [32][64]  U3 . Ah64        : u|v of the NEXT pair kernel straight from the update MLP's last hidden layer l2
    const R* Axf;    // [MAX_SPECIES][64]  Ax64 + c3^T Ah64
    const R* HG;     // [64][32]  [U3 . U1_h ; W3 . U1_M] : first update layer applied to [l2_prev | S]   (message steps only)
    const R* g;      // [32]      U1_M^T b3               : times npad, the hoisted last-layer bias        (message steps only)
};
template <typename R> struct UpdW {       // shared update MLP 80 -> 32 -> 32 -> 48
    const R* U1; const R* c1; const R* U2; const R* c2; const R* U3; const R* c3;
    const R* cb1;    // [32]  c1 + U1_h^T c3 : first-layer bias of every step after the first (h = U3^T l2 + c3 folded in)
};

template <typename R> struct DenseW {      // raw (un-split) views of one MLP step
    const R* Wx64;   // [n_x][64]  x-rows of the first layer: cols 0..31 a_i block, 32..63 a_j block
    const R* Ah64;   // [48][64]
    const R* Aq64;   // [64]
    const R* Cw;     // [48][32]
    const R* b1;     // [32]
    const R* W2; const R* b2; const R* W3; const R* b3;
};

#ifndef EPNN_CPU_EMU
template <typename R>
cudaError_t launch_dense_forward(int B, int N, int n_x, int T, const float* h, const float* e, const float* x, const float* q,
                                 const float* mask, const DenseW<R>* msgw, const UpdW<R>& upd, const DenseW<R>* pasw,
                                 R* a, R* node_mask, R* uv, R* msg, float* q_out, cudaStream_t st);
#endif

// ------------------------------------------------------------------------------------------------
// Per-chunk device workspace (pointers into grow-only buffers owned by the ctx).
struct Workspace {
    int n_atoms, n_sys, sm_count;
    int64_t nnz, P;                    // CSR entries of the e != 0 list; unordered pairs (nnz == 2P)
    // inputs
    const float* xyz; const int* species; const int* sys_off; const float* Qsys; const int* npad;
    // derived
    int* atom_sys;
    const int* deg_all;                // sharded calls: the degrees of ALL rows (all-gathered copy); NULL otherwise
    int* deg; int* degU; int* rowptr; int* ustart; int* col; int* pid;
    int* pair_i; int* pair_j; double* pair_D; float* e; unsigned char* near;
    int ek;                            // floats per row of `e`: ED (48 descriptor values) or EDR (16 basis coefficients)
    int* work_counter;                 // device int: dynamic work queue of the bundle kernels
    int2* bundle; int n_bundles;       // (first atom, atom count) of every bundle of small systems (n <= SMALL_MAX)
    unsigned char* rowl;               // local row (atom - first atom of its bundle) of every CSR entry (small systems)
    int* bundle_nat; unsigned char* perm_j;   // atoms of the bundle (at its first atom); rank of a pair's j inside its tile
    int* far_off; unsigned short* far_list; int64_t n_far;
    int* far0_off; unsigned short* far0_list; unsigned char* far0_w; int* rep; int64_t n_far0; int dedup_far;   // species-compressed far list   // per-bundle list of the GNN's e == 0 ("far") ordered pairs
    int* rg_large; int n_rg_large; int nsplit;    // 4-row groups of the large systems
    const int2* rowblk; int n_rowblk;             // 32-row blocks of the large systems (first atom, system): units of gnn_far_const_kernel
    FarKernel far_kernel;                         // far part of the big-system message sum (ChunkPlan::far); unless FAR_SIMT, planes
                                                  // [0, nsplit-1) of S are the far kernel's, the SIMT kernel (near only) owns the last
    int row_lo, row_hi;                           // rows [row_lo, row_hi) of the chunk belong to this rank (unsharded: [0, n_atoms))
    int rg_begin, rg_end, blk_begin, blk_end;     // 4-row groups / 32-row blocks of the large systems that overlap the slice
    const unsigned char* active;                  // sharded: 1 for owned atoms and their near neighbours (rows whose projections are needed here)
    // species tables of the large systems (exact de-duplication of their far columns, epnn_gnn.cu): entry
    // rgl_off[sys] >> 3 (a large system has >= 13 row groups, so the entries of two systems never collide)
    const int* rgl_off;                           // [n_sys + 1] first row group of every system
    int* sp_tab; int n_sp_tab;                    // [n_sp_tab][32]: atoms per species [16] | first atom of the species [16]
    int* sp_stamp;                                // [n_sp_tab][2]: stamp of the last step whose v rows were NOT species-wise equal | dedup forbidden
    int stamp;                                    // stamp of the current message-passing step (t + 1); 0 = de-duplication off
    int n_species;                                // species of the element table in use (8 or 9)
    KernelChoice kc;                              // kernels of the call (resolve_kernels)
    void* args_dev;                               // 1 KB device scratch: argument block of the kernels that take theirs through global memory
    const float* wf_host; const float* wf_dev;    // packed FP32 weights: host mirror and device base (pair_const passes weights as kernel parameters)
    unsigned long long* near_counter;             // device counter (statistics, may be NULL): unordered pairs in the is_near set
    unsigned long long* slot_counter;             // device counters (statistics): [0] near, [1] far slots evaluated by the row-run GNN kernel
    unsigned long long* dedup_rows;               // device counter (statistics): rows whose far part was collapsed, summed over steps
    void* h; void* S; void* u; void* v; void* delta;   // precision-dependent (float or double)
    void* l2;                          // [n][32] last hidden layer of the update MLP: the state carried between steps
    double* q;
};

// Cell-list state of the big systems of one chunk (epnn_neighbor.cu)
struct CellGrid { float ox, oy, oz, inv_h; int nx, ny, nz, base; };
struct CellWork {
    int n_large; int n_cells;                 // big systems in the chunk; total cell budget (host-side prefix of 4 n + 64)
    const int* large_sys; const int* large_base;   // [n_large] system index, first cell
    CellGrid* grid;                           // [n_sys] (entries of big systems only)
    int* cell_cnt; int* cell_start; int* cell_atoms; double* Dtmp;
};

// Scratch of the fused list building for chunks of small systems only (epnn_bundle_prep.cu)
struct BundlePrepWork {
    unsigned long long* mask;   // [n_atoms] neighbour mask of every row inside its bundle
    int* btot; int* boff;       // [4][n_bundles] per-bundle totals (nnz | P | far | far0), [4][n_bundles + 1] their exclusive scans
    int* atom_b0;               // [n_atoms] first atom of the row's bundle
};

#ifndef EPNN_CPU_EMU
// ------------------------------------------------------------------------------------------------
// Launchers (defined in the .cu files; every one enqueues on `st` and returns cudaGetLastError()).
cudaError_t launch_prep(const Workspace& w, cudaStream_t st, int* n_launch);
cudaError_t launch_cell_build(const Workspace& w, const CellWork& cw, int* scantmp, cudaStream_t st, int* n_launch);
cudaError_t launch_nbr_count(const Workspace& w, const CellWork& cw, cudaStream_t st, int* n_launch);
cudaError_t launch_scan_i32(const int* in, int* out, int n, int* tmp, cudaStream_t st, int* n_launch);
cudaError_t launch_nbr_fill(const Workspace& w, const CellWork& cw, cudaStream_t st, int* n_launch);
cudaError_t launch_edges_dense(int n, const float* xyz, float* e, cudaStream_t st);
cudaError_t upload_rbf_centers(const double* mu);
cudaError_t upload_rbf_basis(const double* B);      // [ED][EDR]

cudaError_t launch_edge_desc(const Workspace& w, cudaStream_t st, int* n_launch, bool gather);   // descriptors + near flags of the pair list (gather: D from the coordinates)
cudaError_t launch_tile_perm(const Workspace& w, const int* atom_b0, cudaStream_t st, int* n_launch);   // if w.kc.tile_perm
cudaError_t launch_bundle_prep_count(const Workspace& w, const BundlePrepWork& bw, int* scantmp, int* flags, cudaStream_t st, int* n_launch);
cudaError_t launch_bundle_prep_fill(const Workspace& w, const BundlePrepWork& bw, cudaStream_t st, int* n_launch);
cudaError_t launch_far_count(const Workspace& w, int* far_cnt, int* atom_b0, cudaStream_t st, int* n_launch);
cudaError_t launch_far_fill(const Workspace& w, const int* atom_b0, cudaStream_t st, int* n_launch);
cudaError_t launch_far0_count(const Workspace& w, int* cnt, cudaStream_t st, int* n_launch);
cudaError_t launch_far0_fill(const Workspace& w, const int* atom_b0, cudaStream_t st, int* n_launch);
template <typename R> cudaError_t launch_gnn_bundle(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* n_launch);
template <typename R> cudaError_t launch_epn_bundle(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* n_launch);
cudaError_t launch_epn_bundle_mma(const Workspace& w, const StepW<float>& sw, cudaStream_t st, int* n_launch);   // option pair_tensor
cudaError_t launch_gnn_bundle_const(const Workspace& w, const StepW<float>& sw, cudaStream_t st, int* n_launch); // option pair_const
cudaError_t launch_epn_bundle_const(const Workspace& w, const StepW<float>& sw, cudaStream_t st, int* n_launch);
cudaError_t launch_gnn_bundle_run(const Workspace& w, const StepW<float>& sw, cudaStream_t st, int* n_launch);   // row-run mapping (FP32 default)
cudaError_t launch_csr_rowl(const Workspace& w, const int* atom_b0, cudaStream_t st, int* n_launch);
cudaError_t launch_gnn_far_const(const Workspace& w, const StepW<float>& sw, int nsplit_far, cudaStream_t st, int* n_launch);   // option pair_const
cudaError_t launch_gnn_far_tc(const Workspace& w, const float* Whi, const float* Wlo, const float* b2, int nsplit_tc,
                              cudaStream_t st, int* n_launch);
cudaError_t launch_gnn_far_tc2(const Workspace& w, const float* Whi, const float* Wlo, const float* b2, int nsplit_tc,
                               cudaStream_t st, int* n_launch);      // warp-specialised variant (epnn_gnn_tc2.cu)
template <typename R> cudaError_t launch_gnn_pair(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* n_launch);
cudaError_t launch_sp_tab_build(const Workspace& w, cudaStream_t st, int* n_launch);                    // once per chunk
template <typename R> cudaError_t launch_sp_check(const Workspace& w, cudaStream_t st, int* n_launch);  // once per step (needs w.stamp)
template <typename R> cudaError_t launch_epn_pair(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* n_launch);
#endif   // !EPNN_CPU_EMU
// mode bits for the per-atom kernel
#define ATOM_UPDATE  1     // h <- update_fn([h | W3^T S + npad*b3])   (finishes a message-passing step)
#define ATOM_QUPDATE 2     // q <- q + sum_j (+/-) delta               (finishes an electron-passing pass)
#define ATOM_PROJECT 4     // u,v <- first-layer projections for the next pair kernel
#define ATOM_OUTPUT  8     // write q to the output buffers
#define ATOM_FIRST   16    // first message-passing step: h = 0, there is no previous l2
#define ATOM_WRITE_H 32    // also materialise h = U3^T l2 + c3 (last message-passing step: epnn_get_hidden)
// R = arithmetic and state type (weights, l2, h); IO = type of the buffers shared with the pair kernels (S planes in, u / v out,
// delta in).  IO = float with R = double is the "mixed" precision: FP32 pair kernels around an FP64 per-atom kernel.
template <typename R, typename IO> struct AtomArgs {
    int n_atoms, mode, nsplit, h_is_zero;
    const int* atom_sys; const int* sys_off; const int* npad; const int* species;
    const IO* Spart; R* h; R* l2; const R* HG; const R* g; const R* cb; UpdW<R> upd;
    const int* rowptr; const int* col; const int* pid; const IO* delta; double* q;
    const R* Pf; const R* Aq64; const R* Ax; IO* u; IO* v;
    float* q_out; double* q_out64;
    // sharded call: which atoms of LARGE systems this launch touches (small systems are replicated on every rank)
    int scope, row_lo, row_hi; const unsigned char* active;     // scope 0 all, 1 owned rows [row_lo, row_hi), 2 active[] (owned + halo)
};
#ifndef EPNN_CPU_EMU
template <typename R> cudaError_t launch_atom(const Workspace& w, int mode, const StepW<R>* prev, const UpdW<R>* upd,
                                              const StepW<R>* next, int h_is_zero, float* q_out, double* q_out64,
                                              cudaStream_t st, int* n_launch, int scope = 0);      // scope: see AtomArgs (sharded calls)
cudaError_t launch_atom_mixed(const Workspace& w, int mode, const StepW<double>* prev, const UpdW<double>* upd, const StepW<double>* next,
                              int h_is_zero, float* q_out, double* q_out64, cudaStream_t st, int* n_launch, int scope = 0);   // precision 48
cudaError_t launch_atom_mma(const Workspace& w, const AtomArgs<float, float>& aa, cudaStream_t st, int* n_launch);   // option atom_tensor (epnn_atom_mma.cu)
cudaError_t launch_atom_const(const Workspace& w, int mode, const StepW<float>* prev, const UpdW<float>* upd, const StepW<float>* next,
                              int h_is_zero, float* q_out, double* q_out64, cudaStream_t st, int* n_launch);   // option pair_const
struct ElstArgs;
cudaError_t launch_elst(const ElstArgs& a, int n_items, int n_large, cudaStream_t st);   // epnn_elst.cu (plan: epnn_elst.cuh)
struct ElstPtArgs;
cudaError_t launch_elst_points(const ElstPtArgs& a, int n_items, int n_red, cudaStream_t st);   // epnn_elst.cu (plan: epnn_elst.cuh)

#endif   // !EPNN_CPU_EMU
static inline int div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
