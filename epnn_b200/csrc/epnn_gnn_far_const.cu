// FP32 kernel for the FAR (e == 0) part of the big-system message sum: the default far kernel of precision 32 for
// systems of 49 .. 16 383 atoms ("pair_const" 1 or 2, the default 2, whenever the tcgen05 kernel of epnn_gnn_tc.cu is
// not selected; that one takes over from "gnn_far_tensor_min" = 16 384 atoms).  Checked on the GPU against the float64
// oracle (tests/test_gpu_large_reference.py, tests/test_gpu_pair_const.py) and by the CPU warp emulation inside whole
// inferences (tests/test_emu_infer.py).
//
// For a row i of a big system the reference sums  m_ij = relu(W2^T relu(u_i + v_j) + b2)  over ALL columns j that are not
// within the cutoff (charge_gn.py:66-70, no mask) -- the O(n^2) part of a step whenever the far-column de-duplication
// does not apply (live hidden state).  Mapping: ONE THREAD OWNS ONE ROW.  A warp takes 32 consecutive rows of one
// system and walks a range of columns; all lanes need the SAME v_j at the same time, so the warp stages 32 v rows at a
// time in shared memory and every lane reads them with broadcast loads; u_i, the 32 second-layer accumulators and the
// 32 running sums stay in the thread's registers; W2 / b2 are uniform operands from a __grid_constant__ parameter
// (FFMA2 R, R.F32, UR.F32x2, R.F32x2).  No scatter, no shuffles: the sum over j IS the thread's accumulator.  Near
// neighbours are skipped with a per-lane cursor into the (ascending) CSR row.  Running sums are kept in FP32 over a
// chunk of 32 columns and folded into FP64 accumulators (shared memory, one row per lane) after every chunk, so the
// result has the same accuracy class as the FP64 row sums of gnn_pair_kernel.  Output goes to the partial-sum planes
// [0, nsplit_far) of S, one per column range, like the tcgen05 far kernel; the near pairs, the pad pair and the
// de-duplicated species slots stay on gnn_pair_kernel (skip_far mode, last plane).
#include "epnn_internal.cuh"

#define FARC_NW 8
#define FARC_COLS 32                       // columns (v rows) staged per chunk

struct alignas(16) FarW { float W2[HID * HID]; float b2[HID]; };

struct FarConstArgs {
    const int2* blk; int unit_begin, unit_end, nsplit, n_atoms;      // blk: (first atom of a 32-row block, system index)
    const int* sys_off; const int* rowptr; const int* col;
    const float* u; const float* v; float* S;
    const int* rgl_off; const int* sp_stamp; int stamp;              // far-column de-duplication (epnn_gnn.cu); stamp == 0: off
};

typedef unsigned long long g2_t;
#ifdef EPNN_CPU_EMU
__device__ __forceinline__ g2_t gpack2(float lo, float hi) { unsigned a, b; memcpy(&a, &lo, 4); memcpy(&b, &hi, 4); return (g2_t)a | ((g2_t)b << 32); }
__device__ __forceinline__ void gunpack2(g2_t v, float& lo, float& hi) { const unsigned a = (unsigned)v, b = (unsigned)(v >> 32); memcpy(&lo, &a, 4); memcpy(&hi, &b, 4); }
__device__ __forceinline__ void gfma2(g2_t& d, g2_t wpair, float a) {
    float d0, d1, w0, w1;
    gunpack2(d, d0, d1); gunpack2(wpair, w0, w1);
    d = gpack2(fmaf(w0, a, d0), fmaf(w1, a, d1));
}
#else
__device__ __forceinline__ g2_t gpack2(float lo, float hi) { g2_t r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void gunpack2(g2_t v, float& lo, float& hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void gfma2(g2_t& d, g2_t wpair, float a) {
    const g2_t aa = gpack2(a, a);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(wpair), "l"(aa));
}
#endif

// per warp: v chunk [FARC_COLS][32] floats, then FP64 sums [32 lanes][33] doubles (padded rows)
#define FARC_PW_BYTES (FARC_COLS * HID * 4 + 32 * 33 * 8)

__global__ void __launch_bounds__(FARC_NW * 32, 2) gnn_far_const_kernel(const __grid_constant__ FarW W, const FarConstArgs a) {
#ifdef EPNN_CPU_EMU
    unsigned char* fsm = reinterpret_cast<unsigned char*>(emu_smem);
#else
    extern __shared__ __align__(16) unsigned char fsm[];
#endif
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* vs = reinterpret_cast<float*>(fsm + (size_t)warp * FARC_PW_BYTES);                  // [FARC_COLS][32]
    double* Sd = reinterpret_cast<double*>(fsm + (size_t)warp * FARC_PW_BYTES + FARC_COLS * HID * 4);   // [32][33]

    for (int unit = a.unit_begin + blockIdx.x * FARC_NW + warp; unit < a.unit_end; unit += gridDim.x * FARC_NW) {
        const int b = unit / a.nsplit, split = unit - b * a.nsplit;
        const int2 bd = a.blk[b];
        const int i0 = bd.x, sys = bd.y;
        const int a0 = a.sys_off[sys], a1 = a.sys_off[sys + 1];
        const int n = a1 - a0;
        int clen = (n + a.nsplit - 1) / a.nsplit;
        clen = (clen + FARC_COLS - 1) / FARC_COLS * FARC_COLS;
        const int jlo = min(a1, a0 + split * clen);
        int jhi = min(a1, jlo + clen);
        if (a.stamp) {                     // gnn_pair_kernel sums this system's far columns species by species at this step
            const int ti = a.rgl_off[sys] >> 3;
            if (a.sp_stamp[2 * ti] != a.stamp && a.sp_stamp[2 * ti + 1] == 0) jhi = jlo;
        }
        const int i = i0 + lane;
        const bool rowok = i < a1 && i < i0 + 32;
        float ui[HID];
#pragma unroll
        for (int c4 = 0; c4 < HID / 4; ++c4) {
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (rowok) x = *reinterpret_cast<const float4*>(a.u + (int64_t)i * HID + c4 * 4);
            ui[4 * c4] = x.x; ui[4 * c4 + 1] = x.y; ui[4 * c4 + 2] = x.z; ui[4 * c4 + 3] = x.w;
        }
        int ptr = 0, rp1 = 0;              // cursor into the ascending CSR row: the next near neighbour at or after the current column
        if (rowok) {
            ptr = a.rowptr[i]; rp1 = a.rowptr[i + 1];
            while (ptr < rp1 && a.col[ptr] < jlo) ++ptr;
        }
        int next_near = ptr < rp1 ? a.col[ptr] : 0x7fffffff;
        __syncwarp();
#pragma unroll 4
        for (int c = 0; c < HID; ++c) Sd[lane * 33 + c] = 0.0;

        for (int jc = jlo; jc < jhi; jc += FARC_COLS) {
            const int ncol = min(FARC_COLS, jhi - jc);
            __syncwarp();                                          // the previous chunk's rows are no longer read
            for (int f = lane; f < ncol * 8; f += 32)              // stage the chunk's v rows: whole 128-byte lines
                *reinterpret_cast<float4*>(vs + f * 4) = *reinterpret_cast<const float4*>(a.v + (int64_t)jc * HID + f * 4);
            __syncwarp();
            float s32[HID];
#pragma unroll
            for (int c = 0; c < HID; ++c) s32[c] = 0.f;
#pragma unroll 1
            for (int jj = 0; jj < ncol; ++jj) {
                const int j = jc + jj;
                bool far = rowok;
                if (j == next_near) {                              // (i, j) is an e != 0 pair: it belongs to the near phase
                    far = false;
                    ++ptr;
                    next_near = ptr < rp1 ? a.col[ptr] : 0x7fffffff;
                }
                g2_t acc[HID / 2];
#pragma unroll
                for (int o = 0; o < HID / 2; ++o) acc[o] = gpack2(W.b2[2 * o], W.b2[2 * o + 1]);
#pragma unroll
                for (int k4 = 0; k4 < HID / 4; ++k4) {
                    const float4 v4 = *reinterpret_cast<const float4*>(vs + jj * HID + 4 * k4);     // same address in every lane: broadcast
                    const float z[4] = {fmaxf(ui[4 * k4] + v4.x, 0.f), fmaxf(ui[4 * k4 + 1] + v4.y, 0.f),
                                        fmaxf(ui[4 * k4 + 2] + v4.z, 0.f), fmaxf(ui[4 * k4 + 3] + v4.w, 0.f)};
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                        for (int o = 0; o < HID / 2; ++o) gfma2(acc[o], *reinterpret_cast<const g2_t*>(&W.W2[(4 * k4 + kk) * HID + 2 * o]), z[kk]);
                }
                if (far) {
#pragma unroll
                    for (int o = 0; o < HID / 2; ++o) {
                        float x, y;
                        gunpack2(acc[o], x, y);
                        s32[2 * o] += fmaxf(x, 0.f); s32[2 * o + 1] += fmaxf(y, 0.f);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < HID; ++c) Sd[lane * 33 + c] += (double)s32[c];       // fold the chunk into the FP64 sums (own row only)
        }
        if (rowok) {
#pragma unroll
            for (int c4 = 0; c4 < HID / 4; ++c4) {
                float4 o4;
                o4.x = (float)Sd[lane * 33 + 4 * c4]; o4.y = (float)Sd[lane * 33 + 4 * c4 + 1];
                o4.z = (float)Sd[lane * 33 + 4 * c4 + 2]; o4.w = (float)Sd[lane * 33 + 4 * c4 + 3];
                *reinterpret_cast<float4*>(a.S + ((int64_t)split * a.n_atoms + i) * HID + c4 * 4) = o4;
            }
        }
    }
}

#ifndef EPNN_CPU_EMU
cudaError_t launch_gnn_far_const(const Workspace& w, const StepW<float>& sw, int nsplit_far, cudaStream_t st, int* nl) {
    if (w.n_rowblk == 0) return cudaSuccess;
    if (!w.wf_host || !w.wf_dev) return cudaErrorInvalidValue;
    auto host = [&](const float* dev) { return w.wf_host + (dev - w.wf_dev); };
    FarW W;
    memcpy(W.W2, host(sw.W2), sizeof(W.W2));
    memcpy(W.b2, host(sw.b2), sizeof(W.b2));
    FarConstArgs fa;
    fa.blk = w.rowblk; fa.nsplit = nsplit_far; fa.n_atoms = w.n_atoms;
    fa.sys_off = w.sys_off; fa.rowptr = w.rowptr; fa.col = w.col;
    fa.u = (const float*)w.u; fa.v = (const float*)w.v; fa.S = (float*)w.S;
    fa.rgl_off = w.rgl_off; fa.sp_stamp = w.sp_stamp; fa.stamp = w.stamp;
    fa.unit_begin = w.blk_begin * nsplit_far; fa.unit_end = w.blk_end * nsplit_far;      // sharded call: the row blocks overlapping this rank's slice
    int grid = div_up(fa.unit_end - fa.unit_begin, FARC_NW);
    if (grid < 1) return cudaSuccess;
    if (grid > 2 * w.sm_count) grid = 2 * w.sm_count;
    const size_t smem = (size_t)FARC_NW * FARC_PW_BYTES;
    cudaError_t e = cudaFuncSetAttribute(gnn_far_const_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    gnn_far_const_kernel<<<grid, FARC_NW * 32, smem, st>>>(W, fa);
    ++*nl;
    return cudaGetLastError();
}
#endif
