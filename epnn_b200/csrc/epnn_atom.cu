// Per-atom kernel: everything between two pair kernels, fused.
//
//   ATOM_UPDATE  finishes message-passing step t (reference charge_gn.py:70-74):
//                  M_i = W3^T S_i + npad * b3        (linear last message layer hoisted out of sum_j)
//                  h_i = update_fn([h_i | M_i])      80 -> 32 relu -> 32 relu -> 48
//                (node_mask is 1 for every atom that exists here; padded atoms are never materialised)
//                The linear maps around the two ReLU layers are composed on the host (float64, exact algebra): with
//                l2 = the update MLP's last hidden layer (the state carried between steps instead of h),
//                  l1  = relu([U3 U1_h ; W3 U1_M]^T [l2_prev | S] + c1 + U1_h^T c3 + npad U1_M^T b3)     64 -> 32
//                  l2  = relu(U2^T l1 + c2)                                                             32 -> 32
//                  u|v = (U3 Ah)^T l2 + (Ax[species] + c3^T Ah) + q Aq                                  32 -> 64
//                -- 5 120 MAC per atom and step instead of 9 216; h = U3^T l2 + c3 itself is only formed at the last step.
//   ATOM_QUPDATE finishes electron-passing pass t (charge_gn.py:116-118):
//                  q_i += sum over the CSR row of i, in column order, of sign(j - i) * delta_pair
//                fixed order, FP64, no atomics: deterministic, and sum_i q_i is conserved by construction.
//   ATOM_PROJECT first-layer projections for the next pair kernel (SURVEY.md 7.2):
//                  u_i = A^T [x_i|h_i|q_i],  v_i = B^T [x_i|h_i|q_i] + b1
//                with the one-hot x part folded into a per-species table.
//   ATOM_OUTPUT  q -> float32 / float64 output buffers.
//
// Work unit = one warp on a tile of 32 consecutive atoms; the dense layers run through tile_gemm.
#include "epnn_internal.cuh"

template <typename R, typename IO> __device__ __forceinline__ Vec4<R> ld_io(const IO* p) {
    const Vec4<IO> t = ldv(p);
    Vec4<R> r; r.x = (R)t.x; r.y = (R)t.y; r.z = (R)t.z; r.w = (R)t.w; return r;
}
template <typename R, typename IO> __device__ __forceinline__ void st_io(IO* p, Vec4<R> v) {
    Vec4<IO> t; t.x = (IO)v.x; t.y = (IO)v.y; t.z = (IO)v.z; t.w = (IO)v.w; stv(p, t);
}

#ifndef ATOM_NW
#define ATOM_NW 12
#endif
#ifndef ATOM_UNR
#define ATOM_UNR 2
#endif
#ifndef ATOM_PREFETCH
#define ATOM_PREFETCH 1      // measured: per-atom kernels -5 % (tools/gpu_ab_atom.sh); keeping 4 CSR entries in flight or 14 warps: no change
#endif
#ifdef EPNN_CPU_EMU
__device__ __forceinline__ void prefetch_l2(const void*) {}
#else
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
#endif
#define ATOM_W_UPD (64 * HID + 2 * HID + HID * HID + HID + HID * HD + HD)                    // 4752
#define ATOM_W_PROJ (HID * 64 + 64 + MAX_SPECIES * 64)                                      // 3136
#define ATOM_TILE (32 * 64 + 32 * HID)                                                      // 3072 per warp

// SCOPED = false: every atom (unsharded calls; the scope fields of AtomArgs are ignored and cost nothing).
template <typename R, int NW, typename IO, bool SCOPED>
__global__ void __launch_bounds__(NW * 32) atom_kernel(const AtomArgs<R, IO> a) {
#ifdef EPNN_CPU_EMU
    unsigned char* smem_raw = reinterpret_cast<unsigned char*>(emu_smem);
#else
    extern __shared__ __align__(32) unsigned char smem_raw[];
#endif
    R* sHG = reinterpret_cast<R*>(smem_raw);   // [64][32]  [U3 U1_h ; W3 U1_M]
    R* scb = sHG + 64 * HID;                   // [32]      first-layer bias of this step
    R* sg = scb + HID;                         // [32]      U1_M^T b3
    R* sU2 = sg + HID;                         // [32][32]
    R* sc2 = sU2 + HID * HID;                  // [32]
    R* sU3 = sc2 + HID;                        // [32][48]
    R* sc3 = sU3 + HID * HD;                   // [48]
    R* sP = sc3 + HD;                          // [32][64]  U3 Ah64 of the next pair kernel
    R* sAq = sP + HID * 64;                    // [64]
    R* sAx = sAq + 64;                         // [MAX_SPECIES][64]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    R* T64 = sAx + MAX_SPECIES * 64 + warp * ATOM_TILE;    // [32][64] = [l2_prev | S]
    R* T32 = T64 + 32 * 64;                                // [32][32]
    R* T32b = T64;                                         // [32][32] l2 tile; aliases T64 once the first layer is done
    R* slot_q = sAx + MAX_SPECIES * 64 + NW * ATOM_TILE + warp * 64;   // [32]
    R* slot_np = slot_q + 32;                                         // [32] npad as real
    int* slot_sp = reinterpret_cast<int*>(sAx + MAX_SPECIES * 64 + NW * ATOM_TILE + NW * 64) + warp * 64;   // [32]
    int* slot_ns = slot_sp + 32;                                      // [32] number of S partial planes

    const bool do_upd = a.mode & ATOM_UPDATE, do_q = a.mode & ATOM_QUPDATE, do_proj = a.mode & ATOM_PROJECT;
    const bool first = a.mode & ATOM_FIRST, write_h = a.mode & ATOM_WRITE_H;
    if (do_upd) {
        for (int t = threadIdx.x; t < 64 * HID; t += NW * 32) sHG[t] = a.HG[t];
        for (int t = threadIdx.x; t < HID * HID; t += NW * 32) sU2[t] = a.upd.U2[t];
        if (write_h) for (int t = threadIdx.x; t < HID * HD; t += NW * 32) sU3[t] = a.upd.U3[t];
        if (threadIdx.x < HID) { scb[threadIdx.x] = a.cb[threadIdx.x]; sg[threadIdx.x] = a.g[threadIdx.x]; sc2[threadIdx.x] = a.upd.c2[threadIdx.x]; }
        if (threadIdx.x < HD) sc3[threadIdx.x] = a.upd.c3[threadIdx.x];
    }
    if (do_proj) {
        if (!a.h_is_zero) for (int t = threadIdx.x; t < HID * 64; t += NW * 32) sP[t] = a.Pf[t];
        for (int t = threadIdx.x; t < MAX_SPECIES * 64; t += NW * 32) sAx[t] = a.Ax[t];
        if (threadIdx.x < 64) sAq[threadIdx.x] = a.Aq64[threadIdx.x];
    }
    __syncthreads();

    const int pg = lane >> 3, og = lane & 7;
    const int n_tiles = (a.n_atoms + 31) / 32;
    R acc[8][4];

    for (int tile = blockIdx.x * NW + warp; tile < n_tiles; tile += gridDim.x * NW) {
        const int base = tile * 32;
        const int me = base + lane;
        const bool me_ok = me < a.n_atoms;
#if ATOM_PREFETCH
        {   // this warp's NEXT tile -> L2 while the current one computes: its l2 rows (4 KB, one 128-byte line per lane) and,
            // for the update, the first partial-sum plane of S (the only plane small systems have)
            const int64_t nb = (int64_t)(tile + gridDim.x * NW) * 32;
            if (nb + lane < a.n_atoms) {
                if ((do_upd && !first) || (do_proj && !do_upd && !a.h_is_zero)) prefetch_l2(a.l2 + (nb + lane) * HID);
                if (do_upd) prefetch_l2(a.Spart + (nb + lane) * HID);
            }
        }
#endif
        // ---------------- per-slot scalars (lane = slot)
        {
            int sp = 0, ns = 0; R npf = R(0);            // ns = 0 marks a slot this launch does not touch
            double qv = 0.0;
            bool in = me_ok;
            int sys = 0, nat = 0;
            if (me_ok) {
                sys = a.atom_sys[me];
                nat = a.sys_off[sys + 1] - a.sys_off[sys];
                if (SCOPED && a.scope && nat > SMALL_MAX) in = a.scope == 1 ? (me >= a.row_lo && me < a.row_hi) : a.active[me] != 0;
            }
            if (in) {
                sp = a.species[me];
                ns = nat > SMALL_MAX ? a.nsplit : 1;
                npf = (R)a.npad[sys];
                qv = a.q[me];
                if (do_q) {
                    const int r0 = a.rowptr[me], r1 = a.rowptr[me + 1];
                    for (int k = r0; k < r1; ++k) {          // fixed (ascending column) order
                        const double d = (double)a.delta[a.pid[k]];
                        qv += a.col[k] > me ? d : -d;
                    }
                    a.q[me] = qv;
                }
                if (a.mode & ATOM_OUTPUT) {
                    if (a.q_out) a.q_out[me] = (float)qv;
                    if (a.q_out64) a.q_out64[me] = qv;
                }
            }
            slot_sp[lane] = sp; slot_ns[lane] = ns; slot_np[lane] = npf; slot_q[lane] = (R)qv;
        }
        __syncwarp();
        if (!do_upd && !do_proj) continue;
        if (SCOPED && a.scope && !__any_sync(0xffffffffu, slot_ns[lane] > 0)) continue;      // nothing of this tile belongs to the launch
        unsigned okm = 0u;                                                         // bit s: slot pg * 8 + s belongs to the launch
        if (!SCOPED) {
            const int left = a.n_atoms - (base + pg * 8);
            okm = left >= 8 ? 0xFFu : (left > 0 ? (1u << left) - 1u : 0u);
        } else {
            const int4 n0 = *reinterpret_cast<const int4*>(slot_ns + pg * 8), n1 = *reinterpret_cast<const int4*>(slot_ns + pg * 8 + 4);
            okm = (n0.x > 0) | (n0.y > 0) << 1 | (n0.z > 0) << 2 | (n0.w > 0) << 3 | (n1.x > 0) << 4 | (n1.y > 0) << 5 | (n1.z > 0) << 6 | (n1.w > 0) << 7;
        }

        if (do_upd) {
            // (1) [l2_prev | S] tile: l2 of the previous step (zeros at the first step: h = 0), S = partial planes summed in fixed order
#pragma unroll 2
            for (int f = lane; f < 32 * (HID / 4); f += 32) {
                const int sl = f >> 3, ch = f & 7;
                const int at = base + sl;
                Vec4<R> lv = vzero<R>(), sv = vzero<R>();
                const int ns = slot_ns[sl];
                if (ns > 0) {
                    if (!first) lv = ldv(a.l2 + (int64_t)at * HID + ch * 4);
                    for (int sp = 0; sp < ns; ++sp)
                        sv = vadd(sv, ld_io<R, IO>(a.Spart + ((int64_t)sp * a.n_atoms + at) * HID + ch * 4));
                }
                stv(T64 + tile_off(sl, ch, 64), lv);
                stv(T64 + tile_off(sl, 8 + ch, 64), sv);
            }
            __syncwarp();
            // (2) first layer with W3 / U3 folded in: relu([U3 U1_h ; W3 U1_M]^T [l2_prev | S] + cb + npad * g)
            zero_acc(acc);
            tile_gemm_unr<R, 64, HID, ATOM_UNR>(T64, sHG, og * 4, acc, pg);
            {
                const Vec4<R> cv = ldv(scb + og * 4);
                const Vec4<R> gv = ldv(sg + og * 4);
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const R np = slot_np[pg * 8 + s];
                    Vec4<R> z;
                    z.x = relu(fma(np, gv.x, acc[s][0] + cv.x)); z.y = relu(fma(np, gv.y, acc[s][1] + cv.y));
                    z.z = relu(fma(np, gv.z, acc[s][2] + cv.z)); z.w = relu(fma(np, gv.w, acc[s][3] + cv.w));
                    stv(T32 + tile_off(pg * 8 + s, og, HID), z);
                }
            }
            __syncwarp();
            // (3) second layer: l2 = relu(U2^T l1 + c2)   (T64 is dead now; the l2 tile reuses its head)
            zero_acc(acc);
            tile_gemm_unr<R, HID, HID, ATOM_UNR>(T32, sU2, og * 4, acc, pg);
            {
                const Vec4<R> cv = ldv(sc2 + og * 4);
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    Vec4<R> z; z.x = relu(acc[s][0] + cv.x); z.y = relu(acc[s][1] + cv.y); z.z = relu(acc[s][2] + cv.z); z.w = relu(acc[s][3] + cv.w);
                    const int at = base + pg * 8 + s;
                    if ((okm >> s) & 1u) stv(a.l2 + (int64_t)at * HID + og * 4, z);
                    stv(T32b + tile_off(pg * 8 + s, og, HID), z);
                }
            }
            __syncwarp();
            // (4) last message-passing step only: the hidden state itself, h = U3^T l2 + c3 (columns 0..31, then 32..47)
            if (write_h) {
                zero_acc(acc);
                tile_gemm<R, HID, HD>(T32b, sU3, og * 4, acc, pg);
                {
                    const Vec4<R> cv = ldv(sc3 + og * 4);
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        Vec4<R> hv; hv.x = acc[s][0] + cv.x; hv.y = acc[s][1] + cv.y; hv.z = acc[s][2] + cv.z; hv.w = acc[s][3] + cv.w;
                        const int at = base + pg * 8 + s;
                        if ((okm >> s) & 1u) stv(a.h + (int64_t)at * HD + og * 4, hv);
                    }
                }
                zero_acc(acc);
                tile_gemm<R, HID, HD>(T32b, sU3, HID + (og & 3) * 4, acc, pg);
                if (og < 4) {
                    const Vec4<R> cv = ldv(sc3 + HID + og * 4);
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        Vec4<R> hv; hv.x = acc[s][0] + cv.x; hv.y = acc[s][1] + cv.y; hv.z = acc[s][2] + cv.z; hv.w = acc[s][3] + cv.w;
                        const int at = base + pg * 8 + s;
                        if ((okm >> s) & 1u) stv(a.h + (int64_t)at * HD + HID + og * 4, hv);
                    }
                }
            }
        } else if (do_proj && !a.h_is_zero) {
#pragma unroll 2
            for (int f = lane; f < 32 * (HID / 4); f += 32) {            // l2 of the last message-passing step
                const int sl = f >> 3, ch = f & 7;
                const int at = base + sl;
                Vec4<R> lv = vzero<R>();
                if (slot_ns[sl] > 0) lv = ldv(a.l2 + (int64_t)at * HID + ch * 4);
                stv(T32b + tile_off(sl, ch, HID), lv);
            }
            __syncwarp();
        }

        if (do_proj) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {           // half 0 -> u (a_i block), half 1 -> v (a_j block, + b1)
                zero_acc(acc);
                if (!a.h_is_zero) tile_gemm_unr<R, HID, 64, ATOM_UNR>(T32b, sP, half * HID + og * 4, acc, pg);
                const Vec4<R> aq = ldv(sAq + half * HID + og * 4);
                IO* dst = half == 0 ? a.u : a.v;
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const int at = base + pg * 8 + s;
                    if ((okm >> s) & 1u) {
                        const Vec4<R> ax = ldv(sAx + slot_sp[pg * 8 + s] * 64 + half * HID + og * 4);
                        const R qv = slot_q[pg * 8 + s];
                        Vec4<R> o;
                        o.x = acc[s][0] + fma(qv, aq.x, ax.x); o.y = acc[s][1] + fma(qv, aq.y, ax.y);
                        o.z = acc[s][2] + fma(qv, aq.z, ax.z); o.w = acc[s][3] + fma(qv, aq.w, ax.w);
                        st_io<R, IO>(dst + (int64_t)at * HID + og * 4, o);
                    }
                }
            }
        }
        __syncwarp();
    }
}

#ifndef EPNN_CPU_EMU
template <typename R, typename IO>
cudaError_t launch_atom_io(const Workspace& w, int mode, const StepW<R>* prev, const UpdW<R>* upd, const StepW<R>* next,
                           int h_is_zero, float* q_out, double* q_out64, cudaStream_t st, int* nl, int scope) {
    if (w.n_atoms == 0) return cudaSuccess;
    const AtomKernel k = scope ? w.kc.atom_scoped : w.kc.atom;
    if constexpr (sizeof(R) == 4) {
        if (k == ATOM_K_CONST) return launch_atom_const(w, mode, prev, upd, next, h_is_zero, q_out, q_out64, st, nl);   // experimental (epnn_atom_const.cu)
    }
    constexpr int NW = sizeof(R) == 4 ? ATOM_NW : 4;
    AtomArgs<R, IO> aa;
    memset(&aa, 0, sizeof(aa));
    aa.n_atoms = w.n_atoms; aa.mode = mode; aa.nsplit = w.nsplit; aa.h_is_zero = h_is_zero;
    aa.atom_sys = w.atom_sys; aa.sys_off = w.sys_off; aa.npad = w.npad; aa.species = w.species;
    aa.Spart = (const IO*)w.S; aa.h = (R*)w.h; aa.l2 = (R*)w.l2;
    if (mode & ATOM_UPDATE) { aa.HG = prev->HG; aa.g = prev->g; aa.upd = *upd; aa.cb = (mode & ATOM_FIRST) ? upd->c1 : upd->cb1; }
    aa.rowptr = w.rowptr; aa.col = w.col; aa.pid = w.pid; aa.delta = (const IO*)w.delta; aa.q = w.q;
    if (mode & ATOM_PROJECT) { aa.Pf = next->Pf; aa.Aq64 = next->Aq64; aa.Ax = h_is_zero ? next->Ax64 : next->Axf; }
    aa.u = (IO*)w.u; aa.v = (IO*)w.v; aa.q_out = q_out; aa.q_out64 = q_out64;
    aa.scope = scope; aa.row_lo = w.row_lo; aa.row_hi = w.row_hi; aa.active = w.active;
    if constexpr (sizeof(R) == 4 && sizeof(IO) == 4) {       // FP32 calls: launches with a dense layer run on the warp-level tensor path
        if (k == ATOM_K_MMA && ((mode & ATOM_UPDATE) || ((mode & ATOM_PROJECT) && !h_is_zero))) return launch_atom_mma(w, aa, st, nl);
    }
    const size_t smem = sizeof(R) * (ATOM_W_UPD + ATOM_W_PROJ + (size_t)NW * ATOM_TILE + NW * 64) + sizeof(int) * NW * 64;
    cudaError_t e = cudaFuncSetAttribute(scope ? atom_kernel<R, NW, IO, true> : atom_kernel<R, NW, IO, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int grid = div_up(div_up(w.n_atoms, 32), NW);
    if (grid > w.sm_count) grid = w.sm_count;
    if (scope) atom_kernel<R, NW, IO, true><<<grid, NW * 32, smem, st>>>(aa);
    else atom_kernel<R, NW, IO, false><<<grid, NW * 32, smem, st>>>(aa);
    ++*nl;
    return cudaGetLastError();
}

template <typename R>
cudaError_t launch_atom(const Workspace& w, int mode, const StepW<R>* prev, const UpdW<R>* upd, const StepW<R>* next,
                        int h_is_zero, float* q_out, double* q_out64, cudaStream_t st, int* nl, int scope) {
    return launch_atom_io<R, R>(w, mode, prev, upd, next, h_is_zero, q_out, q_out64, st, nl, scope);
}
// "mixed" precision: FP64 per-atom arithmetic and state, FP32 buffers towards the pair kernels
cudaError_t launch_atom_mixed(const Workspace& w, int mode, const StepW<double>* prev, const UpdW<double>* upd, const StepW<double>* next,
                              int h_is_zero, float* q_out, double* q_out64, cudaStream_t st, int* nl, int scope) {
    return launch_atom_io<double, float>(w, mode, prev, upd, next, h_is_zero, q_out, q_out64, st, nl, scope);
}

template cudaError_t launch_atom<float>(const Workspace&, int, const StepW<float>*, const UpdW<float>*, const StepW<float>*,
                                        int, float*, double*, cudaStream_t, int*, int);
template cudaError_t launch_atom<double>(const Workspace&, int, const StepW<double>*, const UpdW<double>*, const StepW<double>*,
                                         int, float*, double*, cudaStream_t, int*, int);
#endif
