// Message-passing pair kernel of the GNN layer.
//
// Replaces, per step t, reference charge_gn.py:62-70 (GNN_layer.call): build the (N*N, K) pair-input
// tensor, run message_fns[t] on ALL N^2 pairs and reduce_sum over j without a mask.  Here, exactly
// (SURVEY.md 7.2):
//     S_i = sum_{j real, incl. j = i} relu(W2^T relu(u_i + v_j + C^T e_ij) + b2)
//           + (npad - n) * relu(W2^T relu(u_i + b1) + b2)            (padded atoms: a_j = 0, e = 0)
// with u = A^T a, v = B^T a + b1 from the per-atom kernel and C^T e_ij only for pairs with e != 0.
// The linear last layer (W3, b3) is applied per atom afterwards (epnn_atom.cu).
//
// This file is the LARGE-system variant (n > SMALL_MAX, e.g. the 2220-atom protein); small systems take the
// bundle kernel (epnn_bundle.cu).  Work unit = one warp on a "row group" of 4 consecutive atoms i of one system.
// A tile is 4 rows x 8 j-slots = 32 pair slots; thread (pg, og) owns row pg and hidden columns og*4..og*4+3,
// so the sum over j stays in registers (FP64 accumulators) and is written once: no atomics, fixed order.
//   near phase : 8 CSR neighbours per row at a time; C^T e via tile_gemm<48>, then tile_gemm<32>
//   far phase  : 8 consecutive j at a time with the e != 0 members masked out; the j range is split across
//                warps when there are few row groups (partial-sum planes, added in fixed order per atom).
//
// Exact de-duplication of the far columns ("dedup_far", same idea as in the bundle kernel): a far message
// m(u_i, v_j) = relu(W2^T relu(u_i + v_j) + b2) depends on the column only through v_j = B [x_j | h_j | q_j] + b1.
// q is constant per system during the GNN layer, so when the v rows of a system are equal species by species
// (sp_check_kernel compares every row with the first atom of its species, every step) the O(n) far columns of a row
// collapse to one weighted slot per species:
//     sum_{j far} m(u_i, v_j) = sum_s (N_s - #{near neighbours of i with species s}) * m(u_i, v_rep(s))
// -- O(n * species) instead of O(n^2) for the step.  That is always the case at step 0 (h = 0) and after every step whose
// update left h species-wise constant (3 of the 5 steps of the reference's default decay_model_weights, whose update MLP
// is dead at some steps -- SURVEY trap 6);
// otherwise the full far phase below runs.  No approximation: identical messages are evaluated once and multiplied.
#include "epnn_internal.cuh"

template <typename R> struct GnnArgs {
    const int* rg_atom; int unit_begin; int n_units; int nsplit; int n_atoms; int skip_far; int plane;
    const int* atom_sys; const int* sys_off; const int* npad;
    const int* rowptr; const int* col; const int* pid;
    const float* e;
    const R* u; const R* v;
    const R* Cw; const R* W2; const R* b2; const R* b1;
    R* S;
    // far-column de-duplication (stamp == 0: off)
    const int* species; const int* rgl_off; const int* sp_tab; const int* sp_stamp; int stamp; int n_species;
};

template <typename R, bool LARGE, int NW>
__global__ void __launch_bounds__(NW * 32, sizeof(R) == 4 ? 2 : 1) gnn_pair_kernel(const GnnArgs<R> a) {
#ifdef EPNN_CPU_EMU
    unsigned char* smem_raw = reinterpret_cast<unsigned char*>(emu_smem);
#else
    extern __shared__ __align__(32) unsigned char smem_raw[];
#endif
    constexpr int EK = EKof<R>::v;
    R* sC = reinterpret_cast<R*>(smem_raw);          // [48][32]
    R* sW2 = sC + EK * HID;                          // [32][32]
    R* sb2 = sW2 + HID * HID;                        // [32]
    R* sb1 = sb2 + HID;                              // [32]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    R* at1 = sb1 + HID + warp * (32 * EK + 32 * HID);   // [32][EK] swizzled
    R* at2 = at1 + 32 * EK;                             // [32][32] swizzled
    int* slot_j = reinterpret_cast<int*>(sb1 + HID + NW * (32 * EK + 32 * HID)) + warp * 64;
    int* slot_p = slot_j + 32;

    for (int t = threadIdx.x; t < EK * HID; t += NW * 32) sC[t] = a.Cw[t];
    for (int t = threadIdx.x; t < HID * HID; t += NW * 32) sW2[t] = a.W2[t];
    if (threadIdx.x < HID) { sb2[threadIdx.x] = a.b2[threadIdx.x]; sb1[threadIdx.x] = a.b1[threadIdx.x]; }
    __syncthreads();

    const int pg = lane >> 3, og = lane & 7;
    const Vec4<R> b2v = ldv(sb2 + og * 4);
    const Vec4<R> b1v = ldv(sb1 + og * 4);

    for (int unit = a.unit_begin + blockIdx.x * NW + warp; unit < a.n_units; unit += gridDim.x * NW) {
        const int rg = LARGE ? unit / a.nsplit : unit;
        const int split = LARGE ? unit - rg * a.nsplit : 0;
        const int i0 = a.rg_atom[rg];
        const int sys = a.atom_sys[i0];
        const int a0 = a.sys_off[sys], a1 = a.sys_off[sys + 1];
        const int n = a1 - a0;
        const int padn = a.npad[sys] - n;
        const bool rowok = i0 + pg < a1;
        const int i = rowok ? i0 + pg : i0;
        const int rp0 = a.rowptr[i];
        const int rp1 = rowok ? a.rowptr[i + 1] : rp0;
        const int deg = rp1 - rp0;
        const Vec4<R> ur = rowok ? ldv(a.u + (int64_t)i * HID + og * 4) : vzero<R>();
        double rs0 = 0.0, rs1 = 0.0, rs2 = 0.0, rs3 = 0.0;
        R acc[8][4];
        // far columns de-duplicated for this system at this step?  (uniform over the warp: one system per unit)
        bool dd = false;
        const int* tab = a.sp_tab;
        if (a.stamp) {
            const int ti = a.rgl_off[sys] >> 3;
            dd = a.sp_stamp[2 * ti] != a.stamp && a.sp_stamp[2 * ti + 1] == 0;
            tab = a.sp_tab + ti * 32;
        }
        unsigned long long nc_lo = 0ull, nc_hi = 0ull;   // near neighbours of row pg per species, 8 bits each (degree <= 255 checked)

        // ---------------------------------------------------------------- near phase
        if (split == 0) {
            int maxdeg = deg;
            maxdeg = max(maxdeg, __shfl_xor_sync(0xffffffffu, maxdeg, 8));
            maxdeg = max(maxdeg, __shfl_xor_sync(0xffffffffu, maxdeg, 16));
            for (int b0 = 0; b0 < maxdeg; b0 += 8) {
                {
                    const int k = b0 + og;
                    int j = -2, p = -1;
                    if (k < deg) {
                        j = a.col[rp0 + k]; p = a.pid[rp0 + k];
                        if (dd) {
                            const int sj = a.species[j];
                            if (sj < 8) nc_lo += 1ull << (8 * sj); else nc_hi += 1ull << (8 * (sj - 8));
                        }
                    }
                    slot_j[lane] = j; slot_p[lane] = p;
                }
                __syncwarp();
#pragma unroll 4
                for (int f = lane; f < 32 * (EK / 4); f += 32) {       // stage the descriptor rows (gathered by pair id)
                    const int sl = f / (EK / 4), ch = f - sl * (EK / 4);
                    const int pp = slot_p[sl];
                    Vec4<R> ev = vzero<R>();
                    if (pp >= 0) ev = cvt4<R>(__ldg(reinterpret_cast<const float4*>(a.e + (int64_t)pp * EK) + ch));
                    stv(at1 + tile_off(sl, ch, EK), ev);
                }
                __syncwarp();
                zero_acc(acc);
                tile_gemm<R, EK, HID>(at1, sC, og * 4, acc, pg);
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const int jj = slot_j[pg * 8 + s];
                    Vec4<R> z = vzero<R>();
                    if (jj >= 0) {
                        const Vec4<R> vj = ldv(a.v + (int64_t)jj * HID + og * 4);
                        z.x = relu(acc[s][0] + ur.x + vj.x); z.y = relu(acc[s][1] + ur.y + vj.y);
                        z.z = relu(acc[s][2] + ur.z + vj.z); z.w = relu(acc[s][3] + ur.w + vj.w);
                    }
                    stv(at2 + tile_off(pg * 8 + s, og, HID), z);
                }
                __syncwarp();
                zero_acc(acc);
                tile_gemm<R, HID, HID>(at2, sW2, og * 4, acc, pg);
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    if (slot_j[pg * 8 + s] >= 0) {
                        rs0 += (double)relu(acc[s][0] + b2v.x); rs1 += (double)relu(acc[s][1] + b2v.y);
                        rs2 += (double)relu(acc[s][2] + b2v.z); rs3 += (double)relu(acc[s][3] + b2v.w);
                    }
                }
                __syncwarp();
            }
            if (dd) {                               // per-row totals: the 8 og lanes of a row each counted every 8th neighbour
#pragma unroll
                for (int m = 1; m < 8; m <<= 1) {
                    nc_lo += __shfl_xor_sync(0xffffffffu, nc_lo, m);
                    nc_hi += __shfl_xor_sync(0xffffffffu, nc_hi, m);
                }
            }
        }

        // ---------------------------------------------------------------- far phase, de-duplicated: species 0..7
        if (dd && split == 0) {
            int wg[8], rep[8];
            {
                const int4 c0 = __ldg(reinterpret_cast<const int4*>(tab)), c1 = __ldg(reinterpret_cast<const int4*>(tab) + 1);
                const int4 r0 = __ldg(reinterpret_cast<const int4*>(tab) + 4), r1 = __ldg(reinterpret_cast<const int4*>(tab) + 5);
                wg[0] = c0.x; wg[1] = c0.y; wg[2] = c0.z; wg[3] = c0.w; wg[4] = c1.x; wg[5] = c1.y; wg[6] = c1.z; wg[7] = c1.w;
                rep[0] = r0.x; rep[1] = r0.y; rep[2] = r0.z; rep[3] = r0.w; rep[4] = r1.x; rep[5] = r1.y; rep[6] = r1.z; rep[7] = r1.w;
            }
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                wg[s] = rowok ? wg[s] - (int)((nc_lo >> (8 * s)) & 0xFFull) : 0;     // far columns of species s (the self pair included)
                Vec4<R> z = vzero<R>();
                if (wg[s] > 0) {
                    const Vec4<R> vj = ldv(a.v + (int64_t)rep[s] * HID + og * 4);
                    z.x = relu(ur.x + vj.x); z.y = relu(ur.y + vj.y); z.z = relu(ur.z + vj.z); z.w = relu(ur.w + vj.w);
                }
                stv(at2 + tile_off(pg * 8 + s, og, HID), z);
            }
            __syncwarp();
            zero_acc(acc);
            tile_gemm<R, HID, HID>(at2, sW2, og * 4, acc, pg);
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                if (wg[s] > 0) {
                    const double wd = (double)wg[s];
                    rs0 += wd * (double)relu(acc[s][0] + b2v.x); rs1 += wd * (double)relu(acc[s][1] + b2v.y);
                    rs2 += wd * (double)relu(acc[s][2] + b2v.z); rs3 += wd * (double)relu(acc[s][3] + b2v.w);
                }
            }
            __syncwarp();
        }

        // ---------------------------------------------------------------- far phase, column by column
        if (!a.skip_far && !dd) {
            int clen = (n + a.nsplit - 1) / a.nsplit;
            clen = (clen + 7) & ~7;
            const int jlo = min(a1, a0 + split * clen), jhi = min(a1, jlo + clen);
            int ptr = rp0;
            while (ptr < rp1 && a.col[ptr] < jlo) ++ptr;
            for (int jb = jlo; jb < jhi; jb += 8) {
                unsigned m = 0u;
                while (ptr < rp1 && a.col[ptr] < jb + 8) { m |= 1u << (a.col[ptr] - jb); ++ptr; }
                unsigned okm = 0u;
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const int j = jb + s;
                    const bool ok = rowok && j < jhi && !((m >> s) & 1u);
                    Vec4<R> z = vzero<R>();
                    if (ok) {
                        okm |= 1u << s;
                        const Vec4<R> vj = ldv(a.v + (int64_t)j * HID + og * 4);
                        z.x = relu(ur.x + vj.x); z.y = relu(ur.y + vj.y); z.z = relu(ur.z + vj.z); z.w = relu(ur.w + vj.w);
                    }
                    stv(at2 + tile_off(pg * 8 + s, og, HID), z);
                }
                __syncwarp();
                zero_acc(acc);
                tile_gemm<R, HID, HID>(at2, sW2, og * 4, acc, pg);
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    if ((okm >> s) & 1u) {
                        rs0 += (double)relu(acc[s][0] + b2v.x); rs1 += (double)relu(acc[s][1] + b2v.y);
                        rs2 += (double)relu(acc[s][2] + b2v.z); rs3 += (double)relu(acc[s][3] + b2v.w);
                    }
                }
                __syncwarp();
            }
        }
        {
            // one more tile: slot 0 = the weighted pad pseudo-pair (a_j = 0, e = 0 => v = b1), slots 1..7 = species 8..14 of
            // the de-duplicated far phase (only the 10-wide element table has a ninth species)
            const bool hi_species = dd && a.n_species > 8;
            if (split == 0 && (padn > 0 || hi_species)) {
                int wg[8], rep[8];
#pragma unroll
                for (int s = 0; s < 8; ++s) { wg[s] = 0; rep[s] = 0; }
                if (hi_species) {
                    const int4 c2 = __ldg(reinterpret_cast<const int4*>(tab) + 2), c3 = __ldg(reinterpret_cast<const int4*>(tab) + 3);
                    const int4 r2 = __ldg(reinterpret_cast<const int4*>(tab) + 6), r3 = __ldg(reinterpret_cast<const int4*>(tab) + 7);
                    wg[1] = c2.x; wg[2] = c2.y; wg[3] = c2.z; wg[4] = c2.w; wg[5] = c3.x; wg[6] = c3.y; wg[7] = c3.z;
                    rep[1] = r2.x; rep[2] = r2.y; rep[3] = r2.z; rep[4] = r2.w; rep[5] = r3.x; rep[6] = r3.y; rep[7] = r3.z;
#pragma unroll
                    for (int s = 1; s < 8; ++s) wg[s] = rowok ? wg[s] - (int)((nc_hi >> (8 * (s - 1))) & 0xFFull) : 0;
                }
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    Vec4<R> z = vzero<R>();
                    if (s == 0) {
                        if (rowok && padn > 0) { z.x = relu(ur.x + b1v.x); z.y = relu(ur.y + b1v.y); z.z = relu(ur.z + b1v.z); z.w = relu(ur.w + b1v.w); }
                    } else if (wg[s] > 0) {
                        const Vec4<R> vj = ldv(a.v + (int64_t)rep[s] * HID + og * 4);
                        z.x = relu(ur.x + vj.x); z.y = relu(ur.y + vj.y); z.z = relu(ur.z + vj.z); z.w = relu(ur.w + vj.w);
                    }
                    stv(at2 + tile_off(pg * 8 + s, og, HID), z);
                }
                __syncwarp();
                zero_acc(acc);
                tile_gemm<R, HID, HID>(at2, sW2, og * 4, acc, pg);
                if (rowok && padn > 0) {
                    const R wgt = (R)padn;
                    rs0 += (double)(wgt * relu(acc[0][0] + b2v.x)); rs1 += (double)(wgt * relu(acc[0][1] + b2v.y));
                    rs2 += (double)(wgt * relu(acc[0][2] + b2v.z)); rs3 += (double)(wgt * relu(acc[0][3] + b2v.w));
                }
#pragma unroll
                for (int s = 1; s < 8; ++s) {
                    if (wg[s] > 0) {
                        const double wd = (double)wg[s];
                        rs0 += wd * (double)relu(acc[s][0] + b2v.x); rs1 += wd * (double)relu(acc[s][1] + b2v.y);
                        rs2 += wd * (double)relu(acc[s][2] + b2v.z); rs3 += wd * (double)relu(acc[s][3] + b2v.w);
                    }
                }
                __syncwarp();
            }
        }

        if (rowok) {
            Vec4<R> out; out.x = (R)rs0; out.y = (R)rs1; out.z = (R)rs2; out.w = (R)rs3;
            stv(a.S + ((int64_t)(a.plane + split) * a.n_atoms + i) * HID + og * 4, out);
        }
    }
}

template <typename R> static size_t gnn_smem_bytes(int nw) {
    constexpr int EK = EKof<R>::v;
    return sizeof(R) * (EK * HID + HID * HID + 2 * HID + (size_t)nw * (32 * EK + 32 * HID)) + sizeof(int) * nw * 64;
}

#ifndef EPNN_CPU_EMU
template <typename R, bool LARGE, int NW>
static cudaError_t launch_one(const GnnArgs<R>& ga, int sm_count, cudaStream_t st) {
    const size_t smem = gnn_smem_bytes<R>(NW);
    cudaError_t e = cudaFuncSetAttribute(gnn_pair_kernel<R, LARGE, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int per_sm = sizeof(R) == 4 ? 2 : 1;
    int grid = div_up(ga.n_units - ga.unit_begin, NW);
    if (grid < 1) return cudaSuccess;
    if (grid > sm_count * per_sm) grid = sm_count * per_sm;      // persistent: warps stride over the units
    gnn_pair_kernel<R, LARGE, NW><<<grid, NW * 32, smem, st>>>(ga);
    return cudaGetLastError();
}

template <typename R>
cudaError_t launch_gnn_pair(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* nl) {
    GnnArgs<R> ga;
    ga.n_atoms = w.n_atoms; ga.atom_sys = w.atom_sys; ga.sys_off = w.sys_off; ga.npad = w.npad;
    ga.rowptr = w.rowptr; ga.col = w.col; ga.pid = w.pid; ga.e = w.e;
    ga.u = (const R*)w.u; ga.v = (const R*)w.v; ga.Cw = sw.Cw; ga.W2 = sw.W2; ga.b2 = sw.b2; ga.b1 = sw.b1;
    ga.S = (R*)w.S;
    ga.species = w.species; ga.rgl_off = w.rgl_off; ga.sp_tab = w.sp_tab; ga.sp_stamp = w.sp_stamp; ga.stamp = w.stamp;
    ga.n_species = w.n_species;
    cudaError_t e = cudaSuccess;
    if (w.n_rg_large > 0) {      // small systems (n <= SMALL_MAX) are handled by the bundle kernel (epnn_bundle.cu)
        // tensor-core mode: this kernel does the near pairs + pad pair only (one unit per row group, last plane)
        const int skip_far = w.far_kernel != FAR_SIMT;
        const int ns = skip_far ? 1 : w.nsplit;
        ga.skip_far = skip_far; ga.plane = skip_far ? w.nsplit - 1 : 0;
        // sharded call: the row groups that overlap this rank's slice (rows of a boundary group that lie outside it are computed
        // from whatever their u row holds and never read: S is only consumed for owned rows)
        ga.rg_atom = w.rg_large; ga.nsplit = ns;
        ga.unit_begin = w.rg_begin * ns; ga.n_units = w.rg_end * ns;
        e = launch_one<R, true, 8>(ga, w.sm_count, st);
        ++*nl;
    }
    return e;
}

template cudaError_t launch_gnn_pair<float>(const Workspace&, const StepW<float>&, cudaStream_t, int*);
template cudaError_t launch_gnn_pair<double>(const Workspace&, const StepW<double>&, cudaStream_t, int*);
#endif

// ------------------------------------------------------------------------------------------------
// Species tables of the large systems (built once per chunk) and the per-step equality check of their v rows.
__global__ void sp_tab_init_kernel(int n_entries, int* __restrict__ tab, int* __restrict__ stamp) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_entries * 32) tab[t] = (t & 31) < 16 ? 0 : 0x7fffffff;       // counts | first atom (min)
    if (t < n_entries * 2) stamp[t] = 0;
}

// One thread per atom; the lanes of a warp that hit the same (system, species) entry are combined first
// (match_any), so the table sees one atomicAdd / atomicMin per warp and species.  Integer atomics: order-independent.
__global__ void sp_tab_fill_kernel(int n_atoms, const int* __restrict__ atom_sys, const int* __restrict__ sys_off,
                                   const int* __restrict__ species, const int* __restrict__ rgl_off,
                                   const int* __restrict__ deg, int* __restrict__ tab, int* __restrict__ stamp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int key = -1;
    if (i < n_atoms) {
        const int s = atom_sys[i];
        if (sys_off[s + 1] - sys_off[s] > SMALL_MAX) {
            const int ti = rgl_off[s] >> 3;
            key = ti * 16 + (species[i] & 15);
            if (deg[i] > 255) stamp[2 * ti + 1] = 1;      // the kernel's packed per-species neighbour counts hold 8 bits
        }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) {          // lowest lane of the group = lowest atom index
        int* ent = tab + (key >> 4) * 32;
        atomicAdd(ent + (key & 15), __popc(peers));
        atomicMin(ent + 16 + (key & 15), i);
    }
}

// 8 lanes per atom (4 of the 32 columns each): v_i against v of the first atom of i's species in i's system.
// A mismatch stamps the system with the current step: its far phase then runs column by column.
template <typename R>
__global__ void sp_check_kernel(int n_atoms, const int* __restrict__ atom_sys, const int* __restrict__ sys_off,
                                const int* __restrict__ species, const int* __restrict__ rgl_off, const int* __restrict__ tab,
                                const R* __restrict__ v, int* __restrict__ stamp, int cur) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t i = g >> 3;
    const int og = (int)(g & 7);
    if (i >= n_atoms) return;
    const int s = atom_sys[i];
    if (sys_off[s + 1] - sys_off[s] <= SMALL_MAX) return;
    const int ti = rgl_off[s] >> 3;
    const int rp = tab[ti * 32 + 16 + (species[i] & 15)];
    if (rp == (int)i) return;
    const Vec4<R> x = ldv(v + i * HID + og * 4), y = ldv(v + (int64_t)rp * HID + og * 4);
    if (!(x.x == y.x && x.y == y.y && x.z == y.z && x.w == y.w)) stamp[2 * ti] = cur;
}

// statistics: atoms of the systems whose far phase is de-duplicated at this step
__global__ void sp_tally_kernel(int n_entries, const int* __restrict__ tab, const int* __restrict__ stamp, int cur,
                                unsigned long long* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_entries) return;
    int n = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) n += tab[t * 32 + k];
    if (n > 0 && stamp[2 * t] != cur && stamp[2 * t + 1] == 0) atomicAdd(out, (unsigned long long)n);
}

#ifndef EPNN_CPU_EMU
cudaError_t launch_sp_tab_build(const Workspace& w, cudaStream_t st, int* nl) {
    if (w.n_rg_large == 0 || w.n_sp_tab == 0) return cudaSuccess;
    sp_tab_init_kernel<<<div_up((int64_t)w.n_sp_tab * 32, 256), 256, 0, st>>>(w.n_sp_tab, w.sp_tab, w.sp_stamp);
    sp_tab_fill_kernel<<<div_up(w.n_atoms, 256), 256, 0, st>>>(w.n_atoms, w.atom_sys, w.sys_off, w.species, w.rgl_off, w.deg_all ? w.deg_all : w.deg,
                                                                w.sp_tab, w.sp_stamp);
    *nl += 2;
    return cudaGetLastError();
}

template <typename R> cudaError_t launch_sp_check(const Workspace& w, cudaStream_t st, int* nl) {
    if (w.n_rg_large == 0 || w.stamp == 0) return cudaSuccess;
    sp_check_kernel<R><<<div_up((int64_t)w.n_atoms * 8, 256), 256, 0, st>>>(w.n_atoms, w.atom_sys, w.sys_off, w.species, w.rgl_off,
                                                                             w.sp_tab, (const R*)w.v, w.sp_stamp, w.stamp);
    ++*nl;
    if (w.dedup_rows) {
        sp_tally_kernel<<<div_up(w.n_sp_tab, 256), 256, 0, st>>>(w.n_sp_tab, w.sp_tab, w.sp_stamp, w.stamp, w.dedup_rows);
        ++*nl;
    }
    return cudaGetLastError();
}
template cudaError_t launch_sp_check<float>(const Workspace&, cudaStream_t, int*);
template cudaError_t launch_sp_check<double>(const Workspace&, cudaStream_t, int*);
#endif
