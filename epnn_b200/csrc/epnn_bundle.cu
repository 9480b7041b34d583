// Pair kernels for SMALL systems (n <= SMALL_MAX atoms): the batched many-molecule path (BASELINE config 4).
//
// A "bundle" is a run of consecutive whole systems with at most BUNDLE_ATOMS atoms in total; one warp owns
// one bundle at a time and keeps everything it gathers from in its private slice of shared memory:
//     uv[atom][64]  = first-layer projections u_i | v_i of the bundle's atoms   (staged once per bundle, coalesced)
//     S[atom][32]   = sum_j relu(W2^T relu(...) + b2) accumulators (GNN)          (written back once per bundle)
// so the per-pair work never waits on a global gather, tiles are packed densely across the rows and systems of
// the bundle (no per-row padding), and every UNORDERED e != 0 pair is evaluated once for both directions,
// which share C^T e_ij (e is symmetric):
//
//   GNN step (replaces reference charge_gn.py:62-70, GNN_layer.call, per step t):
//     near tiles: 32 unordered pairs; ce = C^T e  (FP32: (B^T C)^T (B^T e) in the rank-16 descriptor basis);  m_ij = relu(W2^T relu(ce + u_i + v_j) + b2) -> S_i,
//                                                  m_ji = relu(W2^T relu(ce + u_j + v_i) + b2) -> S_j
//     far tiles : 32 ORDERED pairs (i,j) with e_ij == 0 (self pair, pairs beyond the cutoff) from a precomputed
//                 per-bundle list, plus one weighted pseudo-pair per atom for the (npad - n) padded atoms
//                 (a_j = 0, e = 0  =>  v = b1), exactly the reference's unmasked reduce_sum over all N columns.
//   EPN pass (replaces charge_gn.py:101-116, EPN_layer.call, per pass t): near tiles only;
//     delta_p = 0.5 (w3 . m_ij - w3 . m_ji) * is_near_p, written per unordered pair (the +/- scatter into q is the
//     per-atom kernel's fixed-order CSR reduction).
//
// The scatter into S is a warp-private, fixed-order segmented sum over the sorted targets (scatter_sorted): no atomics,
// bitwise reproducible.  Only the descriptor rows (EK floats per pair: 64 B in FP32, streamed once per launch) and the index lists come from
// global memory inside the tile loop, and both are prefetched one tile ahead into registers.
#include "epnn_internal.cuh"

#ifndef EPN_NW
#define EPN_NW 8
#endif
#ifndef GNN_NW
#define GNN_NW 8
#endif
#ifndef GNN_UNR
#define GNN_UNR 2            // k-loop unroll of the GNN variant's tile products (EPN: fully unrolled, see tile_gemm_unr)
#endif
#ifndef EPN_DIR_UNROLL
#define EPN_DIR_UNROLL 1     // 2: also unroll the EPN variant's direction loop
#endif

template <typename R> struct BundleArgs {
    int n_bundles; const int2* bundle; int* work_counter;      // dynamic bundle queue (zeroed before the launch)
    const int* ustart; const int* pair_i; const int* pair_j; const unsigned char* near; const float* e;
    const unsigned char* perm_j;                              // per pair: rank of its j among the pairs of its tile
    const int* far_off; const unsigned short* far_list;
    // species-compressed far list: one weighted slot per (row, species of the column) -- used when the v rows of a
    // bundle depend on the species only (always true at step 0; at every step if the hidden state is species-wise constant)
    const int* far0_off; const unsigned short* far0_list; const unsigned char* far0_w; const int* rep; int dedup;
    const int* atom_sys; const int* sys_off; const int* npad;
    const R* u; const R* v;
    const R* Cw; const R* W2; const R* b2; const R* x32;      // x32 = b1 (GNN) or w3 (EPN)
    R* S; R* delta;
};

#ifdef EPNN_CPU_EMU
__device__ __forceinline__ void prefetch_l2(const void*) {}
#else
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
#endif

// Segmented add of one sorted tile into S.  Thread (pg, og) holds, for the tile positions pg*8 .. pg*8+7, the values
// val[s] (hidden columns og*4 .. og*4+3) and the target rows tgt[s]; targets ascend over the 32 positions and
// tgt < 0 marks the (trailing) invalid positions.  Runs of equal targets are summed in registers (in position
// order; a run that crosses threads is carried pg -> pg+1 through shuffles), and the thread that holds the LAST
// position of a run adds the total to S[row].  Every row is therefore written once per call: no two lanes touch the
// same address, the read-modify-writes are independent (their loads are hoisted), the order of every floating-point
// addition is fixed -> bitwise reproducible, no atomics.
template <typename R>
__device__ __forceinline__ void scatter_sorted(Vec4<R> (&val)[8], const int (&tgt)[8], R* __restrict__ S, int pg, int og) {
    const unsigned full = 0xffffffffu;
    const int prev_last = __shfl_up_sync(full, tgt[7], 8);
    bool b[8];                                   // a run starts at position s
    b[0] = pg == 0 || tgt[0] != prev_last;
#pragma unroll
    for (int s = 1; s < 8; ++s) b[s] = tgt[s] != tgt[s - 1];
    const int next_b0 = __shfl_down_sync(full, (int)b[0], 8);
    Vec4<R> run[8];                              // inclusive sums inside this thread (carry not yet applied)
    run[0] = val[0];
#pragma unroll
    for (int s = 1; s < 8; ++s) run[s] = b[s] ? val[s] : vadd(run[s - 1], val[s]);
    bool inhead[8];                              // position s still belongs to the run position 0 belongs to
    inhead[0] = true;
#pragma unroll
    for (int s = 1; s < 8; ++s) inhead[s] = inhead[s - 1] && !b[s];
    // carry across the four row groups (sequential by construction: pg = 1, 2, 3)
    Vec4<R> cin = vzero<R>();
    Vec4<R> cout = run[7];
#pragma unroll
    for (int r = 1; r < 4; ++r) {
        Vec4<R> up;
        up.x = __shfl_up_sync(full, cout.x, 8); up.y = __shfl_up_sync(full, cout.y, 8);
        up.z = __shfl_up_sync(full, cout.z, 8); up.w = __shfl_up_sync(full, cout.w, 8);
        if (pg == r && !b[0]) {
            cin = up;
            if (inhead[7]) cout = vadd(up, run[7]);
        }
    }
    bool fl[8];                                  // position s is the last of its run
#pragma unroll
    for (int s = 0; s < 7; ++s) fl[s] = b[s + 1] && tgt[s] >= 0;
    fl[7] = (pg == 3 || next_b0) && tgt[7] >= 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {                // two batches of four: loads first, then add + store
        Vec4<R> cur[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int s = h * 4 + k;
            cur[k] = vzero<R>();
            if (fl[s]) cur[k] = ldv(S + tgt[s] * HID + og * 4);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int s = h * 4 + k;
            if (fl[s]) {
                Vec4<R> tot = run[s];
                if (inhead[s] && !b[0]) tot = vadd(cin, run[s]);
                stv(S + tgt[s] * HID + og * 4, vadd(cur[k], tot));
            }
        }
    }
}

template <typename R, bool EPN> struct BundleSmem {
    static constexpr int EK = EKof<R>::v;
    static constexpr int W_ELEMS = EK * HID + HID * HID + 2 * HID;                                  // shared weights
    static constexpr int PW = BUNDLE_ATOMS * 64 + (EPN ? 0 : BUNDLE_ATOMS * HID + BUNDLE_ATOMS) + 32 * (EK > HID ? EK : HID);   // per warp (tile buffer: e rows, then z rows)
    static constexpr int PI = 128;                                                                  // ints per warp
    static size_t bytes(int nw) { return sizeof(R) * (W_ELEMS + (size_t)nw * PW) + sizeof(int) * nw * PI; }
};

template <typename R, int NW, bool EPN>
__global__ void __launch_bounds__(NW * 32, 1) bundle_kernel(const BundleArgs<R> a) {
#ifdef EPNN_CPU_EMU
    unsigned char* smem_raw = reinterpret_cast<unsigned char*>(emu_smem);
#else
    extern __shared__ __align__(32) unsigned char smem_raw[];
#endif
    using L = BundleSmem<R, EPN>;
    constexpr int EK = L::EK;
    R* sC = reinterpret_cast<R*>(smem_raw);          // [EK][32]
    R* sW2 = sC + EK * HID;                          // [32][32]
    R* sb2 = sW2 + HID * HID;                        // [32]
    R* sx = sb2 + HID;                               // [32]  b1 (GNN) / w3 (EPN)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    R* uv = sx + HID + warp * L::PW;                 // [BUNDLE_ATOMS][64]
    R* S = uv + BUNDLE_ATOMS * 64;                   // [BUNDLE_ATOMS][32]      (GNN only)
    R* padw = S + BUNDLE_ATOMS * HID;                // [BUNDLE_ATOMS]          (GNN only)
    R* eb = uv + BUNDLE_ATOMS * 64 + (EPN ? 0 : BUNDLE_ATOMS * HID + BUNDLE_ATOMS);   // [32][EK] descriptor tile, then [32][32] z tile
    int* sl_i = reinterpret_cast<int*>(sx + HID + NW * L::PW) + warp * L::PI;
    int* sl_c = sl_i + 32;                           // packed slot code: local i | local j << 8 (0xFF = pad pseudo-atom), -1 = empty
    int* sl_p = sl_i + 64;                           // near: position of the slot when the tile is sorted by j
    int* sl_t = sl_i + 96;                           // near: j targets in that sorted order

    for (int t = threadIdx.x; t < EK * HID; t += NW * 32) sC[t] = a.Cw[t];
    for (int t = threadIdx.x; t < HID * HID; t += NW * 32) sW2[t] = a.W2[t];
    if (threadIdx.x < HID) { sb2[threadIdx.x] = a.b2[threadIdx.x]; sx[threadIdx.x] = a.x32[threadIdx.x]; }
    __syncthreads();

    const int pg = lane >> 3, og = lane & 7;
    const Vec4<R> b2v = ldv(sb2 + og * 4);
    const Vec4<R> xv = ldv(sx + og * 4);             // b1 columns (GNN) / w3 columns (EPN)
    R* zt = eb;

    // Bundles differ in cost (7 .. 48 atoms), so the warps pull them from a queue instead of striding; every warp holds
    // the index of its NEXT bundle already, to prefetch that bundle's u / v rows.  Which warp handles a bundle has no
    // influence on the result (each bundle is self-contained and its arithmetic order is fixed).
    auto grab = [&]() {
        int t = 0;
        if (lane == 0) t = atomicAdd(a.work_counter, 1);
        return __shfl_sync(0xffffffffu, t, 0);
    };
    int b = grab();
    int b_next = grab();
    for (; b < a.n_bundles; b = b_next, b_next = grab()) {
        const int2 bd = a.bundle[b];
        const int atom0 = bd.x, nat = bd.y;
        const int p0 = a.ustart[atom0], p1 = a.ustart[atom0 + nat];
        const int ntile = (p1 - p0 + 31) >> 5;
        // ---- software prefetch (registers) of tile 0: indices + e rows
        int n_i = 0, n_j = 0;                        // raw (global) indices of the prefetched tile; rebased when consumed
        unsigned char n_x = 0;                       // near flag (EPN) / j-order position (GNN)
        float4 er[EK / 4];
        auto fetch_tile = [&](int tb) {
            const int rows = min(32, p1 - tb);
            if (lane < rows) {
                n_i = a.pair_i[tb + lane]; n_j = a.pair_j[tb + lane];
                n_x = EPN ? a.near[tb + lane] : a.perm_j[tb + lane];
            }
            const float4* esrc = reinterpret_cast<const float4*>(a.e + (int64_t)tb * EK);
#pragma unroll
            for (int m = 0; m < EK / 4; ++m) {
                const int f = lane + 32 * m;
                er[m] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (f / (EK / 4) < rows) er[m] = __ldg(esrc + f);
            }
        };
        if (ntile > 0) fetch_tile(p0);
        if (b_next < a.n_bundles) {                  // next bundle's u / v rows -> L2
            const int2 nd = a.bundle[b_next];
            const int nbytes = nd.y * HID * (int)sizeof(R);
            for (int o = lane * 128; o < nbytes; o += 32 * 128) {
                prefetch_l2(reinterpret_cast<const char*>(a.u + (int64_t)nd.x * HID) + o);
                prefetch_l2(reinterpret_cast<const char*>(a.v + (int64_t)nd.x * HID) + o);
            }
        }
        // ---- stage u | v (and zero S, pad weights)
        for (int f = lane; f < nat * 16; f += 32) {
            const int row = f >> 4, ch = f & 15;
            const R* src = (ch < 8 ? a.u : a.v) + (int64_t)(atom0 + row) * HID + (ch & 7) * 4;
            stv(uv + row * 64 + ch * 4, ldv(src));
        }
        if (!EPN) {
            for (int f = lane; f < nat * (HID / 4); f += 32) stv(S + f * 4, vzero<R>());
            for (int r = lane; r < nat; r += 32) {
                const int sys = a.atom_sys[atom0 + r];
                padw[r] = (R)(a.npad[sys] - (a.sys_off[sys + 1] - a.sys_off[sys]));
            }
        }
        __syncwarp();

        // ---------------------------------------------------------------- near tiles (unordered e != 0 pairs)
        for (int t = 0; t < ntile; ++t) {
            const int tb = p0 + t * 32;
            const bool ok = lane < min(32, p1 - tb);
            const R nearf = ok ? (R)n_x : R(0);
            {
                const int li = ok ? n_i - atom0 : -1, lj = ok ? n_j - atom0 : -1;
                const int lp = ok ? (int)n_x : lane;
                sl_c[lane] = ok ? (li | (lj << 8)) : -1;
                if (!EPN) { sl_i[lane] = li; sl_p[lane] = lp; sl_t[lp] = lj; }
            }
#pragma unroll
            for (int m = 0; m < EK / 4; ++m) {                          // prefetched e rows -> swizzled tile
                const int f = lane + 32 * m;
                const int sl = f / (EK / 4), ch = f - sl * (EK / 4);
                stv(eb + tile_off(sl, ch, EK), cvt4<R>(er[m]));
            }
            if (t + 1 < ntile) fetch_tile(tb + 32);                     // next tile's loads fly during this tile's math
            __syncwarp();
            R ce[8][4];
            zero_acc(ce);
            tile_gemm_unr<R, EK, HID, EPN ? 8 : GNN_UNR>(eb, sC, og * 4, ce, pg);
            __syncwarp();                                              // e tile consumed; eb becomes the z tile

            R part[8];
            R acc[8][4];
            int code[8];                                               // this thread's 8 slots: i | j << 8, or -1
            {
                const int4 c0 = *reinterpret_cast<const int4*>(sl_c + pg * 8);
                const int4 c1 = *reinterpret_cast<const int4*>(sl_c + pg * 8 + 4);
                code[0] = c0.x; code[1] = c0.y; code[2] = c0.z; code[3] = c0.w;
                code[4] = c1.x; code[5] = c1.y; code[6] = c1.z; code[7] = c1.w;
            }
            constexpr int DIR_UNR = EPN ? EPN_DIR_UNROLL : 1;
#pragma unroll DIR_UNR
            for (int dir = 0; dir < 2; ++dir) {
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const int slot = pg * 8 + s;
                    int ii = code[s] & 0xFF, jj = (code[s] >> 8) & 0xFF;
                    if (dir) { const int tmp = ii; ii = jj; jj = tmp; }
                    Vec4<R> z = vzero<R>();
                    if (code[s] >= 0) {
                        const Vec4<R> ui = ldv(uv + ii * 64 + og * 4);
                        const Vec4<R> vj = ldv(uv + jj * 64 + HID + og * 4);
                        Vec4<R> cv; cv.x = ce[s][0]; cv.y = ce[s][1]; cv.z = ce[s][2]; cv.w = ce[s][3];
                        z = vrelu(vadd(vadd(cv, ui), vj));
                    }
                    stv(zt + tile_off(slot, og, HID), z);
                }
                __syncwarp();
                zero_acc(acc);
                tile_gemm_unr<R, HID, HID, EPN ? 8 : GNN_UNR>(zt, sW2, og * 4, acc, pg);
                __syncwarp();
                if (EPN) {
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        R f = relu(acc[s][0] + b2v.x) * xv.x;
                        f = fma(relu(acc[s][1] + b2v.y), xv.y, f);
                        f = fma(relu(acc[s][2] + b2v.z), xv.z, f);
                        f = fma(relu(acc[s][3] + b2v.w), xv.w, f);
                        part[s] = dir ? part[s] - f : f;      // (dir is a run-time value now: the dir loop is not unrolled)
                    }
                } else {
                    Vec4<R> val[8];
                    int tg[8];
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        Vec4<R> av; av.x = acc[s][0]; av.y = acc[s][1]; av.z = acc[s][2]; av.w = acc[s][3];
                        val[s] = vrelu(vadd(av, b2v));
                    }
                    if (dir == 0) {                                    // targets i: the pair list is sorted by i already
#pragma unroll
                        for (int s = 0; s < 8; ++s) tg[s] = sl_i[pg * 8 + s];
                    } else {                                           // targets j: permute the tile into j order through smem
#pragma unroll
                        for (int s = 0; s < 8; ++s) stv(zt + tile_off(sl_p[pg * 8 + s], og, HID), val[s]);
                        __syncwarp();
#pragma unroll
                        for (int s = 0; s < 8; ++s) { val[s] = ldv(zt + tile_off(pg * 8 + s, og, HID)); tg[s] = sl_t[pg * 8 + s]; }
                    }
                    scatter_sorted<R>(val, tg, S, pg, og);
                    __syncwarp();
                }
            }
            if (EPN) {
                // reduce-scatter part[0..7] over the 8 og lanes: lane og ends with the total of slot pg*8 + og = lane
                R r4[4], r2[2], r1;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const R send = (og & 4) ? part[q] : part[q + 4];
                    const R keep = (og & 4) ? part[q + 4] : part[q];
                    r4[q] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                }
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const R send = (og & 2) ? r4[q] : r4[q + 2];
                    const R keep = (og & 2) ? r4[q + 2] : r4[q];
                    r2[q] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
                }
                {
                    const R send = (og & 1) ? r2[0] : r2[1];
                    const R keep = (og & 1) ? r2[1] : r2[0];
                    r1 = keep + __shfl_xor_sync(0xffffffffu, send, 1);
                }
                if (ok) a.delta[tb + lane] = R(0.5) * r1 * nearf;      // charge_gn.py:116
            }
            __syncwarp();
        }

        if (!EPN) {
            // ------------------------------------------------------------ far tiles (ordered pairs with e == 0, pad pseudo-pairs)
            // Exact de-duplication: a far message depends on the column j only through v_j.  If every atom of the bundle
            // has the same v row (bit for bit) as the first atom of its system with the same species, the far columns of a
            // row collapse to one weighted slot per species: sum_j m(u_i, v_j) = sum_s count_is * m(u_i, v_rep(s)).
            bool use0 = a.dedup != 0;
            if (use0) {
                bool same = true;
                for (int r = lane; r < nat; r += 32) {
                    const int rp = a.rep[atom0 + r] - atom0;
                    if (rp != r) {
#pragma unroll
                        for (int c = 0; c < HID / 4; ++c) {
                            const Vec4<R> x = ldv(uv + r * 64 + HID + c * 4), y = ldv(uv + rp * 64 + HID + c * 4);
                            same = same && x.x == y.x && x.y == y.y && x.z == y.z && x.w == y.w;
                        }
                    }
                }
                use0 = __all_sync(0xffffffffu, same);
            }
            const unsigned short* flist = use0 ? a.far0_list : a.far_list;
            const int f0 = use0 ? a.far0_off[atom0] : a.far_off[atom0], f1 = use0 ? a.far0_off[atom0 + nat] : a.far_off[atom0 + nat];
            const int nft = (f1 - f0 + 31) >> 5;
            R acc[8][4];
            int n_code = (f0 + lane < f1) ? (int)flist[f0 + lane] : -1;
            int n_cnt = (use0 && f0 + lane < f1) ? (int)a.far0_w[f0 + lane] : 1;
            for (int t = 0; t < nft; ++t) {
                int my_code;
                R my_w;
                {
                    int li = -1, lj = 0;
                    R wv = R(1);
                    if (n_code >= 0) {
                        li = n_code >> 8; lj = n_code & 0xFF;
                        wv = lj == 0xFF ? padw[li] : (R)n_cnt;        // pad pseudo-pair: npad - n; compressed slot: column count
                    }
                    my_code = li < 0 ? -1 : (li | (lj << 8)); my_w = wv;
                }
                {
                    const int k = f0 + (t + 1) * 32 + lane;
                    n_code = k < f1 ? (int)flist[k] : -1;
                    n_cnt = (use0 && k < f1) ? (int)a.far0_w[k] : 1;
                }
                int tg[8];
                R wcode[8];
#pragma unroll
                for (int s = 0; s < 8; ++s) {                           // this thread's 8 slots, straight from the owner lanes
                    tg[s] = __shfl_sync(0xffffffffu, my_code, pg * 8 + s);
                    wcode[s] = __shfl_sync(0xffffffffu, my_w, pg * 8 + s);
                }
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const int slot = pg * 8 + s;
                    const int ii = tg[s] & 0xFF, jj = (tg[s] >> 8) & 0xFF;
                    const bool live = tg[s] >= 0;
                    tg[s] = live ? ii : -1;
                    Vec4<R> z = vzero<R>();
                    if (live) {
                        const Vec4<R> ui = ldv(uv + ii * 64 + og * 4);
                        const Vec4<R> vj = jj == 0xFF ? xv : ldv(uv + jj * 64 + HID + og * 4);
                        z = vrelu(vadd(ui, vj));
                    }
                    stv(zt + tile_off(slot, og, HID), z);
                }
                __syncwarp();
                zero_acc(acc);
                tile_gemm_unr<R, HID, HID, GNN_UNR>(zt, sW2, og * 4, acc, pg);
                Vec4<R> val[8];
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    Vec4<R> av; av.x = acc[s][0]; av.y = acc[s][1]; av.z = acc[s][2]; av.w = acc[s][3];
                    val[s] = vscale(vrelu(vadd(av, b2v)), wcode[s]);
                }
                scatter_sorted<R>(val, tg, S, pg, og);
                __syncwarp();
            }
            // ---- S -> global (plane 0 of the partial-sum planes the per-atom kernel reads)
            for (int f = lane; f < nat * (HID / 4); f += 32) stv(a.S + (int64_t)atom0 * HID + f * 4, ldv(S + f * 4));
        }
        __syncwarp();
    }
}

#ifndef EPNN_CPU_EMU
template <typename R, bool EPN>
static cudaError_t launch_bundle(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* nl) {
    if (w.n_bundles == 0) return cudaSuccess;
    constexpr int NW = sizeof(R) == 4 ? (EPN ? EPN_NW : GNN_NW) : 4;   // the EPN variant has no S accumulators: more warps fit
    BundleArgs<R> ba;
    ba.n_bundles = w.n_bundles; ba.bundle = w.bundle; ba.work_counter = w.work_counter;
    cudaError_t e0 = cudaMemsetAsync(w.work_counter, 0, sizeof(int), st);
    if (e0 != cudaSuccess) return e0;
    ba.ustart = w.ustart; ba.pair_i = w.pair_i; ba.pair_j = w.pair_j; ba.near = w.near; ba.e = w.e;
    ba.perm_j = w.perm_j;
    ba.far_off = w.far_off; ba.far_list = w.far_list;
    ba.far0_off = w.far0_off; ba.far0_list = w.far0_list; ba.far0_w = w.far0_w; ba.rep = w.rep; ba.dedup = w.dedup_far;
    ba.atom_sys = w.atom_sys; ba.sys_off = w.sys_off; ba.npad = w.npad;
    ba.u = (const R*)w.u; ba.v = (const R*)w.v;
    ba.Cw = sw.Cw; ba.W2 = sw.W2; ba.b2 = sw.b2; ba.x32 = EPN ? sw.W3 : sw.b1;
    ba.S = (R*)w.S; ba.delta = (R*)w.delta;
    const size_t smem = BundleSmem<R, EPN>::bytes(NW);
    cudaError_t e = cudaFuncSetAttribute(bundle_kernel<R, NW, EPN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int grid = div_up(w.n_bundles, NW);
    if (grid > w.sm_count) grid = w.sm_count;         // persistent: one CTA per SM, warps stride over the bundles
    bundle_kernel<R, NW, EPN><<<grid, NW * 32, smem, st>>>(ba);
    ++*nl;
    return cudaGetLastError();
}
#endif

#ifndef EPNN_CPU_EMU
template <typename R> cudaError_t launch_gnn_bundle(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* nl) {
    if constexpr (sizeof(R) == 4) {
        if (w.kc.gnn == GNN_RUN) return launch_gnn_bundle_run(w, sw, st, nl);      // row-run mapping (epnn_bundle_run.cu): FP32 default
        if (w.kc.gnn == GNN_CONST) return launch_gnn_bundle_const(w, sw, st, nl);  // pair-per-thread variant with transpose (epnn_bundle_const.cu)
    }
    return launch_bundle<R, false>(w, sw, st, nl);
}
template <typename R> cudaError_t launch_epn_bundle(const Workspace& w, const StepW<R>& sw, cudaStream_t st, int* nl) {
    if constexpr (sizeof(R) == 4) {
        if (w.kc.epn == EPN_MMA) return launch_epn_bundle_mma(w, sw, st, nl);       // optional 3xTF32 mma.sync variant (epnn_bundle_mma.cu)
        if (w.kc.epn == EPN_CONST) return launch_epn_bundle_const(w, sw, st, nl);   // pair-per-thread variant (epnn_bundle_const.cu): FP32 default
    }
    return launch_bundle<R, true>(w, sw, st, nl);
}
template cudaError_t launch_gnn_bundle<float>(const Workspace&, const StepW<float>&, cudaStream_t, int*);
template cudaError_t launch_gnn_bundle<double>(const Workspace&, const StepW<double>&, cudaStream_t, int*);
template cudaError_t launch_epn_bundle<float>(const Workspace&, const StepW<float>&, cudaStream_t, int*);
template cudaError_t launch_epn_bundle<double>(const Workspace&, const StepW<double>&, cudaStream_t, int*);
#endif

// ------------------------------------------------------------------------------------------------
// Far-pair lists, built once per chunk (geometry does not change between steps).
// far_cnt[i] = (n_sys - deg_i) + (npad > n)  for atoms of small systems (the self pair is not in the CSR, so it is
// counted by n - deg), 0 for atoms of large systems.  atom_b0[i] = first atom of i's bundle.
__global__ void far_count_kernel(int n_atoms, const int* __restrict__ atom_sys, const int* __restrict__ sys_off,
                                 const int* __restrict__ npad, const int* __restrict__ rowptr, int* __restrict__ far_cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const int s = atom_sys[i];
    const int n = sys_off[s + 1] - sys_off[s];
    far_cnt[i] = n <= SMALL_MAX ? (n - (rowptr[i + 1] - rowptr[i])) + (npad[s] > n ? 1 : 0) : 0;
}

__global__ void bundle_mark_kernel(int n_bundles, const int2* __restrict__ bundle, int* __restrict__ atom_b0,
                                   int* __restrict__ bundle_nat) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_bundles) return;
    const int2 bd = bundle[b];
    for (int k = 0; k < bd.y; ++k) atom_b0[bd.x + k] = bd.x;
    bundle_nat[bd.x] = bd.y;                     // atom count of the bundle, stored at its first atom
}

#ifndef EPNN_CPU_EMU
cudaError_t launch_far_count(const Workspace& w, int* far_cnt, int* atom_b0, cudaStream_t st, int* nl) {
    if (w.n_atoms == 0) return cudaSuccess;
    far_count_kernel<<<div_up(w.n_atoms, 256), 256, 0, st>>>(w.n_atoms, w.atom_sys, w.sys_off, w.npad, w.rowptr, far_cnt);
    ++*nl;
    if (w.n_bundles > 0) {
        bundle_mark_kernel<<<div_up(w.n_bundles, 128), 128, 0, st>>>(w.n_bundles, w.bundle, atom_b0, w.bundle_nat);
        ++*nl;
    }
    return cudaGetLastError();
}
#endif

// code = (i - b0) << 8 | (j - b0), j ascending over the complement of row i's CSR columns within its system
// (includes j == i); then 0xFF in the low byte for the weighted pad pseudo-pair.
__global__ void far_fill_kernel(int n_atoms, const int* __restrict__ atom_sys, const int* __restrict__ sys_off,
                                const int* __restrict__ npad, const int* __restrict__ rowptr, const int* __restrict__ col,
                                const int* __restrict__ atom_b0, const int* __restrict__ far_off,
                                unsigned short* __restrict__ far_list) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const int s = atom_sys[i];
    const int a0 = sys_off[s], a1 = sys_off[s + 1];
    if (a1 - a0 > SMALL_MAX) return;
    const int b0 = atom_b0[i];
    int w = far_off[i];
    int ptr = rowptr[i];
    const int r1 = rowptr[i + 1];
    const int hi = (i - b0) << 8;
    for (int j = a0; j < a1; ++j) {
        if (ptr < r1 && col[ptr] == j) { ++ptr; continue; }
        far_list[w++] = (unsigned short)(hi | (j - b0));
    }
    if (npad[s] > a1 - a0) far_list[w++] = (unsigned short)(hi | 0xFF);
}

// Species-compressed far list.  PASS 0: rep[i] (first atom of i's system with i's species) and the number of slots of
// row i = #{species s with at least one far column} + (pad ? 1 : 0).  PASS 1: the slots, species ascending:
// code = (i - b0) << 8 | (rep_s - b0), weight = number of far columns of species s (the self pair counts as far).
template <int PASS>
__global__ void far0_kernel(int n_atoms, const int* __restrict__ atom_sys, const int* __restrict__ sys_off,
                            const int* __restrict__ npad, const int* __restrict__ species, const int* __restrict__ rowptr,
                            const int* __restrict__ col, const int* __restrict__ atom_b0, int* __restrict__ rep,
                            int* __restrict__ cnt_out, const int* __restrict__ off, unsigned short* __restrict__ list,
                            unsigned char* __restrict__ wgt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const int s = atom_sys[i];
    const int a0 = sys_off[s], a1 = sys_off[s + 1];
    if (a1 - a0 > SMALL_MAX) { if (PASS == 0) { cnt_out[i] = 0; rep[i] = i; } return; }
    int cnt[MAX_SPECIES], first[MAX_SPECIES];
#pragma unroll
    for (int k = 0; k < MAX_SPECIES; ++k) { cnt[k] = 0; first[k] = -1; }
    for (int j = a0; j < a1; ++j) {
        const int sj = species[j] & (MAX_SPECIES - 1);
        ++cnt[sj];
        if (first[sj] < 0) first[sj] = j;
    }
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) --cnt[species[col[k]] & (MAX_SPECIES - 1)];
    const bool pad = npad[s] > a1 - a0;
    if (PASS == 0) {
        int n = pad ? 1 : 0;
#pragma unroll
        for (int k = 0; k < MAX_SPECIES; ++k) n += cnt[k] > 0;
        cnt_out[i] = n;
        rep[i] = first[species[i] & (MAX_SPECIES - 1)];
    } else {
        const int b0 = atom_b0[i];
        const int hi = (i - b0) << 8;
        int w = off[i];
#pragma unroll
        for (int k = 0; k < MAX_SPECIES; ++k)
            if (cnt[k] > 0) { list[w] = (unsigned short)(hi | (first[k] - b0)); wgt[w] = (unsigned char)cnt[k]; ++w; }
        if (pad) { list[w] = (unsigned short)(hi | 0xFF); wgt[w] = 0; }
    }
}

#ifndef EPNN_CPU_EMU
cudaError_t launch_far0_count(const Workspace& w, int* cnt, cudaStream_t st, int* nl) {
    if (w.n_atoms == 0) return cudaSuccess;
    far0_kernel<0><<<div_up(w.n_atoms, 128), 128, 0, st>>>(w.n_atoms, w.atom_sys, w.sys_off, w.npad, w.species, w.rowptr, w.col,
                                                           nullptr, w.rep, cnt, nullptr, nullptr, nullptr);
    ++*nl;
    return cudaGetLastError();
}
#endif

#ifndef EPNN_CPU_EMU
cudaError_t launch_far0_fill(const Workspace& w, const int* atom_b0, cudaStream_t st, int* nl) {
    if (w.n_atoms == 0 || w.n_bundles == 0) return cudaSuccess;
    far0_kernel<1><<<div_up(w.n_atoms, 128), 128, 0, st>>>(w.n_atoms, w.atom_sys, w.sys_off, w.npad, w.species, w.rowptr, w.col,
                                                           atom_b0, nullptr, nullptr, w.far0_off, w.far0_list, w.far0_w);
    ++*nl;
    return cudaGetLastError();
}
#endif

// perm_j[p] = position of pair p inside its 32-pair tile when the tile's valid pairs are ordered by (j, slot).  Tiles
// start at the first pair of the bundle (ustart[b0]); one thread per pair, the <= 31 other j's come from L1.
__global__ void tile_perm_kernel(int64_t P, const int* __restrict__ pair_i, const int* __restrict__ pair_j,
                                 const int* __restrict__ atom_sys, const int* __restrict__ sys_off,
                                 const int* __restrict__ atom_b0, const int* __restrict__ ustart, const int* __restrict__ bundle_nat,
                                 unsigned char* __restrict__ perm) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int i = pair_i[p];
    const int s = atom_sys[i];
    if (sys_off[s + 1] - sys_off[s] > SMALL_MAX) { perm[p] = 0; return; }
    const int b0 = atom_b0[i];
    const int p0 = ustart[b0], p1 = ustart[b0 + bundle_nat[b0]];
    const int slot = (int)(p - p0) & 31;
    const int tb = (int)p - slot;
    const int rows = min(32, p1 - tb);
    const int j = pair_j[p];
    int rank = 0;
    for (int k = 0; k < rows; ++k) {
        const int jk = pair_j[tb + k];
        rank += (jk < j) || (jk == j && k < slot);
    }
    perm[p] = (unsigned char)rank;
}

#ifndef EPNN_CPU_EMU
cudaError_t launch_tile_perm(const Workspace& w, const int* atom_b0, cudaStream_t st, int* nl) {
    if (w.n_atoms == 0 || w.n_bundles == 0) return cudaSuccess;
    if (w.P > 0 && w.kc.tile_perm) {
        tile_perm_kernel<<<div_up(w.P, 256), 256, 0, st>>>(w.P, w.pair_i, w.pair_j, w.atom_sys, w.sys_off, atom_b0,
                                                           w.ustart, w.bundle_nat, w.perm_j);
        ++*nl;
    }
    return cudaGetLastError();
}

cudaError_t launch_far_fill(const Workspace& w, const int* atom_b0, cudaStream_t st, int* nl) {
    if (w.n_atoms == 0 || w.n_bundles == 0) return cudaSuccess;
    cudaError_t e0 = launch_tile_perm(w, atom_b0, st, nl);
    if (e0 != cudaSuccess) return e0;
    far_fill_kernel<<<div_up(w.n_atoms, 128), 128, 0, st>>>(w.n_atoms, w.atom_sys, w.sys_off, w.npad, w.rowptr, w.col,
                                                            atom_b0, w.far_off, w.far_list);
    ++*nl;
    return cudaGetLastError();
}
#endif
