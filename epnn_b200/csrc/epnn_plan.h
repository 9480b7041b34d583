// Host-side planning of the inference path, shared by epnn_api.cu and the CPU warp emulation (tools/emu): the chunks of a
// call, the row slices of a sharded call, the kernel choice of a call and the plan of one chunk.  Pure functions of host data.
#pragma once
#include <limits.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

#ifdef EPNN_CPU_EMU
#include "../../tools/emu/cuda_emu.h"      // int2
#else
#include <vector_types.h>
#endif
#include "epnn_consts.h"

// Splits [0, n_sys) into chunks of at most chunk_atoms atoms (a single larger system gets its own chunk).
static inline void plan_chunks(const int32_t* off, int64_t n_sys, int64_t chunk_atoms, std::vector<int64_t>& bounds) {
    bounds.clear();
    bounds.push_back(0);
    int64_t s = 0;
    while (s < n_sys) {
        int64_t e = s + 1;
        while (e < n_sys && (int64_t)off[e + 1] - off[s] <= chunk_atoms) ++e;
        bounds.push_back(e);
        s = e;
    }
}

// Equal slices of the atom index space of a batch: rank r owns rows [r * slice, (r + 1) * slice) clipped to n;
// slice = ceil(n / world) rounded up to 32 rows (all-gathers need equal counts; 32 = the row block of the far kernels).
static inline int64_t shard_slice_rows(int64_t n, int world) { const int64_t s = (n + world - 1) / world; return (s + 31) / 32 * 32; }

// ------------------------------------------------------------------------------------------------
// Kernel choice of a call.  The FP32 pair kernels run at precision 32 and 48; FP64 calls run the warp-tile kernels.
enum GnnBundleKernel { GNN_TILE, GNN_CONST, GNN_RUN };      // bundle_kernel (epnn_bundle.cu), bundle_const (epnn_bundle_const.cu), bundle_run (epnn_bundle_run.cu)
enum EpnBundleKernel { EPN_TILE, EPN_CONST, EPN_MMA };      // bundle_kernel, bundle_const, bundle_epn_mma (epnn_bundle_mma.cu)
enum AtomKernel { ATOM_K_SIMT, ATOM_K_MMA, ATOM_K_CONST };  // atom_kernel (epnn_atom.cu); atom_mma (epnn_atom_mma.cu) for the launches with a
                                                            // dense layer, atom_kernel for the others; atom_const (epnn_atom_const.cu)
enum FarKernel { FAR_SIMT, FAR_TC, FAR_TC2, FAR_CONST };    // far part of the systems above SMALL_MAX atoms: the planes of gnn_pair_kernel
                                                            // (epnn_gnn.cu), tcgen05 (epnn_gnn_tc.cu, epnn_gnn_tc2.cu), gnn_far_const (epnn_gnn_far_const.cu)

// The options of epnn_set_option that pick kernels (besides "precision" and "atom_tensor", which the auto precision probe sets per call).
struct KernelOptions {
    int pair_const = 2;          // "pair_const"
    int pair_tensor = 0;         // "pair_tensor"
    int far_tensor = 2;          // "gnn_far_tensor": 0 off, 1 on, 2 auto
    int far_tensor_min = 16384;  // "gnn_far_tensor_min"
    int far_tensor_impl = 1;     // "gnn_far_tensor_impl"
};

struct KernelChoice {
    int precision;               // 32, 48 (FP32 pair kernels around an FP64 per-atom kernel) or 64
    GnnBundleKernel gnn;         // GNN bundle kernel (systems of at most SMALL_MAX atoms)
    EpnBundleKernel epn;         // EPN bundle kernel
    AtomKernel atom;             // FP32 per-atom kernel of the launches over all atoms (precision 48 / 64: atom_kernel<double, IO>)
    AtomKernel atom_scoped;      // ... of the launches restricted to a rank's rows (sharded calls): atom_const has no such scope
    FarKernel far;               // far part of a chunk whose largest system has fewer than far_tc_min atoms
    FarKernel far_tc;            // ... and of one whose largest system has at least far_tc_min atoms
    int far_tc_min;
    bool csr_rowl;               // the row-run GNN bundle kernel reads rowl (local row of every CSR entry)
    bool tile_perm;              // the warp-tile GNN bundle kernel reads perm_j.  It is also built for GNN_CONST, whose kernels do
                                 // not read it: a later removal (it is one launch of epnn_stats.n_launches)
};

static inline KernelChoice resolve_kernels(int precision, int atom_tensor, const KernelOptions& o) {
    KernelChoice k;
    k.precision = precision;
    const bool fp32 = precision != 64;
    const int pc = fp32 ? o.pair_const : 0;
    k.gnn = pc == 2 ? GNN_RUN : pc == 1 ? GNN_CONST : GNN_TILE;
    k.epn = fp32 && o.pair_tensor ? EPN_MMA : pc ? EPN_CONST : EPN_TILE;
    k.atom_scoped = precision == 32 && atom_tensor ? ATOM_K_MMA : ATOM_K_SIMT;
    k.atom = precision == 32 && pc == 1 ? ATOM_K_CONST : k.atom_scoped;
    k.far = pc ? FAR_CONST : FAR_SIMT;
    const bool tc = fp32 && o.far_tensor != 0;
    k.far_tc = !tc ? k.far : o.far_tensor_impl == 2 ? FAR_TC2 : FAR_TC;
    k.far_tc_min = !tc ? INT_MAX : o.far_tensor == 1 ? 0 : o.far_tensor_min;
    k.csr_rowl = k.gnn == GNN_RUN;
    k.tile_perm = k.gnn != GNN_RUN;
    return k;
}

// ------------------------------------------------------------------------------------------------
// Cell lists of the systems of more than CELL_MIN atoms: a budget of 4 n + 64 cells each, so the first cell of every
// system is known on the host.  off: n_sys + 1 offsets.  tab = [the systems | their first cells]; returns the cell count.
static inline long long plan_cells(const int32_t* off, int n_sys, std::vector<int>& tab) {
    tab.clear();
    std::vector<int> base;
    long long cells = 0;
    for (int s = 0; s < n_sys; ++s) {
        const int n = off[s + 1] - off[s];
        if (n > CELL_MIN) { tab.push_back(s); base.push_back((int)cells); cells += 4ll * n + 64; }
    }
    tab.insert(tab.end(), base.begin(), base.end());
    return cells;
}

// Everything about one chunk that follows from its offsets, the SM count, the shard rank / world and the kernel choice.
// Atom indices are chunk-local.
struct ChunkPlan {
    std::vector<int2> bundles;   // (first atom, atoms): greedy runs of consecutive systems of at most SMALL_MAX atoms, <= BUNDLE_ATOMS atoms
    std::vector<int> cell_tab;   // plan_cells
    int n_large;                 // systems with a cell list
    long long n_cells, big_atoms;
    bool has_large;              // a system of more than SMALL_MAX atoms
    int max_n, n_rg_large;       // largest system; 4-row groups of the systems above SMALL_MAX atoms
    bool sharded;                // world > 1 and has_large: the rows of the large systems are split over the ranks
    int64_t slice, rows_pad;     // rows per rank; rows of an exchanged array (world slices)
    int row_lo, row_hi;          // rows of this rank: epnn_shard_slice (unsharded: all)
    int rg_begin, rg_end;        // 4-row groups (numbered over the large systems in order) that overlap [row_lo, row_hi)
    std::vector<int2> rowblk;    // (first atom, system) of every 32-row block of the large systems
    int blk_begin, blk_end;      // the row blocks that overlap [row_lo, row_hi)
    FarKernel far;               // far part of the large systems
    int nsplit;                  // partial-sum planes of S
};

// off: the chunk's n_sys + 1 offsets (off[0] = its first atom).  Returns false when the cell grid would reach 2^31 cells.
static inline bool plan_chunk(const int32_t* off, int n_sys, int sm_count, int rank, int world, const KernelChoice& k, ChunkPlan& p) {
    const int base = off[0], n_atoms = off[n_sys] - off[0];
    p.bundles.clear();
    p.has_large = false;
    p.max_n = p.n_rg_large = 0;
    int cur0 = -1, cur_n = 0;
    for (int s = 0; s < n_sys; ++s) {
        const int a0 = off[s] - base, n = off[s + 1] - off[s];
        p.max_n = std::max(p.max_n, n);
        if (n > SMALL_MAX) {
            if (cur_n) { p.bundles.push_back(int2{cur0, cur_n}); cur_n = 0; }
            p.has_large = true;
            p.n_rg_large += (n + 3) >> 2;
            continue;
        }
        if (cur_n && cur_n + n > BUNDLE_ATOMS) { p.bundles.push_back(int2{cur0, cur_n}); cur_n = 0; }
        if (!cur_n) cur0 = a0;
        cur_n += n;
    }
    if (cur_n) p.bundles.push_back(int2{cur0, cur_n});

    p.n_cells = plan_cells(off, n_sys, p.cell_tab);
    if (p.n_cells + 1 >= (1ll << 31)) return false;
    p.n_large = (int)p.cell_tab.size() / 2;
    p.big_atoms = 0;
    for (int j = 0; j < p.n_large; ++j) p.big_atoms += off[p.cell_tab[j] + 1] - off[p.cell_tab[j]];

    p.sharded = world > 1 && p.has_large;
    if (!p.sharded) { rank = 0; world = 1; }
    p.slice = p.sharded ? shard_slice_rows(n_atoms, world) : n_atoms;
    p.rows_pad = p.slice * world;
    p.row_lo = (int)std::min<int64_t>(p.slice * rank, n_atoms);
    p.row_hi = (int)std::min<int64_t>(p.slice * (rank + 1), n_atoms);
    int rg_b = -1, rg_e = 0, g = 0;
    p.rowblk.clear();
    for (int s = 0; s < n_sys; ++s) {
        const int a0 = off[s] - base, n = off[s + 1] - off[s];
        if (n <= SMALL_MAX) continue;
        for (int i = 0; i < n; i += 4, ++g)
            if (a0 + i + 3 >= p.row_lo && a0 + i < p.row_hi) { if (rg_b < 0) rg_b = g; rg_e = g + 1; }
        for (int i = 0; i < n; i += 32) p.rowblk.push_back(int2{a0 + i, s});
    }
    p.rg_begin = rg_b < 0 ? 0 : rg_b; p.rg_end = rg_b < 0 ? 0 : rg_e;
    int bb = -1, be = 0;
    for (int b = 0; b < (int)p.rowblk.size(); ++b)
        if (p.rowblk[b].x + 31 >= p.row_lo && p.rowblk[b].x < p.row_hi) { if (bb < 0) bb = b; be = b + 1; }
    p.blk_begin = bb < 0 ? 0 : bb; p.blk_end = bb < 0 ? 0 : be;

    // partial-sum planes: the tensor-core and row-per-thread far kernels own planes [0, nsplit - 1), gnn_pair_kernel (near
    // pairs, pad pair, species slots) the last one; the SIMT planes split the columns of every row group nsplit ways
    auto planes = [](int64_t units_wanted, int64_t units, int cap) { return (int)std::min<int64_t>(std::max<int64_t>((units_wanted + units - 1) / units, 1), cap); };
    p.far = FAR_SIMT;
    p.nsplit = 1;
    if (p.n_rg_large > 0) {
        p.far = p.max_n >= k.far_tc_min ? k.far_tc : k.far;
        if (p.far == FAR_TC || p.far == FAR_TC2) p.nsplit = planes((int64_t)sm_count * 8, p.n_rg_large, 15) + 1;
        else if (p.far == FAR_CONST) p.nsplit = planes((int64_t)sm_count * 32, (int64_t)p.rowblk.size(), 15) + 1;
        else p.nsplit = planes((int64_t)sm_count * 64, p.n_rg_large, 32);
    }
    return true;
}
