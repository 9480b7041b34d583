// C entry points over the host-side planning of the inference path, epnn_b200/csrc/epnn_plan.h (test infrastructure:
// tests/test_emu_plan.py).  Nothing here plans anything of its own.
// Build: g++ -O1 -std=c++17 -shared -fPIC -DEPNN_CPU_EMU -o build/libemu_plan.so tools/emu/emu_plan.cpp
#define EPNN_CPU_EMU 1
#include "../../epnn_b200/csrc/epnn_plan.h"

static KernelOptions options(const int* o) {      // pair_const, pair_tensor, gnn_far_tensor, gnn_far_tensor_min, gnn_far_tensor_impl
    KernelOptions k;
    k.pair_const = o[0]; k.pair_tensor = o[1]; k.far_tensor = o[2]; k.far_tensor_min = o[3]; k.far_tensor_impl = o[4];
    return k;
}

// bounds: n_sys + 1 entries; returns the number written
extern "C" int emu_plan_chunks(const int32_t* off, int64_t n_sys, int64_t chunk_atoms, int64_t* bounds) {
    std::vector<int64_t> b;
    plan_chunks(off, n_sys, chunk_atoms, b);
    std::copy(b.begin(), b.end(), bounds);
    return (int)b.size();
}

// out: gnn, epn, atom, atom_scoped, far, far_tc, far_tc_min, csr_rowl, tile_perm
extern "C" void emu_resolve_kernels(int precision, int atom_tensor, const int* opts, int* out) {
    const KernelChoice k = resolve_kernels(precision, atom_tensor, options(opts));
    const int v[] = {k.gnn, k.epn, k.atom, k.atom_scoped, k.far, k.far_tc, k.far_tc_min, k.csr_rowl, k.tile_perm};
    std::copy(v, v + 9, out);
}

// bundles: 2 ints per bundle (room for n_sys); out: ok, n_bundles, has_large, max_n, n_rg_large, sharded, row_lo, row_hi,
// rg_begin, rg_end, n_rowblk, blk_begin, blk_end, far, nsplit, n_large, n_cells
extern "C" void emu_plan_chunk(const int32_t* off, int n_sys, int sm_count, int rank, int world, int precision, int atom_tensor,
                               const int* opts, int* bundles, int64_t* out) {
    ChunkPlan p{};
    const bool ok = plan_chunk(off, n_sys, sm_count, rank, world, resolve_kernels(precision, atom_tensor, options(opts)), p);
    for (size_t b = 0; b < p.bundles.size(); ++b) { bundles[2 * b] = p.bundles[b].x; bundles[2 * b + 1] = p.bundles[b].y; }
    const int64_t v[] = {ok, (int64_t)p.bundles.size(), p.has_large, p.max_n, p.n_rg_large, p.sharded, p.row_lo, p.row_hi,
                         p.rg_begin, p.rg_end, (int64_t)p.rowblk.size(), p.blk_begin, p.blk_end, p.far, p.nsplit, p.n_large, p.n_cells};
    std::copy(v, v + 17, out);
}
