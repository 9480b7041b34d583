// CPU emulation driver for the neighbour-list and descriptor kernels, epnn_b200/csrc/epnn_neighbor.cu (test
// infrastructure; see cuda_emu.h).  Same launch sequence as build_lists (epnn_api.cu): prep -> cell build (systems with
// more than CELL_MIN atoms, cell bases of plan_cells, epnn_plan.h) -> count -> scans -> fill -> reverse edges -> descriptors.
// Build: g++ -O1 -std=c++17 -ffp-contract=off -shared -fPIC -pthread -DEPNN_CPU_EMU -o build/libemu_neighbor.so tools/emu/emu_neighbor.cpp
#define EPNN_CPU_EMU 1
#include "../../epnn_b200/csrc/epnn_neighbor.cu"

static void exclusive_scan(const int* in, int* out, int n) { int s = 0; for (int i = 0; i < n; ++i) { out[i] = s; s += in[i]; } out[n] = s; }

extern "C" int emu_neighbor_counts(const double* mu, const double* B, int n_atoms, int n_sys, const int* sys_off, const float* xyz,
                                   const float* Qsys, int* atom_sys, double* q0, int* deg, int* degU, int* rowptr, int* ustart,
                                   int* grid_ints /* 8 ints per system */, int* cell_start, int* cell_atoms, int n_cells_cap) {
    emu_set_rbf(mu, B);
    emu_launch_simple(div_up(n_atoms, 256), 256, [&] { prep_kernel(n_atoms, n_sys, sys_off, Qsys, atom_sys, q0); });
    std::vector<int> tab;
    const long long cells = plan_cells(sys_off, n_sys, tab);
    const int n_large = (int)tab.size() / 2;
    if (cells + 1 > n_cells_cap) return -1;
    CellGrid* grid = reinterpret_cast<CellGrid*>(grid_ints);
    if (n_large) {
        std::vector<int> cnt((size_t)cells + 2, 0);
        emu_launch_grid(n_large, 8, 0, [&] { cell_setup_kernel(n_large, tab.data(), tab.data() + n_large, sys_off, xyz, grid); });
        emu_launch_simple(div_up(n_atoms, 256), 256, [&] { cell_bin_kernel<0>(n_atoms, atom_sys, sys_off, xyz, grid, cnt.data(), nullptr, nullptr); });
        exclusive_scan(cnt.data(), cell_start, (int)cells);
        std::fill(cnt.begin(), cnt.end(), 0);
        emu_launch_simple(div_up(n_atoms, 256), 256, [&] { cell_bin_kernel<1>(n_atoms, atom_sys, sys_off, xyz, grid, cnt.data(), cell_start, cell_atoms); });
    }
    emu_launch_grid(div_up(n_atoms, 128), 4, 0, [&] {
        nbr_kernel<false>(n_atoms, atom_sys, sys_off, xyz, deg, degU, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, grid, cell_start, cell_atoms, nullptr, 0, n_atoms); });
    exclusive_scan(deg, rowptr, n_atoms);
    exclusive_scan(degU, ustart, n_atoms);
    return 0;
}

extern "C" int emu_neighbor_fill(int n_atoms, const int* atom_sys, const int* sys_off, const float* xyz, const int* degU,
                                 const int* rowptr, const int* ustart, const int* grid_ints, const int* cell_start, const int* cell_atoms,
                                 int* col, int* pid, int* pair_i, int* pair_j, double* pair_D, double* Dtmp,
                                 int ek, float* e, unsigned char* near) {
    const CellGrid* grid = reinterpret_cast<const CellGrid*>(grid_ints);
    emu_launch_grid(div_up(n_atoms, 128), 4, 0, [&] {
        nbr_kernel<true>(n_atoms, atom_sys, sys_off, xyz, nullptr, nullptr, rowptr, ustart, col, pair_i, pair_j, pair_D, grid, cell_start, cell_atoms, Dtmp, 0, n_atoms); });
    emu_launch_simple(div_up(n_atoms, 128), 128, [&] { nbr_rev_kernel(n_atoms, rowptr, ustart, degU, col, pid); });
    const int64_t P = ustart[n_atoms];
    if (P > 0) {
        if (ek == ED) emu_launch_grid(div_up(P, EDGE_PAIRS), EDGE_PAIRS / 32, 0, [&] { edge_desc_kernel<ED>(P, pair_D, e, near, nullptr, nullptr, nullptr, nullptr); });
        else          emu_launch_grid(div_up(P, EDGE_PAIRS), EDGE_PAIRS / 32, 0, [&] { edge_desc_kernel<EDR>(P, pair_D, e, near, nullptr, nullptr, nullptr, nullptr); });
    }
    return 0;
}
