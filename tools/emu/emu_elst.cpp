// CPU emulation driver for epnn_b200/csrc/epnn_elst.cu, the electrostatics kernels (test infrastructure; see cuda_emu.h).
// Build: g++ -O1 -std=c++17 -ffp-contract=off -shared -fPIC -pthread -DEPNN_CPU_EMU -o build/libemu_elst.so tools/emu/emu_elst.cpp
#define EPNN_CPU_EMU 1
#include "../../epnn_b200/csrc/epnn_elst.cu"

extern "C" int emu_elst_parts(int n, long long target_ctas) { return elst_parts(n, target_ctas); }

// One call of the library's chunk: the plan epnn_api.cu builds, then the three kernels in launch order.  target_ctas
// stands for ELST_CTAS_PER_SM * SM count, so that small systems reach every source split.  Outputs may be NULL.
extern "C" int emu_elst(int n_sys, const int* off, const float* xyz, const double* q, const int* frag, long long target_ctas,
                        double* energy, double* dipole, double* phi) {
    std::vector<ElstItem> items;
    std::vector<ElstSys> sys;
    const long long plen = elst_plan(off, n_sys, target_ctas, items, sys);
    std::vector<double> partial((size_t)plen + 1, std::nan(""));
    ElstArgs a;
    a.n_sys = n_sys; a.base = off[0]; a.off = off;
    a.xyz = xyz; a.q = q; a.frag = frag;
    a.energy = energy; a.dipole = dipole; a.phi = phi;
    a.items = items.data(); a.sys = sys.data(); a.partial = partial.data();
    emu_launch_grid((n_sys + ELST_WARPS - 1) / ELST_WARPS, ELST_WARPS, 0, [&] { elst_small_kernel(a); });
    if (!items.empty()) emu_launch_grid((int)items.size(), ELST_TILE / 32, 0, [&] { elst_pair_kernel(a); });
    if (!sys.empty()) emu_launch_grid((int)sys.size(), ELST_RED / 32, 0, [&] { elst_reduce_kernel(a); });
    return (int)items.size();
}
