// CPU emulation driver for epnn_b200/csrc/epnn_bundle_run.cu, the row-run GNN bundle kernel (test infrastructure; see cuda_emu.h).
// Build: g++ -O1 -std=c++17 -ffp-contract=off -shared -fPIC -pthread -DEPNN_CPU_EMU -o build/libemu_bundle_run.so tools/emu/emu_bundle_run.cpp
#define EPNN_CPU_EMU 1
#include "../../epnn_b200/csrc/epnn_bundle_run.cu"

// weights: Cw[16*32] | W2[32*32] | b2[32] | b1[32];  slots (may be NULL): [0] near, [1] far slots the kernel walked
extern "C" int emu_bundle_run(int n_warps, const float* weights,
                              int n_bundles, const int* bundle_xy, int* work_counter,
                              const int* rowptr, const int* col, const int* pid, const unsigned char* rowl, const float* e, const int* ustart,
                              const int* far_off, const unsigned short* far_list,
                              const int* far0_off, const unsigned short* far0_list, const unsigned char* far0_w, const int* rep, int dedup,
                              const int* atom_sys, const int* sys_off, const int* npad,
                              const float* u, const float* v, float* S, unsigned long long* slots) {
    if (n_warps < 1 || n_warps > RUN_NW) return -1;
    RunW W;
    memcpy(W.W2, weights + EDR * HID, sizeof(W.W2));
    RunArgs a;
    a.n_bundles = n_bundles; a.bundle = reinterpret_cast<const int2*>(bundle_xy); a.work_counter = work_counter;
    a.rowptr = rowptr; a.col = col; a.pid = pid; a.rowl = rowl; a.e = e; a.ustart = ustart;
    a.far_off = far_off; a.far_list = far_list;
    a.far0_off = far0_off; a.far0_list = far0_list; a.far0_w = far0_w; a.rep = rep; a.dedup = dedup;
    a.atom_sys = atom_sys; a.sys_off = sys_off; a.npad = npad;
    a.u = u; a.v = v; a.S = S;
    a.Cw = weights; a.b2 = weights + EDR * HID + HID * HID; a.b1 = weights + EDR * HID + HID * HID + HID;
    a.slot_counter = slots;
    *work_counter = 0;
    emu_launch_cta(n_warps, RunSmem::bytes() / sizeof(float), [&] { bundle_run_kernel(W, &a); });
    return 0;
}
