// CPU emulation of a WHOLE charge inference through the product's own kernels (test infrastructure; see cuda_emu.h).
//
// Weights are packed / folded by the product's own host code (epnn_pack.h, the code epnn_create runs); the chunk plan and
// the kernel choice are the library's (epnn_plan.h: plan_chunk, resolve_kernels for precision 32 with the options of the
// variant, "atom_tensor" 0 and "gnn_far_tensor" 0); then the kernels of epnn_neighbor / epnn_bundle /
// epnn_bundle_const / epnn_bundle_run / epnn_bundle_mma / epnn_gnn / epnn_gnn_far_const / epnn_epn / epnn_atom /
// epnn_atom_const that the choice names run in the launch order of build_lists and run_layers (epnn_api.cu), FP32, one
// chunk.  The only code that is not the product's is this orchestration (without streams and workspaces), the host-side
// scans and the row groups of the large systems (sys_prep_kernel, rg_fill_kernel).
// tests/test_emu_infer.py compares the result with the oracle and with the reference's shipped predictions.
// Build: g++ -O1 -std=c++17 -ffp-contract=off -shared -fPIC -pthread -DEPNN_CPU_EMU -o build/libemu_infer.so tools/emu/emu_infer.cpp
#define EPNN_CPU_EMU 1
#include "../../epnn_b200/csrc/epnn_internal.cuh"
#include "../../epnn_b200/csrc/epnn_pack.h"
namespace k_nbr {
#include "../../epnn_b200/csrc/epnn_neighbor.cu"
}
namespace k_bundle {
#include "../../epnn_b200/csrc/epnn_bundle.cu"
}
namespace k_gnn {
#include "../../epnn_b200/csrc/epnn_gnn.cu"
}
namespace k_epn {
#include "../../epnn_b200/csrc/epnn_epn.cu"
}
namespace k_atom {
#include "../../epnn_b200/csrc/epnn_atom.cu"
}
namespace k_bconst {
#include "../../epnn_b200/csrc/epnn_bundle_const.cu"
}
namespace k_aconst {
#include "../../epnn_b200/csrc/epnn_atom_const.cu"
}
namespace k_farc {
#include "../../epnn_b200/csrc/epnn_gnn_far_const.cu"
}
namespace k_mma {
#include "../../epnn_b200/csrc/epnn_bundle_mma.cu"
}
namespace k_brun {
#include "../../epnn_b200/csrc/epnn_bundle_run.cu"
}

static void exclusive_scan(const int* in, int* out, int n) { int s = 0; for (int i = 0; i < n; ++i) { out[i] = s; s += in[i]; } out[n] = s; }

extern "C" int emu_infer(int T, int n_x, const float* w_packed, size_t n_w, int n_sys, const int* off, const float* xyz,
                         const int* species, const float* Q, const int* npad_in, int variant, int dedup,
                         float* q_out, double* q_out64, float* h_out, long long* dedup_rows_out) {
    if (n_w != expected_floats(T, n_x) || variant < 0 || variant > 3) return -1;
    // variant: 0 "pair_const" 0, 1 "pair_const" 1, 2 "pair_const" 0 with "pair_tensor" 1, 3 "pair_const" 2 (the shipped set)
    KernelOptions opt;
    opt.pair_const = variant == 1 ? 1 : variant == 3 ? 2 : 0;
    opt.pair_tensor = variant == 2;
    opt.far_tensor = 0;
    const KernelChoice kc = resolve_kernels(32, 0, opt);
    // one SM: the partial-sum planes grow with the SM count; at one the 49..90-atom systems of the tests still get 3 to 16
    constexpr int kSmCount = 1;
    ChunkPlan pl;
    if (!plan_chunk(off, n_sys, kSmCount, 0, 1, kc, pl)) return -1;
    const int n = off[n_sys];
    const int n_species = n_x - 1;
    // ---------------------------------------------------------------- weights: the product's own packing and folding
    double mu[ED];
    rbf_centers_impl(mu);
    std::vector<double> basis(ED * EDR);
    compute_rbf_basis(basis.data());
    k_nbr::emu_set_rbf(mu, basis.data());
    PackedOffsets po;
    std::vector<double> P;
    pack_all(T, n_x, n_species, w_packed, basis.data(), po, P);
    std::vector<float> Pf(po.total);
    for (size_t i = 0; i < po.total; ++i) Pf[i] = (float)P[i];
    std::vector<StepW<float>> msg(T), pas(T);
    for (int t = 0; t < T; ++t) { msg[t] = step_view<float>(Pf.data(), po.msg[t]); pas[t] = step_view<float>(Pf.data(), po.pas[t]); }
    const UpdW<float> upd = upd_view<float>(Pf.data(), po);

    // ---------------------------------------------------------------- prep + neighbour list + descriptors
    std::vector<int> npad(n_sys), atom_sys(n), deg(n), degU(n), rowptr(n + 1), ustart(n + 1);
    for (int s = 0; s < n_sys; ++s) npad[s] = npad_in ? npad_in[s] : off[s + 1] - off[s];
    std::vector<double> q(n);
    emu_launch_simple(div_up(n, 256), 256, [&] { k_nbr::prep_kernel(n, n_sys, off, Q, atom_sys.data(), q.data()); });
    const long long cells = pl.n_cells;
    std::vector<CellGrid> grid(n_sys + 1);
    std::vector<int> cell_start((size_t)cells + 2, 0), cell_atoms(n + 1, 0);
    if (pl.n_large) {
        std::vector<int> cnt((size_t)cells + 2, 0);
        emu_launch_grid(pl.n_large, 8, 0, [&] { k_nbr::cell_setup_kernel(pl.n_large, pl.cell_tab.data(), pl.cell_tab.data() + pl.n_large, off, xyz, grid.data()); });
        emu_launch_simple(div_up(n, 256), 256, [&] { k_nbr::cell_bin_kernel<0>(n, atom_sys.data(), off, xyz, grid.data(), cnt.data(), nullptr, nullptr); });
        exclusive_scan(cnt.data(), cell_start.data(), (int)cells);
        std::fill(cnt.begin(), cnt.end(), 0);
        emu_launch_simple(div_up(n, 256), 256, [&] { k_nbr::cell_bin_kernel<1>(n, atom_sys.data(), off, xyz, grid.data(), cnt.data(), cell_start.data(), cell_atoms.data()); });
    }
    emu_launch_grid(div_up(n, 128), 4, 0, [&] {
        k_nbr::nbr_kernel<false>(n, atom_sys.data(), off, xyz, deg.data(), degU.data(), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                 grid.data(), cell_start.data(), cell_atoms.data(), nullptr, 0, n); });
    exclusive_scan(deg.data(), rowptr.data(), n);
    exclusive_scan(degU.data(), ustart.data(), n);
    const int nnz = rowptr[n], Pn = ustart[n];
    std::vector<int> col(nnz + 1), pid(nnz + 1), pair_i(Pn + 1), pair_j(Pn + 1);
    std::vector<double> pair_D(Pn + 1), Dtmp(nnz + 1);
    std::vector<float> e((size_t)(Pn + 1) * EDR);
    std::vector<unsigned char> near(Pn + 16), perm_j(Pn + 16);
    emu_launch_grid(div_up(n, 128), 4, 0, [&] {
        k_nbr::nbr_kernel<true>(n, atom_sys.data(), off, xyz, nullptr, nullptr, rowptr.data(), ustart.data(), col.data(), pair_i.data(), pair_j.data(),
                                pair_D.data(), grid.data(), cell_start.data(), cell_atoms.data(), Dtmp.data(), 0, n); });
    emu_launch_simple(div_up(n, 128), 128, [&] { k_nbr::nbr_rev_kernel(n, rowptr.data(), ustart.data(), degU.data(), col.data(), pid.data()); });
    if (Pn > 0)
        emu_launch_grid(div_up(Pn, EDGE_PAIRS), EDGE_PAIRS / 32, 0, [&] { k_nbr::edge_desc_kernel<EDR>((int64_t)Pn, pair_D.data(), e.data(), near.data(), nullptr, nullptr, nullptr, nullptr); });

    // ---------------------------------------------------------------- bundles, far lists, row groups, species tables
    std::vector<int2> bundles = pl.bundles;
    const int n_bundles = (int)bundles.size();
    bundles.push_back(make_int2(0, 0));
    std::vector<int> far_cnt(n + 1, 0), far_off(n + 1, 0), far0_cnt(n + 1, 0), far0_off(n + 1, 0), rep(n + 1, 0), atom_b0(n + 1, 0), bundle_nat(n + 1, 0);
    emu_launch_simple(div_up(n, 256), 256, [&] { k_bundle::far_count_kernel(n, atom_sys.data(), off, npad.data(), rowptr.data(), far_cnt.data()); });
    if (n_bundles) emu_launch_simple(div_up(n_bundles, 128), 128, [&] { k_bundle::bundle_mark_kernel(n_bundles, bundles.data(), atom_b0.data(), bundle_nat.data()); });
    exclusive_scan(far_cnt.data(), far_off.data(), n);
    std::vector<unsigned short> far_list(far_off[n] + 2), far0_list((size_t)(MAX_SPECIES + 1) * n + 2);
    std::vector<unsigned char> far0_w((size_t)(MAX_SPECIES + 1) * n + 16);
    if (n_bundles) {
        if (kc.tile_perm && Pn > 0)
            emu_launch_simple(div_up(Pn, 256), 256, [&] {
                k_bundle::tile_perm_kernel((int64_t)Pn, pair_i.data(), pair_j.data(), atom_sys.data(), off, atom_b0.data(), ustart.data(),
                                           bundle_nat.data(), perm_j.data()); });
        emu_launch_simple(div_up(n, 128), 128, [&] {
            k_bundle::far_fill_kernel(n, atom_sys.data(), off, npad.data(), rowptr.data(), col.data(), atom_b0.data(), far_off.data(), far_list.data()); });
    }
    emu_launch_simple(div_up(n, 128), 128, [&] {
        k_bundle::far0_kernel<0>(n, atom_sys.data(), off, npad.data(), species, rowptr.data(), col.data(), nullptr, rep.data(), far0_cnt.data(),
                                 nullptr, nullptr, nullptr); });
    exclusive_scan(far0_cnt.data(), far0_off.data(), n);
    if (n_bundles)
        emu_launch_simple(div_up(n, 128), 128, [&] {
            k_bundle::far0_kernel<1>(n, atom_sys.data(), off, npad.data(), species, rowptr.data(), col.data(), atom_b0.data(), nullptr, nullptr,
                                     far0_off.data(), far0_list.data(), far0_w.data()); });
    std::vector<unsigned char> rowl(nnz + 16, 0);
    if (kc.csr_rowl && n_bundles && nnz > 0)
        emu_launch_simple(div_up(n, 256), 256, [&] { k_brun::csr_rowl_kernel(n, atom_sys.data(), off, rowptr.data(), atom_b0.data(), rowl.data()); });
    std::vector<int> rgl_off(n_sys + 1, 0), rg;
    for (int s = 0; s < n_sys; ++s) {
        const int ns = off[s + 1] - off[s];
        rgl_off[s + 1] = rgl_off[s] + (ns > SMALL_MAX ? (ns + 3) >> 2 : 0);
        if (ns > SMALL_MAX) for (int i = off[s]; i < off[s + 1]; i += 4) rg.push_back(i);
    }
    const int n_rg = pl.n_rg_large;
    rg.push_back(0);
    const int nsplit = pl.nsplit;
    const int n_sp_tab = n_rg / 8 + 2;
    std::vector<int> sp_tab((size_t)n_sp_tab * 32, 0), sp_stamp((size_t)n_sp_tab * 2, 0);
    unsigned long long dedup_rows = 0;
    const bool use_tabs = n_rg > 0 && dedup;
    if (use_tabs) {
        emu_launch_simple(div_up((int64_t)n_sp_tab * 32, 256), 256, [&] { k_gnn::sp_tab_init_kernel(n_sp_tab, sp_tab.data(), sp_stamp.data()); });
        emu_launch_grid(div_up(n, 256), 8, 0, [&] {
            k_gnn::sp_tab_fill_kernel(n, atom_sys.data(), off, species, rgl_off.data(), deg.data(), sp_tab.data(), sp_stamp.data()); });
    }

    // ---------------------------------------------------------------- state
    std::vector<float> h((size_t)n * HD, 0.f), l2((size_t)n * HID, 0.f), S((size_t)nsplit * n * HID, 0.f), u((size_t)n * HID), v((size_t)n * HID), delta(Pn + 1, 0.f);
    int work_counter = 0;
    constexpr int NW = 8;

    auto atom = [&](int mode, const StepW<float>* prev, const StepW<float>* next, int h_is_zero) {
        if (kc.atom == ATOM_K_CONST) {
            k_aconst::AtomW W;
            memset(&W, 0, sizeof(W));
            k_aconst::AtomConstArgs aa;
            memset(&aa, 0, sizeof(aa));
            if (mode & ATOM_UPDATE) {
                memcpy(W.HG, prev->HG, sizeof(W.HG)); memcpy(W.g, prev->g, sizeof(W.g));
                memcpy(W.cb, (mode & ATOM_FIRST) ? upd.c1 : upd.cb1, sizeof(W.cb));
                memcpy(W.U2, upd.U2, sizeof(W.U2)); memcpy(W.c2, upd.c2, sizeof(W.c2)); memcpy(W.U3, upd.U3, sizeof(W.U3)); memcpy(W.c3, upd.c3, sizeof(W.c3));
            }
            if (mode & ATOM_PROJECT) { memcpy(W.Pf, next->Pf, sizeof(W.Pf)); memcpy(W.Aq, next->Aq64, sizeof(W.Aq)); aa.Ax = h_is_zero ? next->Ax64 : next->Axf; }
            aa.n_atoms = n; aa.mode = mode; aa.nsplit = nsplit; aa.h_is_zero = h_is_zero;
            aa.atom_sys = atom_sys.data(); aa.sys_off = off; aa.npad = npad.data(); aa.species = species;
            aa.Spart = S.data(); aa.h = h.data(); aa.l2 = l2.data(); aa.rowptr = rowptr.data(); aa.col = col.data(); aa.pid = pid.data();
            aa.delta = delta.data(); aa.q = q.data(); aa.u = u.data(); aa.v = v.data(); aa.q_out = q_out; aa.q_out64 = q_out64;
            emu_launch_grid(2, ACONST_NW, (size_t)ACONST_NW * 32 * ATS, [&] { k_aconst::atom_const_kernel(W, aa); });
            return;
        }
        AtomArgs<float, float> aa;
        memset(&aa, 0, sizeof(aa));
        aa.n_atoms = n; aa.mode = mode; aa.nsplit = nsplit; aa.h_is_zero = h_is_zero;
        aa.atom_sys = atom_sys.data(); aa.sys_off = off; aa.npad = npad.data(); aa.species = species;
        aa.Spart = S.data(); aa.h = h.data(); aa.l2 = l2.data();
        if (mode & ATOM_UPDATE) { aa.HG = prev->HG; aa.g = prev->g; aa.upd = upd; aa.cb = (mode & ATOM_FIRST) ? upd.c1 : upd.cb1; }
        aa.rowptr = rowptr.data(); aa.col = col.data(); aa.pid = pid.data(); aa.delta = delta.data(); aa.q = q.data();
        if (mode & ATOM_PROJECT) { aa.Pf = next->Pf; aa.Aq64 = next->Aq64; aa.Ax = h_is_zero ? next->Ax64 : next->Axf; }
        aa.u = u.data(); aa.v = v.data(); aa.q_out = q_out; aa.q_out64 = q_out64;
        constexpr int ANW = 4;
        const size_t smem = sizeof(float) * (ATOM_W_UPD + ATOM_W_PROJ + (size_t)ANW * ATOM_TILE + ANW * 64) + sizeof(int) * ANW * 64;
        emu_launch_grid(2, ANW, smem / sizeof(float) + 8, [&] { k_atom::atom_kernel<float, ANW, float, false>(aa); });
    };
    auto bundle = [&](bool epn, const StepW<float>& sw) {
        if (!n_bundles) return;
        work_counter = 0;
        if (epn && kc.epn == EPN_MMA) {
            k_mma::EpnMmaArgs a;
            a.n_bundles = n_bundles; a.bundle = bundles.data(); a.work_counter = &work_counter;
            a.ustart = ustart.data(); a.pair_i = pair_i.data(); a.pair_j = pair_j.data(); a.near = near.data(); a.e = e.data();
            a.u = u.data(); a.v = v.data(); a.Cw = sw.Cw; a.W2 = sw.W2; a.b2 = sw.b2; a.w3 = sw.W3; a.delta = delta.data();
            emu_launch_cta(MMA_NW, (size_t)MMA_NW * BUNDLE_ATOMS * UVS, [&] { k_mma::bundle_epn_mma_kernel(a); });
            return;
        }
        if (!epn && kc.gnn == GNN_RUN) {
            k_brun::RunW W;
            memcpy(W.W2, sw.W2, sizeof(W.W2));
            k_brun::RunArgs a;
            memset(&a, 0, sizeof(a));
            a.n_bundles = n_bundles; a.bundle = bundles.data(); a.work_counter = &work_counter;
            a.rowptr = rowptr.data(); a.col = col.data(); a.pid = pid.data(); a.rowl = rowl.data(); a.e = e.data(); a.ustart = ustart.data();
            a.far_off = far_off.data(); a.far_list = far_list.data();
            a.far0_off = far0_off.data(); a.far0_list = far0_list.data(); a.far0_w = far0_w.data(); a.rep = rep.data(); a.dedup = dedup;
            a.atom_sys = atom_sys.data(); a.sys_off = off; a.npad = npad.data(); a.u = u.data(); a.v = v.data(); a.S = S.data();
            a.Cw = sw.Cw; a.b2 = sw.b2; a.b1 = sw.b1;
            emu_launch_cta(RUN_NW, k_brun::RunSmem::bytes() / sizeof(float), [&] { k_brun::bundle_run_kernel(W, &a); });
            return;
        }
        if (epn ? kc.epn == EPN_CONST : kc.gnn == GNN_CONST) {
            k_bconst::PairW W;
            memcpy(W.W2, sw.W2, sizeof(W.W2));
            k_bconst::ConstArgs a;
            a.n_bundles = n_bundles; a.bundle = bundles.data(); a.work_counter = &work_counter;
            a.ustart = ustart.data(); a.pair_i = pair_i.data(); a.pair_j = pair_j.data(); a.near = near.data(); a.e = e.data();
            a.far_off = far_off.data(); a.far_list = far_list.data();
            a.far0_off = far0_off.data(); a.far0_list = far0_list.data(); a.far0_w = far0_w.data(); a.rep = rep.data(); a.dedup = dedup;
            a.atom_sys = atom_sys.data(); a.sys_off = off; a.npad = npad.data(); a.u = u.data(); a.v = v.data(); a.S = S.data(); a.delta = delta.data();
            a.Cw = sw.Cw; a.b2 = sw.b2; a.x32 = epn ? sw.W3 : sw.b1;
            if (epn) emu_launch_cta(CONST_NW, (size_t)CONST_NW * k_bconst::ConstSmem<true>::PW + k_bconst::ConstSmem<true>::SHARED, [&] { k_bconst::bundle_const_kernel<true>(W, &a); });
            else     emu_launch_cta(CONST_NW, (size_t)CONST_NW * k_bconst::ConstSmem<false>::PW + k_bconst::ConstSmem<false>::SHARED, [&] { k_bconst::bundle_const_kernel<false>(W, &a); });
            return;
        }
        k_bundle::BundleArgs<float> a;
        a.n_bundles = n_bundles; a.bundle = bundles.data(); a.work_counter = &work_counter;
        a.ustart = ustart.data(); a.pair_i = pair_i.data(); a.pair_j = pair_j.data(); a.near = near.data(); a.e = e.data(); a.perm_j = perm_j.data();
        a.far_off = far_off.data(); a.far_list = far_list.data();
        a.far0_off = far0_off.data(); a.far0_list = far0_list.data(); a.far0_w = far0_w.data(); a.rep = rep.data(); a.dedup = dedup;
        a.atom_sys = atom_sys.data(); a.sys_off = off; a.npad = npad.data(); a.u = u.data(); a.v = v.data();
        a.Cw = sw.Cw; a.W2 = sw.W2; a.b2 = sw.b2; a.x32 = epn ? sw.W3 : sw.b1; a.S = S.data(); a.delta = delta.data();
        if (epn) emu_launch_cta(NW, k_bundle::BundleSmem<float, true>::bytes(NW) / sizeof(float) + 8, [&] { k_bundle::bundle_kernel<float, NW, true>(a); });
        else     emu_launch_cta(NW, k_bundle::BundleSmem<float, false>::bytes(NW) / sizeof(float) + 8, [&] { k_bundle::bundle_kernel<float, NW, false>(a); });
    };

    // ---------------------------------------------------------------- GNN layer (charge_gn.py:60-74), launch order of run_layers
    atom(ATOM_PROJECT, nullptr, &msg[0], 1);
    for (int t = 0; t < T; ++t) {
        bundle(false, msg[t]);
        if (n_rg > 0) {
            const int stamp = use_tabs ? t + 1 : 0;
            if (stamp) {
                emu_launch_simple(div_up((int64_t)n * 8, 256), 256, [&] {
                    k_gnn::sp_check_kernel<float>(n, atom_sys.data(), off, species, rgl_off.data(), sp_tab.data(), v.data(), sp_stamp.data(), stamp); });
                emu_launch_simple(div_up(n_sp_tab, 256), 256, [&] { k_gnn::sp_tally_kernel(n_sp_tab, sp_tab.data(), sp_stamp.data(), stamp, &dedup_rows); });
            }
            // FAR_CONST: the far columns of the live steps go to the row-per-thread kernel (planes 0 .. nsplit - 2), gnn_pair_kernel
            // keeps the near pairs, the pad pair and the species slots on the last plane
            const bool far_const = pl.far == FAR_CONST;
            if (far_const) {
                k_farc::FarW FW;
                memcpy(FW.W2, msg[t].W2, sizeof(FW.W2)); memcpy(FW.b2, msg[t].b2, sizeof(FW.b2));
                k_farc::FarConstArgs fa;
                fa.blk = pl.rowblk.data(); fa.nsplit = nsplit - 1; fa.n_atoms = n;
                fa.unit_begin = pl.blk_begin * (nsplit - 1); fa.unit_end = pl.blk_end * (nsplit - 1);
                fa.sys_off = off; fa.rowptr = rowptr.data(); fa.col = col.data(); fa.u = u.data(); fa.v = v.data(); fa.S = S.data();
                fa.rgl_off = rgl_off.data(); fa.sp_stamp = sp_stamp.data(); fa.stamp = stamp;
                emu_launch_grid(2, FARC_NW, (size_t)FARC_NW * FARC_PW_BYTES / sizeof(float) + 8, [&] { k_farc::gnn_far_const_kernel(FW, fa); });
            }
            k_gnn::GnnArgs<float> ga;
            const int ns = far_const ? 1 : nsplit;
            ga.rg_atom = rg.data(); ga.unit_begin = pl.rg_begin * ns; ga.n_units = pl.rg_end * ns; ga.nsplit = ns; ga.n_atoms = n;
            ga.skip_far = far_const ? 1 : 0; ga.plane = far_const ? nsplit - 1 : 0;
            ga.atom_sys = atom_sys.data(); ga.sys_off = off; ga.npad = npad.data(); ga.rowptr = rowptr.data(); ga.col = col.data(); ga.pid = pid.data();
            ga.e = e.data(); ga.u = u.data(); ga.v = v.data(); ga.Cw = msg[t].Cw; ga.W2 = msg[t].W2; ga.b2 = msg[t].b2; ga.b1 = msg[t].b1; ga.S = S.data();
            ga.species = species; ga.rgl_off = rgl_off.data(); ga.sp_tab = sp_tab.data(); ga.sp_stamp = sp_stamp.data(); ga.stamp = stamp; ga.n_species = n_species;
            emu_launch_grid(2, NW, k_gnn::gnn_smem_bytes<float>(NW) / sizeof(float) + 8, [&] { k_gnn::gnn_pair_kernel<float, true, NW>(ga); });
        }
        const StepW<float>* next = t + 1 < T ? &msg[t + 1] : &pas[0];
        atom(ATOM_UPDATE | ATOM_PROJECT | (t == 0 ? ATOM_FIRST : 0) | (t + 1 == T ? ATOM_WRITE_H : 0), &msg[t], next, 0);
    }
    if (h_out) memcpy(h_out, h.data(), sizeof(float) * (size_t)n * HD);
    // ---------------------------------------------------------------- EPN layer (charge_gn.py:98-118)
    for (int t = 0; t < T; ++t) {
        bundle(true, pas[t]);
        if (n_rg > 0 && Pn > 0) {
            k_epn::EpnArgs<float> ea;
            ea.P = Pn; ea.tile_begin = 0; ea.tile_end = (Pn + 31) / 32;
            ea.pair_i = pair_i.data(); ea.pair_j = pair_j.data(); ea.near = near.data(); ea.e = e.data(); ea.atom_sys = atom_sys.data(); ea.sys_off = off;
            ea.u = u.data(); ea.v = v.data(); ea.Cw = pas[t].Cw; ea.W2 = pas[t].W2; ea.b2 = pas[t].b2; ea.w3 = pas[t].W3; ea.delta = delta.data();
            const size_t smem = sizeof(float) * (EDR * HID + HID * HID + 2 * HID + (size_t)NW * (32 * EDR + 32 * HID)) + sizeof(int) * NW * 64;
            emu_launch_grid(2, NW, smem / sizeof(float) + 8, [&] { k_epn::epn_pair_kernel<float, NW>(ea); });
        }
        if (t + 1 < T) atom(ATOM_QUPDATE | ATOM_PROJECT, nullptr, &pas[t + 1], 0);
        else atom(ATOM_QUPDATE | ATOM_OUTPUT, nullptr, nullptr, 0);
    }
    if (dedup_rows_out) *dedup_rows_out = (long long)dedup_rows;
    return 0;
}
