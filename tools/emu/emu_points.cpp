// CPU emulation driver for the point kernels of epnn_b200/csrc/epnn_elst.cu (test infrastructure; see cuda_emu.h).
// Build: g++ -O1 -std=c++17 -ffp-contract=off -shared -fPIC -pthread -DEPNN_CPU_EMU -o build/libemu_points.so tools/emu/emu_points.cpp
#define EPNN_CPU_EMU 1
#include "../../epnn_b200/csrc/epnn_elst.cu"

extern "C" int emu_points_parts(int n) { return elst_pt_parts(n); }

// The chunks of a call (s0, s1, p0, p1 per chunk into out, at most cap of them); returns their number.
extern "C" int emu_points_chunks(long long n_sys, const int* off, const long long* poff, long long max_atoms, long long budget,
                                 long long* out, int cap) {
    std::vector<ElstPtChunk> chunks;
    elst_pt_chunks(off, (const int64_t*)poff, n_sys, max_atoms, budget, chunks);
    for (size_t k = 0; k < chunks.size() && (int)k < cap; ++k) {
        out[4 * k] = chunks[k].s0; out[4 * k + 1] = chunks[k].s1; out[4 * k + 2] = chunks[k].p0; out[4 * k + 3] = chunks[k].p1;
    }
    return (int)chunks.size();
}

// One call of the library: the chunks and plans epnn_api.cu builds, then the point and reduction kernels of each chunk in
// launch order.  max_atoms and budget stand for the ctx's chunk_atoms and ELST_PT_CHUNK, so that small calls reach
// chunk boundaries.  phi or field may be NULL (not both).  Returns the number of point CTAs.
extern "C" long long emu_points(long long n_sys, const int* off, const float* xyz, const double* q, const long long* poff,
                                const double* pts, long long max_atoms, long long budget, double* phi,
                                double* field) {
    std::vector<ElstPtChunk> chunks;
    elst_pt_chunks(off, (const int64_t*)poff, n_sys, max_atoms, budget, chunks);
    std::vector<ElstPtItem> items;
    std::vector<ElstPtRed> red;
    long long n_items = 0;
    for (const ElstPtChunk& ch : chunks) {
        const long long rows = elst_pt_plan(off, (const int64_t*)poff, ch, items, red);
        std::vector<double> partial((size_t)(rows * (field ? 4 : 1)) + 1, std::nan(""));
        ElstPtArgs a;
        a.xyz = xyz + 3 * (size_t)off[ch.s0]; a.q = q + off[ch.s0]; a.pts = pts + 3 * ch.p0;
        a.phi = phi ? phi + ch.p0 : nullptr; a.field = field ? field + 3 * ch.p0 : nullptr;
        a.items = items.data(); a.red = red.data(); a.partial = partial.data();
        if (field) {
            emu_launch_grid((int)items.size(), ELST_PT_TILE / 32, 0, [&] { elst_point_kernel<true>(a); });
            if (!red.empty()) emu_launch_grid((int)red.size(), ELST_PT_TILE / 32, 0, [&] { elst_point_reduce_kernel<true>(a); });
        } else {
            emu_launch_grid((int)items.size(), ELST_PT_TILE / 32, 0, [&] { elst_point_kernel<false>(a); });
            if (!red.empty()) emu_launch_grid((int)red.size(), ELST_PT_TILE / 32, 0, [&] { elst_point_reduce_kernel<false>(a); });
        }
        n_items += (long long)items.size();
    }
    return n_items;
}
