// Work plan of the electrostatics kernels (epnn_elst.cu), shared by epnn_api.cu and the CPU warp emulation (tools/emu).
#pragma once
#include <stdint.h>

#include <algorithm>
#include <vector>

#define ELST_SMALL_MAX 48      // systems of at most this many atoms: one warp each (the bundle bound, SMALL_MAX)
#define ELST_WARPS 8           // warps per CTA of the small-system kernel
#define ELST_TILE 128          // large systems: targets per pair CTA = sources per shared-memory tile
#define ELST_MIN_PART 256      // fewest sources in one part of a split source range
#define ELST_CTAS_PER_SM 32    // pair CTAs a split aims at per SM (several waves: the last, partial one costs little)
#define ELST_RED 256           // threads of the per-system reduction CTA

// One pair CTA: targets [t0, t0 + ELST_TILE) of the system whose chunk-local first atom is a0, against sources [s0, s1)
// of the same system; its partial potentials go to partial[pw + t].
struct ElstItem { int a0, n, t0, s0, s1, pad; long long pw; };
// One large system: chunk-local first atom, size, system index in the chunk, source parts, first partial row.
struct ElstSys { int a0, n, s, parts; long long pofs; };

// Source parts of a system of n > ELST_SMALL_MAX atoms: enough pair CTAs to fill `target_ctas` (ELST_CTAS_PER_SM per SM)
// when the system has too few target tiles, but no part shorter than ELST_MIN_PART sources.  Depends on n and the SM
// count only, so a system's sums do not depend on the other systems of the call.
static inline int elst_parts(int n, int64_t target_ctas) {
    const int64_t tiles = (n + ELST_TILE - 1) / ELST_TILE;
    const int64_t want = (target_ctas + tiles - 1) / tiles;
    const int64_t cap = (n + ELST_MIN_PART - 1) / ELST_MIN_PART;
    return (int)std::max<int64_t>(1, std::min(want, cap));
}

// Pair CTAs and reduction rows of the large systems of a chunk.  off: the chunk's n_sys + 1 offsets (off[0] = the chunk's
// first atom).  Returns the length of the partial-potential buffer (sum over large systems of parts * n).
static inline long long elst_plan(const int32_t* off, int64_t n_sys, int64_t target_ctas, std::vector<ElstItem>& items,
                                  std::vector<ElstSys>& sys) {
    items.clear();
    sys.clear();
    long long len = 0;
    for (int64_t s = 0; s < n_sys; ++s) {
        const int n = off[s + 1] - off[s];
        if (n <= ELST_SMALL_MAX) continue;
        const int a0 = off[s] - off[0], parts = elst_parts(n, target_ctas);
        sys.push_back(ElstSys{a0, n, (int)s, parts, len});
        for (int p = 0; p < parts; ++p) {
            const int s0 = (int)((int64_t)p * n / parts), s1 = (int)((int64_t)(p + 1) * n / parts);
            for (int t0 = 0; t0 < n; t0 += ELST_TILE) items.push_back(ElstItem{a0, n, t0, s0, s1, 0, len + (long long)p * n});
        }
        len += (long long)parts * n;
    }
    return len;
}

// ---- potential and field at given points (epnn_potential_points) ---------------------------------------------------
#define ELST_PT_TILE 128       // points per CTA of the point kernel = atoms per shared-memory tile
#ifndef ELST_PT_PART
#define ELST_PT_PART 1024      // atoms per source part: a system of n atoms has ceil(n / ELST_PT_PART) parts
#endif
#define ELST_PT_CHUNK 4194304  // cost units per chunk: a point costs 1, or its system's part count when that exceeds 1

// One point CTA: points [p0, p0 + np) of the chunk (one system's) against the atoms [s0, s1) of that system, whose
// chunk-local first atom is a0.  pw < 0: a single-part system, the CTA writes the outputs; otherwise its partial sums go
// to partial rows pw + t.
struct ElstPtItem { long long p0, pw; int a0, s0, s1, np; };
// One reduction CTA: points [p0, p0 + np) of a split system; part k of point t is partial row pw + k * stride + t.
struct ElstPtRed { long long p0, pw, stride; int np, parts; };
// One chunk: the systems [s0, s1) it touches and its points [p0, p1).
struct ElstPtChunk { int64_t s0, s1, p0, p1; };

static inline int elst_pt_parts(int n) { return (n + ELST_PT_PART - 1) / ELST_PT_PART; }
static inline int64_t elst_pt_cost(int n) { return std::max(1, elst_pt_parts(n)); }

// Cuts the points of a call into chunks of at most `budget` cost units (ELST_PT_CHUNK in the library, so the partial
// workspace stays bounded; at least the largest part count) and at most max_atoms atoms (unless one system has more).
// One system's points may span chunks: a point's sums do not depend on which other points share its chunk.
// poff: int64 point offsets, poff[0] = 0, non-decreasing.
static inline void elst_pt_chunks(const int32_t* off, const int64_t* poff, int64_t n_sys, int64_t max_atoms, int64_t budget,
                                  std::vector<ElstPtChunk>& chunks) {
    chunks.clear();
    int64_t s = 0, p = 0;                                         // next system, next point
    for (;;) {
        while (s < n_sys && poff[s + 1] <= p) ++s;                 // systems without points left
        if (s >= n_sys) break;
        ElstPtChunk c{s, s, p, p};
        int64_t used = 0;
        while (s < n_sys) {
            if (c.s1 > c.s0 && (int64_t)off[s + 1] - off[c.s0] > max_atoms) break;
            const int64_t cost = elst_pt_cost(off[s + 1] - off[s]);
            const int64_t take = std::min(poff[s + 1] - p, (budget - used) / cost);
            if (take <= 0 && poff[s + 1] > p) break;              // the budget is spent
            p += take; used += take * cost;
            c.s1 = s + 1; c.p1 = p;
            if (p < poff[s + 1]) break;
            ++s;
        }
        chunks.push_back(c);
    }
}

// Point CTAs and reduction CTAs of one chunk.  Returns the number of partial rows (sum over split systems of their points
// in the chunk times their part count).
static inline long long elst_pt_plan(const int32_t* off, const int64_t* poff, const ElstPtChunk& c,
                                     std::vector<ElstPtItem>& items, std::vector<ElstPtRed>& red) {
    items.clear();
    red.clear();
    long long rows = 0;
    for (int64_t s = c.s0; s < c.s1; ++s) {
        const int64_t q0 = std::max(poff[s], c.p0), q1 = std::min(poff[s + 1], c.p1);
        if (q1 <= q0) continue;
        const int n = off[s + 1] - off[s], a0 = off[s] - off[c.s0], parts = elst_pt_parts(n);
        for (int64_t t0 = q0; t0 < q1; t0 += ELST_PT_TILE) {
            const int np = (int)std::min<int64_t>(ELST_PT_TILE, q1 - t0);
            for (int k = 0; k < parts; ++k) {
                const int s0 = k * ELST_PT_PART, s1 = std::min(n, s0 + ELST_PT_PART);
                const long long pw = parts == 1 ? -1 : rows + (long long)k * (q1 - q0) + (t0 - q0);
                items.push_back(ElstPtItem{t0 - c.p0, pw, a0, s0, s1, np});
            }
            if (parts > 1) red.push_back(ElstPtRed{t0 - c.p0, rows + (t0 - q0), q1 - q0, np, parts});
        }
        if (parts > 1) rows += (long long)parts * (q1 - q0);
    }
    return rows;
}

// Everything the point kernels read and write; atoms, points and outputs are chunk-local, phi or field may be NULL.
struct ElstPtArgs {
    const float* xyz;                // [3 * atoms]
    const double* q;                 // [atoms]
    const double* pts;               // [3 * points]
    double* phi;                     // [points]
    double* field;                   // [3 * points]
    const ElstPtItem* items;
    const ElstPtRed* red;
    double* partial;                 // [rows * 4] with the field, [rows] without
};

// Everything the three kernels read and write; atom arrays and outputs are chunk-local, each output may be NULL.
struct ElstArgs {
    int n_sys, base;                 // systems of the chunk; base = absolute index of its first atom (off[0])
    const int* off;                  // n_sys + 1 absolute offsets
    const float* xyz;                // [3 * atoms]
    const double* q;                 // [atoms]
    const int* frag;                 // [atoms] fragment labels, or NULL
    double* energy;                  // [n_sys]
    double* dipole;                  // [3 * n_sys]
    double* phi;                     // [atoms]
    const ElstItem* items;
    const ElstSys* sys;
    double* partial;
};
