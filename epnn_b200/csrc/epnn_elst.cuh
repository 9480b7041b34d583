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
