/*
 * epnn_b200.h -- C-ABI of the B200-native EPNN charge-inference library (libepnn_b200.so).
 *
 * The reference (derekmetcalf/epnn) has no FFI/plugin interface: its boundary is the Python surface
 * of charge_gn.py / infer.py.  Each entry point below names the reference code it replaces; the
 * Python facade in epnn_b200/charge_gn.py + epnn_b200/infer.py binds these through ctypes (see
 * INTEGRATION.md for the stub a maintainer of the reference would add).
 *
 * Conventions
 *   - every function returns int: 0 = ok, negative = error (EPNN_E_*); nothing throws across the ABI;
 *     epnn_last_error() returns the message for the last failure on that ctx (or, with ctx == NULL,
 *     of the last failed epnn_create on this thread).
 *   - the caller owns every buffer.  Un-suffixed entry points take HOST pointers and do their own
 *     host<->device copies on the ctx stream; *_dev entry points take DEVICE pointers on the ctx device.
 *   - a ctx owns its device weights, workspaces and one CUDA stream; one ctx per GPU; a ctx is not
 *     thread-safe; distinct ctxs are independent; there is no global state.
 *   - there is no CPU fallback: if no CUDA device is usable, epnn_create fails with EPNN_E_CUDA.
 */
#ifndef EPNN_B200_H
#define EPNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EPNN_OK            0
#define EPNN_E_INVALID    -1   /* bad argument (null pointer, negative size, npad < n, species out of range, ...) */
#define EPNN_E_CUDA       -2   /* CUDA runtime / driver failure; message holds cudaGetErrorString */
#define EPNN_E_NOMEM      -3   /* host or device allocation failed */
#define EPNN_E_CAPACITY   -4   /* caller-provided output buffer too small */
#define EPNN_E_UNSUPPORTED -5  /* shape outside what the kernels were built for */

#define EPNN_H_DIM 48          /* hidden width h_dim  (reference infer.py:38) */
#define EPNN_E_DIM 48          /* radial basis size e_dim (reference infer.py:39, charge_gn.py:331) */
#define EPNN_HID   32          /* hidden width of message/pass MLPs (reference charge_gn.py:52,84) */

typedef struct epnn_ctx epnn_ctx;

/* Per-call statistics (all optional).  Times are CUDA-event milliseconds on the ctx stream and are
 * only filled when the "timing" option is on (events serialise nothing, but they are extra work). */
typedef struct epnn_stats {
    int64_t n_systems;
    int64_t n_atoms;
    int64_t n_pairs_e;        /* unordered pairs with 0 <= D < 3.0 A, i != j  (e_ij != 0 set) */
    int64_t n_pairs_near;     /* unordered pairs in the reference's is_near set (charge_gn.py:90-94) */
    int64_t n_row_groups;     /* GNN work units: bundles of small systems + 4-row groups of large systems */
    int64_t n_chunks;         /* internal batches the call was split into */
    int64_t n_launches;       /* kernels launched by this call */
    float ms_total;           /* first H2D copy -> last D2H copy */
    float ms_h2d;
    float ms_neighbor;        /* neighbour list + radial descriptors */
    float ms_gnn_pair;        /* sum over the T message-passing pair kernels */
    float ms_gnn_atom;        /* per-atom update / projection kernels of the GNN layer */
    float ms_epn_pair;        /* sum over the T electron-passing pair kernels */
    float ms_epn_atom;        /* segmented charge reductions + projections of the EPN layer */
    float ms_d2h;
    int64_t n_far_dedup_rows; /* rows of systems with more than 48 atoms whose far (e == 0) columns were collapsed to one
                                 weighted slot per species, summed over the T message-passing steps ("dedup_far") */
    int64_t n_gnn_near_slots; /* ordered near (e != 0) slots and far slots (far columns, or one weighted slot per species where the */
    int64_t n_gnn_far_slots;  /*   exact de-duplication applied, + pad slots) the small-system GNN kernel evaluated, summed over the T steps */
    int32_t precision_used;   /* 32, 48 (mixed) or 64: what "precision" resolved to for this call */
    float probe_err32;        /* "precision" 0 (auto): max |dq| of the FP32 / mixed kernels against the FP64 kernels on the */
    float probe_err48;        /*   probe sample of the first call (e); -1 if that candidate was not needed / no probe ran */
    int32_t atom_tensor_used; /* 1 if the FP32 per-atom kernel of this call ran on the warp-level tensor path ("atom_tensor") */
} epnn_stats;

/* Build a context on CUDA device `device` and upload the model once.
 * Replaces: charge_gn.make_model(layers,h_dim,T,n_elems,natom) + model.load_weights(prefix)
 *           (reference charge_gn.py:369-391, infer.py:56-57).
 * packed_weights (host, float32), n_floats = T*(K*32+32+32*32+32+32*32+32) + (80*32+32+32*32+32+32*48+48)
 *           + T*(K*32+32+32*32+32+32+1) with K = 2*(n_x+49)+48, in this order, every kernel row-major (in,out):
 *   for t in 0..T-1: message MLP t:  W1[K][32] b1[32] W2[32][32] b2[32] W3[32][32] b3[32]
 *   update MLP:                       U1[80][32] c1[32] U2[32][32] c2[32] U3[32][48] c3[48]
 *   for t in 0..T-1: pass MLP t:     P1[K][32] b1[32] P2[32][32] b2[32] P3[32][1]  b3[1]
 * First-layer row order is [x_i | h_i | q_i | x_j | h_j | q_j | e_ij] (reference charge_gn.py:62-65).
 * n_x selects the element table: 9 -> H C N O F S Cl Br (infer.py:13-30), 10 -> H C N O F P S Cl Br
 * (charge_gn.py:9-28); per-atom features are x = [Z, onehot]. */
int epnn_create(int device, int T, int n_x, const float* packed_weights, size_t n_floats, epnn_ctx** out);

void epnn_destroy(epnn_ctx* ctx);

const char* epnn_last_error(const epnn_ctx* ctx);

/* Options: "precision" 32 (default: FP32 SIMT kernels, charges carried in FP64), 48 (mixed: FP32 pair kernels around an FP64
 * per-atom kernel -- update MLP, first-layer projections and the hidden state in FP64), 64 (every kernel in FP64) or
 * 0 (auto: the first call runs a bounded prefix of its systems -- at most 64 systems / 8192 atoms -- through all three and
 * keeps the cheapest candidate (FP32 with the tensor per-atom kernel if "atom_tensor" is on, FP32 SIMT, mixed) whose charges
 * are within "auto_tol", default 2.5e-6 e, of the FP64 kernels; sticky for the ctx; reported in epnn_stats).  The reference's 1e-5 e tolerance needs 32 for decay_model_weights, 48 for model2_weights
 * and 64 for model_weights (|h| reaches 150 there: FP32 pair kernels alone are 6e-5 off); "timing" 0/1; "chunk_atoms" (internal batch size);
 * "keep_hidden" 0/1 (retain the final GNN hidden state for epnn_get_hidden);
 * "dedup_far" 1 (default) / 0: far columns whose v rows are identical (same system, same species, same hidden
 * state -- always the case at the first message-passing step, and after every step that leaves the hidden state
 * species-wise constant: 3 of the 5 steps of the reference's default decay_model_weights) are collapsed into one weighted slot per
 * species: an exact reuse of identical messages, checked on the device at every step, switched off only for
 * ablation.  For systems with more than 48 atoms this turns the O(n^2) unmasked message sum of a step into
 * O(n * species) whenever the check holds; otherwise the full sum runs;
 * "gnn_far_tensor" 2 (default: auto) / 1 (on) / 0 (off): systems with more than 48 atoms evaluate the e == 0 ("far") part of
 * the message sum -- the O(n^2) part -- on the tcgen05 tensor cores with a 3xTF32 error-compensated split and FP32
 * accumulation in tensor memory instead of FP32 SIMT (FP32 / mixed precision only; results differ from the SIMT path at
 * the level of FP32 round-off, about 1e-6 relative in the hidden state).  Auto switches it on for calls that hold a
 * system of at least "gnn_far_tensor_min" atoms (default 16384), where the O(n^2) part is > 99 % of the work and the
 * tensor kernel is 1.5x the FP32 SIMT one;
 * "pair_tensor" 0 (default) / 1: systems with at most 48 atoms evaluate the electron-passing pair MLP on the warp-level
 * tensor path (mma.sync m16n8k8 TF32 inputs, 3xTF32 split, FP32 accumulation, operands chained through registers)
 * instead of FP32 SIMT (FP32 / mixed precision only; per-pair transfers differ from the SIMT path by about 1e-6 relative);
 * "atom_tensor" 1 (default) / 0: FP32 calls run the dense layers of the per-atom kernel (folded update MLP, first-layer
 * projections: GEMMs over all atoms of a chunk) on the warp-level tensor path, 3xTF32 split with FP32 accumulation
 * (epnn_atom_mma.cu), which leaves that kernel bound by its HBM traffic; 0 = the FP32 SIMT warp-tile kernel.  Same
 * formulas; results differ at the level of FP32 round-off.  Mixed / FP64 calls are not affected;
 * "fused_prep" 1 (default) / 0: chunks that hold only systems of at most 48 atoms build all their lists (CSR, pair list, far
 * lists) with two warp-per-bundle kernels from one 48-bit neighbour mask per row (epnn_bundle_prep.cu) instead of the general
 * thread-per-atom kernels; identical lists (0 = A/B);
 * "chunk_streams" 1 (default) / 2: multi-chunk calls keep two chunks in flight on two streams with separate workspaces, so
 * the list building and host sync of one chunk run beside the pair kernels of the other (identical results; +2 % throughput
 * on a million molecules, but the per-phase times of epnn_stats then overlap and add up to more than the wall clock);
 * "pair_const": the FP32 kernel set.  2 (default): row-run GNN bundle kernel (epnn_bundle_run.cu: one contiguous run of
 * pair slots per lane, row sums in registers) + pair-per-thread EPN bundle kernel + row-per-thread far kernel for large
 * systems, all with the weights as uniform FFMA2 operands (kernel parameters); 1: pair-per-thread kernels everywhere
 * (incl. the per-atom kernel; slower, kept for A/B); 0: the round-1 warp-tile kernels (shared-memory operands).  All three
 * evaluate the same formulas in plain FP32; only the -- fixed -- order of the additions differs. */
int epnn_set_option(epnn_ctx* ctx, const char* key, double value);

/* Charge inference for a packed batch of systems, host buffers.
 * Replaces: the data-prep of charge_gn.gen_padded_init_state (charge_gn.py:292-366: featurise,
 *           get_init_edges, pad, mask) + model([h,e,x,q,mask]) (infer.py:32-35,73), for every system.
 *   n_sys          number of systems
 *   atom_offsets   int32[n_sys+1], atom_offsets[0] = 0; system s owns atoms [off[s], off[s+1])
 *   xyz            float32[3*n_atoms], Angstrom, AoS
 *   species        int32[n_atoms], index into the element table chosen by n_x
 *   Q              float32[n_sys], net charge of each system; q0 = float32(Q)/n per atom (charge_gn.py:337)
 *   npad           int32[n_sys] or NULL: the pad size N the reference's dense model would be built with
 *                  (charge_gn.py:340; results depend on it, SURVEY.md 3.3).  NULL = no padding (N = n).
 *   q_out          float32[n_atoms] predicted charges (real atoms only)
 *   q_out_f64      optional double[n_atoms] (NULL to skip): the charges before rounding to float32
 *   stats          optional */
int epnn_infer_batch(epnn_ctx* ctx, int64_t n_sys, const int32_t* atom_offsets, const float* xyz,
                     const int32_t* species, const float* Q, const int32_t* npad,
                     float* q_out, double* q_out_f64, epnn_stats* stats);

/* Same with DEVICE pointers for the bulk data (inputs already resident in HBM, outputs left in HBM).
 * atom_offsets and npad stay HOST arrays: they drive launch geometry and are tiny (4 B per system).
 * Work is enqueued on the ctx stream; the call returns after the stream has been synchronised. */
int epnn_infer_batch_dev(epnn_ctx* ctx, int64_t n_sys, const int32_t* atom_offsets_host,
                         const float* xyz_dev, const int32_t* species_dev, const float* Q_dev,
                         const int32_t* npad_host, float* q_out_dev, double* q_out_f64_dev, epnn_stats* stats);

/* Electrostatics of a packed batch of point charges, typically the charges epnn_infer_batch predicted.
 * (No counterpart in the reference, which stops at the charges; it loads the SSI dimer split <stem>splits.npy,
 *  charge_gn.py:305-308, but never uses it.)
 *
 * Let s be a system, atoms i, j in s, and r_ij = |x_i - x_j|.  Units are e and Angstrom; the C-ABI does no unit
 * conversion.  The optional `fragment` argument gives an int32 label per atom.  Only equality of labels within one
 * system matters.
 * A pair (i, j) is included when all three hold:
 *   - i != j;
 *   - r_ij > 0 (coincident atoms are skipped; they contribute nothing);
 *   - `fragment` is NULL, or fragment_i != fragment_j.
 * The outputs:
 *   - phi_i = sum_{j included} q_j / r_ij, the potential at atom i, in e/A.
 *   - E_s = 1/2 sum_{i in s} q_i phi_i = sum_{i<j included} q_i q_j / r_ij, in e^2/A.  With NULL fragments this is the
 *     Coulomb energy of the whole system.  With a dimer split it is the inter-monomer energy.
 *   - mu_s = sum_{i in s} q_i (x_i - c_s), where c_s is the unweighted centroid of the atoms of s, in e*A.  Fragments do
 *     not change mu.
 * Everything after loading the float32 coordinates is computed in FP64.  The float32 -> double conversion is exact.
 *
 *   atom_offsets   int32[n_sys+1] as in epnn_infer_batch (validated the same way)
 *   xyz            float32[3*n_atoms]
 *   q              double[n_atoms], the layout of q_out_f64 of epnn_infer_batch
 *   fragment       int32[n_atoms] or NULL
 *   energy_out     double[n_sys] or NULL;  dipole_out double[3*n_sys] (x, y, z per system) or NULL;
 *   phi_out        double[n_atoms] or NULL.  At least one output must be given.
 * Every sum has a fixed order and no result is accumulated with atomics: the outputs are bitwise repeatable, and a
 * system's outputs do not depend on which other systems share the call.  Runs on the ctx's GPU (a sharded ctx too). */
int epnn_electrostatics(epnn_ctx* ctx, int64_t n_sys, const int32_t* atom_offsets, const float* xyz,
                        const double* q, const int32_t* fragment, double* energy_out, double* dipole_out,
                        double* phi_out);

/* Same with DEVICE pointers: atom_offsets stays a HOST array as in epnn_infer_batch_dev, every other pointer is a DEVICE
 * pointer, so epnn_infer_batch_dev -> epnn_electrostatics_dev chains on the ctx stream with no host copy.  Work is
 * enqueued on the ctx stream; the call returns after the stream has been synchronised. */
int epnn_electrostatics_dev(epnn_ctx* ctx, int64_t n_sys, const int32_t* atom_offsets_host, const float* xyz_dev,
                            const double* q_dev, const int32_t* fragment_dev, double* energy_out_dev,
                            double* dipole_out_dev, double* phi_out_dev);

/* Electrostatic potential and field of a packed batch of point charges at arbitrary points: an ESP map on a grid, the
 * potential or field at given sites, or the field at the atoms themselves.
 *
 * Let s be a system with atoms j at positions x_j (float32, widened exactly to FP64) and charges q_j (FP64).  Let p be a
 * point of s (FP64, Angstrom) and r_pj = |p - x_j|.  Atoms with r_pj = 0 are skipped, as coincident atoms are in
 * epnn_electrostatics.
 *   - phi(p) = sum_j q_j / r_pj, in e/A.
 *   - E(p) = -grad phi(p) = sum_j q_j (p - x_j) / r_pj^3, in e/A^2.
 * Everything after the loads is FP64.  If the points of a system are its own atom coordinates, phi equals the phi_out of
 * epnn_electrostatics with NULL fragments (to rounding), and q_i E(x_i) is the Coulomb force on atom i at fixed charges.
 *
 *   atom_offsets   int32[n_sys+1] as in epnn_infer_batch (validated the same way)
 *   xyz            float32[3*n_atoms]
 *   q              double[n_atoms], the layout of q_out_f64 of epnn_infer_batch
 *   point_offsets  int64[n_sys+1]: system s owns the points [point_offsets[s], point_offsets[s+1]); point_offsets[0] = 0,
 *                  the offsets do not decrease (a system may have no points)
 *   points         double[3*n_points] (x, y, z per point); may be NULL only when there are no points
 *   phi_out        double[n_points] or NULL;  field_out double[3*n_points] (x, y, z per point) or NULL.
 *                  At least one output must be given.
 * No result is accumulated with atomics and every sum has a fixed order: the outputs at a point depend only on that
 * point, its system's atoms and charges, and the build -- not on the system's other points, the other systems, the
 * chunking of the call or the GPU's SM count.  Runs on the ctx's GPU (a sharded ctx too). */
int epnn_potential_points(epnn_ctx* ctx, int64_t n_sys, const int32_t* atom_offsets, const float* xyz, const double* q,
                          const int64_t* point_offsets, const double* points, double* phi_out, double* field_out);

/* Same with DEVICE pointers: atom_offsets and point_offsets stay HOST arrays, every other pointer is a DEVICE pointer, so
 * epnn_infer_batch_dev -> epnn_potential_points_dev chains on the ctx stream with no host copy.  Work is enqueued on the
 * ctx stream; the call returns after the stream has been synchronised. */
int epnn_potential_points_dev(epnn_ctx* ctx, int64_t n_sys, const int32_t* atom_offsets_host, const float* xyz_dev,
                              const double* q_dev, const int64_t* point_offsets_host, const double* points_dev,
                              double* phi_out_dev, double* field_out_dev);

/* Neighbour list only (for the bit-exactness check against the reference's is_near mask).
 * Replaces: get_init_edges + the is_near predicate (charge_gn.py:122-163, 90-94).
 *   which = 0: is_near set;  which = 1: the e != 0 set (i != j, D < 3.0).
 * rowptr: int32[n_atoms+1]; col: int32[col_capacity], GLOBAL atom indices, ascending within a row;
 * *nnz receives the number of entries (EPNN_E_CAPACITY if col_capacity is too small; *nnz is still set). */
int epnn_neighbors(epnn_ctx* ctx, int64_t n_sys, const int32_t* atom_offsets, const float* xyz,
                   int which, int32_t* rowptr, int32_t* col, int64_t col_capacity, int64_t* nnz);

/* Radial descriptors of one system, dense: e float32[n*n*48] exactly as get_init_edges returns them
 * (charge_gn.py:122-163).  Intended for tests and for the charge_gn.get_init_edges facade. */
int epnn_init_edges(epnn_ctx* ctx, int32_t n, const float* xyz, float* e_out);

/* Keras-shaped compatibility path: the model called on the dense padded tensors that
 * gen_padded_init_state produces.  Replaces model([h,e,x,q,mask]) (charge_gn.py:369-391) literally:
 * un-tiling by divide_no_nan, unmasked all-pairs GNN, EPN masked by mask*is_near(e).
 *   h float32[B][N][N][48], e float32[B][N][N][48], x float32[B][N][N][n_x], q float32[B][N][N][1],
 *   mask float32[B][N][N]; q_out float32[B][N] (the reference returns (B,N,1)). */
int epnn_infer_dense(epnn_ctx* ctx, int32_t B, int32_t N, const float* h, const float* e, const float* x,
                     const float* q, const float* mask, float* q_out);

/* Final GNN hidden state of the last epnn_infer_batch call (needs option keep_hidden=1 and a
 * single-chunk call): h_out float32[n_atoms*48].  Test hook: the shipped default checkpoint's GNN
 * output is a dead constant, so charges alone cannot validate the GNN kernels (SURVEY.md trap 6). */
int epnn_get_hidden(epnn_ctx* ctx, float* h_out, int64_t n_floats);

/* Host-side ingest of the reference's xyz dialect (no GPU involved): multi-threaded parse of a list of files into
 * the packed arrays epnn_infer_batch takes.  Replaces the Python parsing loop of charge_gn.gen_padded_init_state
 * (charge_gn.py:301-338): line 2 first token = Q (float32), atom lines "Elem x y z [ignored]", numbers parsed as
 * float64 and rounded once to float32 like numpy; element symbols index the table chosen by n_x.  The file ORDER is
 * the caller's (os.listdir order upstream, charge_gn.py:301).  On a malformed file / unknown element the call returns
 * EPNN_E_INVALID and the batch only carries the error (kind 1 cannot open, 2 malformed, 3 unknown element -- the
 * reference raises KeyError, charge_gn.py:326-327 -- plus the index of the first offending file and a message). */
typedef struct epnn_xyz_batch epnn_xyz_batch;
int epnn_xyz_load(const char* const* paths, int64_t n_files, int n_x, int threads, epnn_xyz_batch** out);
int epnn_xyz_parse_text(const char* text, size_t len, int n_x, epnn_xyz_batch** out);
int64_t epnn_xyz_n_systems(const epnn_xyz_batch* b);
int64_t epnn_xyz_n_atoms(const epnn_xyz_batch* b);
const int32_t* epnn_xyz_offsets(const epnn_xyz_batch* b);     /* int32[n_systems + 1] */
const float* epnn_xyz_coords(const epnn_xyz_batch* b);        /* float32[3 * n_atoms] */
const int32_t* epnn_xyz_species(const epnn_xyz_batch* b);     /* int32[n_atoms] */
const float* epnn_xyz_charges(const epnn_xyz_batch* b);       /* float32[n_systems] */
int epnn_xyz_error(const epnn_xyz_batch* b, int* kind, int* file_index);
const char* epnn_xyz_error_message(const epnn_xyz_batch* b);
void epnn_xyz_free(epnn_xyz_batch* b);

/* Pinned host memory helpers so that callers can make the H2D/D2H copies asynchronous. */
int epnn_host_alloc(void** ptr, size_t bytes);
int epnn_host_free(void* ptr);

/* Multi-GPU sharding of LARGE systems (n > 48 atoms; BASELINE config 5: one big system on several GPUs of one node).
 * (No counterpart in the reference: infer.py:62-73 is single-process, batch 1.)
 * One process per GPU; every rank is given the SAME epnn_infer_batch call.  The atom index space of a batch is cut into
 * `world` equal slices (epnn_shard_slice); a rank OWNS the rows of large systems that fall into its slice:
 *   - the neighbour list, the descriptors and the pair list are built for owned rows only (a pair cut by a slice boundary
 *     is held by both owners, always as (min, max));
 *   - per-atom kernels (update MLP, projections, charge reduction) run on owned rows; the electron-passing projections
 *     additionally on the near neighbours of owned rows;
 *   - the message-passing kernels (the exact all-pairs sum) run on owned rows against ALL columns;
 *   - exchanges, each one in-place ncclAllGather of equal slices on the ctx stream (NVLink / NVSwitch): v after every
 *     message-passing step but the last (128 B/atom), the update MLP's last hidden layer once (128 B/atom), the charges
 *     after every electron-passing pass (8 B/atom).  Cut pairs are evaluated by both owners in the same orientation, so
 *     no transfer is exchanged and charge conservation holds on every rank.
 * Small systems (n <= 48) of the same call are replicated on every rank.  Every row is computed by exactly the
 * arithmetic of a single-GPU run: the result is bit-identical to it, on every rank (each rank returns all charges).
 * NCCL is bound at run time (dlopen of libnccl.so.2: the copy already in the process, e.g. torch's, else the system's).
 *   epnn_shard_unique_id(id)             rank 0: a fresh 128-byte ncclUniqueId, to be handed to every rank by the caller
 *                                        (torch.distributed.broadcast in epnn_b200/shard.py, MPI_Bcast, a file, ...)
 *   epnn_shard_init(ctx, rank, world, id) collective over the `world` ranks: builds this ctx's communicator.
 *                                        world == 1 (id may be NULL) tears it down and switches sharding off.
 *   epnn_shard_slice(n, rank, world, &b, &e)  the rows [b, e) rank owns in a batch of n atoms (pure function)
 *   epnn_shard_stats(ctx, &calls, &bytes) all-gathers issued / bytes received by this rank since epnn_shard_init */
int epnn_shard_unique_id(void* id128);
int epnn_shard_init(epnn_ctx* ctx, int rank, int world, const void* id128);
int epnn_shard_slice(int64_t n_atoms, int rank, int world, int64_t* begin, int64_t* end);
int epnn_shard_stats(epnn_ctx* ctx, int64_t* calls, int64_t* bytes);

/* The CUDA stream (cudaStream_t, returned as void*) every kernel and copy of this ctx is enqueued on, so
 * that a caller can record its own CUDA events around a sequence of calls (bench.py does). */
int epnn_get_stream(epnn_ctx* ctx, void** stream_out);

/* Make the ctx enqueue on the CALLER's stream (a cudaStream_t passed as void*; must belong to the ctx's device and outlive
 * its use) -- what the `_dev` entry points need to be ordered after the producer of their inputs without a host sync.
 * NULL restores the ctx's own stream.  The call synchronises the stream in use before switching.  (The legacy default
 * stream, handle 0, cannot be selected: NULL means "own stream".) */
int epnn_set_stream(epnn_ctx* ctx, void* stream);

/* FP32 FMA micro-benchmark on the ctx device: the measured SIMT peak (TFLOP/s, 2 flops per FMA, best of
 * `repeats` launches timed with CUDA events) that the pair-MLP kernels' roofline fraction is quoted against
 * (MEASURED_PEAKS.json only holds HBM and tensor peaks; SURVEY.md 8d). */
int epnn_measure_fp32_peak(epnn_ctx* ctx, int repeats, double* tflops_out);

/* The 48 Gaussian centres mu_k = linspace(0.1, 3.0, 48) the kernels use (charge_gn.py:123). */
int epnn_rbf_centers(double* mu_out48);

/* Orthonormal basis B[48][16] (row-major) of the numerically rank-16 family of radial descriptors; the FP32 pair
 * kernels carry B^T e (16 coefficients) per pair instead of e (48 values): max |e - B B^T e| < 1e-9 for every D. */
int epnn_rbf_basis(double* B48x16);

/* Library / build identification, e.g. "epnn_b200 0.1.0 sm_100a". */
const char* epnn_version(void);

#ifdef __cplusplus
}
#endif
#endif /* EPNN_B200_H */
