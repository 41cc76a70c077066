/*
 * pgp.h -- C ABI of the B200-native PCS -> LCP -> TrICP hot path (libpgp.so).
 *
 * This is the drop-in boundary under the reference's hypothesis-generation stage.  Every entry
 * point cites the reference interface it replaces.  Paths are relative to the reference tree:
 *   S4  = src/3rdparty/super4pcs/src/super4pcs
 *   PPE = src/physim_pose_estimation
 *
 * Conventions
 *   - plain C types, caller-owned buffers, no exceptions cross the boundary;
 *   - every function returns PGP_OK (0) or a negative pgp_status; pgp_last_error() gives the text;
 *   - one context per GPU (one process per GPU); all work of a context is ordered on its stream;
 *   - transforms are ROW-MAJOR 3x4 fp32 in the CENTRED frame the reference scores in
 *     (Tr(-c_P) . T . Tr(c_Q), S4/algorithms/match4pcsBase.cc:1601-1610); pgp_pose_to_centred /
 *     pgp_centred_to_pose convert to and from camera-frame 4x4 poses exactly as
 *     match4pcsBase.cc:1474-1482 does;
 *   - "host" pointers are ordinary (ideally pinned) CPU memory, "dev" pointers are CUDA device
 *     memory of the context's device;
 *   - there is NO CPU fallback: without a CUDA device pgp_create fails.
 */
#ifndef PGP_H_
#define PGP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGP_API __attribute__((visibility("default")))

typedef struct pgp_ctx pgp_ctx;

typedef enum pgp_status {
  PGP_OK = 0,
  PGP_E_INVALID = -1,      /* bad argument */
  PGP_E_CUDA = -2,         /* CUDA runtime error (text in pgp_last_error) */
  PGP_E_NO_SCENE = -3,     /* pgp_set_scene has not been called */
  PGP_E_NO_MODEL = -4,     /* pgp_set_model has not been called for this object */
  PGP_E_NO_SCORES = -5,    /* top-k / chain requested before any scoring call */
  PGP_E_TOO_LARGE = -6,    /* scene extent / delta needs more grid cells than PGP_MAX_CELLS */
  PGP_E_NOMEM = -7,
  PGP_E_CAPACITY = -8,     /* an output list overflowed the capacity the caller gave */
  PGP_E_COMM = -9          /* NCCL could not be loaded or a collective failed (text in pgp_last_error) */
} pgp_status;

/* LCP scoring modes: which reference function a scoring call reproduces. */
typedef enum pgp_lcp_mode {
  PGP_LCP_COUNT = 0,       /* Match4PCSBase::Verify          S4/algorithms/match4pcsBase.cc:1699-1731 */
  PGP_LCP_WEIGHTED = 1     /* Match4PCSBase::WeightedVerify  S4/algorithms/match4pcsBase.cc:1733-1766 */
} pgp_lcp_mode;

/* One scored hypothesis as it leaves the device (64 bytes; the record the multi-GPU merge moves). */
typedef struct pgp_hyp {
  int64_t index;    /* generation index (global, i.e. including the rank's index_base) */
  uint32_t count;   /* COUNT: inlier count;  WEIGHTED: number of gated in-range points */
  float score;      /* what the reference stores in allPose[i].second: count/|Qval| or sum(prior)/|Qval| */
  float T[12];      /* centred-frame row-major 3x4 */
} pgp_hyp;

/* Options of the congruent-set generator (Match4PCSOptions, S4/shared4pcs.h:146-174, as set by
 * S4/super4pcs_test.cc:91-99, plus the compile-time caps of match4pcsBase.cc:290-291,1858). */
typedef struct pgp_pcs_opts {
  int n_bases;               /* max_number_of_bases_ = 100            match4pcsBase.cc:290  */
  int max_quads_per_base;    /* max_sampled_csets  = 100              match4pcsBase.cc:1858; <=0: keep all */
  float max_base_diameter;   /* <=0: estimate like init(), match4pcsBase.cc:274-283 */
  float overlap;             /* overlap_estimation (only scales the wide-base target), default 0.5 */
  int base_trials;           /* kNumberOfDiameterTrials = 1000 random triangles per base, :377-410 */
  int mode;                  /* operMode (match4pcsBase.cc:300): 0 = wide random base + Super4PCS pair extraction (default here),
                                1 = StoCS base sampling + PPF-map pair lookup (what the reference ships; needs a PPF map),
                                2 = V4PCS: tetrahedron base (SelectTetrahedronBase :466-503) + six-distance join (:978-1044) */
} pgp_pcs_opts;

/* ---------------------------------------------------------------- context ------------------ */

/* One context drives ONE GPU.  Several GPUs: one context per GPU, joined by the communicator calls of the multi-GPU section
 * below (one process per GPU), or pgp_group_create (one process, n devices) -- SURVEY.md 8(b) `pgp_create(n_devices, ids)`.
 * Creates a context on CUDA device `device`.  Returns NULL when no CUDA device is usable (there
 * is no CPU path).  Replaces the construction of match_4pcs::MatchSuper4PCS
 * (S4/super4pcs_test.cc:100, S4/algorithms/super4pcs.cc:70-73). */
PGP_API pgp_ctx* pgp_create(int device);
PGP_API void pgp_destroy(pgp_ctx* ctx);
PGP_API const char* pgp_last_error(const pgp_ctx* ctx);   /* ctx may be NULL: error of pgp_create */
PGP_API const char* pgp_version(void);
/* Makes later calls of this context run on an externally owned cudaStream_t (e.g. the caller's
 * current stream).  NULL restores the context's own stream. */
PGP_API int pgp_set_stream(pgp_ctx* ctx, void* cuda_stream);
PGP_API int pgp_synchronize(pgp_ctx* ctx);

/* ---------------------------------------------------------------- K1: scene ---------------- */

/* Scene segment "P": centring + kd-tree of Match4PCSBase::init (match4pcsBase.cc:242-270) and
 * initKdTree (:1046-1056 -> S4/accelerators/kdtree.h:355-370).  xyz: n x 3 camera-frame metres;
 * nrm: n x 3 or NULL (normalised like Point3D::set_normal, S4/shared4pcs.h:85-87; |n|^2 < 0.01
 * -> zero, S4/utils/geometry.h:56-82).  Builds the delta-cell voxel grid on the device (K1).
 * Priors default to 1.0. */
PGP_API int pgp_set_scene(pgp_ctx* ctx, const float* xyz_host, const float* nrm_host, int n, float delta);

/* Per-scene-point prior from the probability image (match4pcsBase.cc:317-340): value/10000 at the
 * pin-hole projection of the un-centred point through K (row-major 3x3).  img: rows x cols uint16.
 * (The reference indexes the image unchecked; here row/col are clamped into the image.) */
PGP_API int pgp_set_scene_prior_image(pgp_ctx* ctx, const uint16_t* img_host, int rows, int cols, const float* K9);
/* Or hand the priors over directly (orig_probabilities_, one per scene point).  Any finite value is accepted, negative ones too:
 * a weighted score is then the exact ordered sum and may be negative, and selection orders it as an fp32 value (a score <= 0
 * never enters the improving chain).  A NaN or infinite prior is refused with PGP_E_INVALID and the previous priors stay. */
PGP_API int pgp_set_scene_priors(pgp_ctx* ctx, const float* prior_host);
PGP_API int pgp_get_scene_priors(pgp_ctx* ctx, float* prior_host);

/* Model clouds of object slot `obj` (0..PGP_MAX_OBJECTS-1): "Q" = search sampling
 * (model_search.ply), "Q_validation" = validation sampling (model_validation.ply); both centred
 * on the centroid of the SEARCH cloud (match4pcsBase.cc:248-261). */
PGP_API int pgp_set_model(pgp_ctx* ctx, int obj, const float* search_xyz, const float* search_nrm, int nq,
                          const float* val_xyz, const float* val_nrm, int nv);

PGP_API int pgp_get_centroids(pgp_ctx* ctx, int obj, float* cP3, float* cQ3);
/* camera-frame pose (row-major 4x4 double) <-> centred row-major 3x4 float. */
PGP_API int pgp_pose_to_centred(pgp_ctx* ctx, int obj, const double* pose16, float* T12);
PGP_API int pgp_centred_to_pose(pgp_ctx* ctx, int obj, const float* T12, double* pose16);

/* Grid facts for reports: dims[3], number of cells, occupied cells, cell size, bytes of the grid. */
PGP_API int pgp_grid_info(pgp_ctx* ctx, int* dims3, int64_t* n_cells, int64_t* n_occupied, float* cell, int64_t* bytes);

/* Statistics of the tri-state label structure K1b builds over the grid (no reference counterpart; reports and
 * tuning): out8 = {cells whose 512 sub-voxels are all OUT, all IN, mixed; sub-voxels OUT, IN, AMBIG; overflow
 * records of the AMBIG candidate lists (candidates beyond the two each AMBIG voxel keeps inline); entries of the
 * nearest-candidate lists (0 until a WEIGHTED call built them)}. */
PGP_API int pgp_label_stats(pgp_ctx* ctx, int64_t* out8);

/* ---------------------------------------------------------------- K3: LCP scoring ---------- */

/* Scores n hypotheses (verifyRigidTransform, match4pcsBase.cc:1490-1502, over the loop at
 * :1888-1901).  T_host: n x 12.  counts_host / scores_host may be NULL.  Copies in, scores,
 * copies out, and returns after the results are on the host.  The batch stays resident on the
 * device for pgp_topk / pgp_improving_chain. */
PGP_API int pgp_score_lcp(pgp_ctx* ctx, int obj, const float* T_host, int64_t n, int mode,
                          uint32_t* counts_host, float* scores_host);
/* The same call in two halves, for callers that want to queue the selection (pgp_topk_dev) and their collective behind the
 * scoring launch before waiting: _begin enqueues upload + scoring + the downloads (T_host and the two output buffers should be
 * pinned and must stay valid until _end) and returns at once; _end waits until counts_host / scores_host are filled.  _end
 * returns 1 (not an error) in the one case where the batch had to be scored a second time -- the upload that is streamed under
 * the scoring launch stalled (a profiler serialising streams) -- and work queued in between must be repeated; 0 otherwise.
 * One batch at a time per context.  Replaces the same loop of the reference as pgp_score_lcp (match4pcsBase.cc:1888-1901). */
PGP_API int pgp_score_lcp_begin(pgp_ctx* ctx, int obj, const float* T_host, int64_t n, int mode,
                                uint32_t* counts_host, float* scores_host);
PGP_API int pgp_score_lcp_end(pgp_ctx* ctx);
/* Same with everything already in device memory; asynchronous on the context's stream.
 * counts_dev (n x u32) and scores_dev (n x f32) are caller-owned and must stay alive until the
 * top-k / chain calls that follow. */
PGP_API int pgp_score_lcp_dev(pgp_ctx* ctx, int obj, const float* T_dev, int64_t n, int mode,
                              uint32_t* counts_dev, float* scores_dev);
/* Scene indices matched by ONE pose in WEIGHTED mode, in model-point order (the
 * registered_indices of match4pcsBase.cc:1760,1894; registered_points of
 * PPE/src/hypothesis_generation/ObjectPoseCandidateSet.hpp:8-22).  Returns the number written. */
PGP_API int pgp_registered_points(pgp_ctx* ctx, int obj, const float* T12_host, int32_t* idx_host, int cap);
/* Nearest in-range scene index (or -1) of every transformed validation point for one pose:
 * KdTree::doQueryRestrictedClosestIndex (S4/accelerators/kdtree.h:394-459) per point. */
PGP_API int pgp_nearest_in_range(pgp_ctx* ctx, int obj, const float* T12_host, int32_t* idx_host);

/* Tuning / test switches (no counterpart in the reference; none of them changes a result):
 *   "force_coarse" = 1      score on the plain 27-cell path even when the fine tri-state grid exists (cross-check in the tests)
 *   "group_cull" = 0        do not skip the 32-point model groups whose bounding sphere cannot reach the scene (cross-check)
 *   "tail_split" = 1..16    model chunks per hypothesis in the last wave of the persistent scoring grid (default 4)
 *   "stream_upload" = 0     pgp_score_lcp uploads the whole batch before the scoring launch (use under profilers, which
 *                           serialise streams) */
PGP_API int pgp_set_option(pgp_ctx* ctx, const char* name, int value);
/* Number of my kernels launched by this context so far (bench.py's gpu_launches). */
PGP_API int64_t pgp_launch_count(const pgp_ctx* ctx);

/* ---------------------------------------------------------------- K4: selection ------------ */

/* Top-k of the last scored batch, ordered by (score desc, index asc); replaces the serial
 * best-so-far scan of Perform_N_steps (match4pcsBase.cc:1888-1901).  index_base is added to the
 * local indices (the rank's offset when hypotheses are sharded).  Returns the number written.
 * On a context that belongs to a communicator (pgp_comm_init, world > 1) the call is COLLECTIVE: every rank calls it, K4 runs on
 * every rank's shard, the per-rank records are all-gathered over NCCL and merged, and every rank receives the same global top-k
 * -- identical to the single-GPU answer on the concatenated batch.  index_base = PGP_INDEX_AUTO numbers the hypotheses rank after
 * rank (rank r's first index = the batch sizes of ranks < r, which travel in the same all-gather). */
PGP_API int pgp_topk(pgp_ctx* ctx, int obj, int k, int64_t index_base, pgp_hyp* out_host);
#define PGP_INDEX_AUTO (-1ll)
/* The same in two halves, so that the collective never sits on the scoring stream: _begin enqueues K4 on the context's stream
 * and -- behind an event, on the context's own exchange stream -- the all-gather and the download of the gathered records, and
 * returns a ticket (>= 0) at once; the next batch can be scored while the exchange is in flight.  _end waits for the ticket and
 * merges on the host (k records at most; returns the number written).  Up to 8 tickets may be in flight per context.  Works
 * without a communicator too (then it is the local top-k). */
PGP_API int pgp_topk_begin(pgp_ctx* ctx, int obj, int k, int64_t index_base);
PGP_API int pgp_topk_end(pgp_ctx* ctx, int ticket, pgp_hyp* out_host);
/* Makes the context's stream wait until the ticket's exchange has delivered its records to the host buffer (lets a caller time
 * the exchange with events on its own stream; not needed for correctness). */
PGP_API int pgp_topk_stream_wait(pgp_ctx* ctx, int ticket);
/* Same, asynchronous, with the k records written straight into caller-owned DEVICE memory (the
 * send buffer of the multi-GPU all-gather); slots beyond the batch size get index = -1.  Always local:
 * PGP_INDEX_AUTO means base 0. */
PGP_API int pgp_topk_dev(pgp_ctx* ctx, int obj, int k, int64_t index_base, pgp_hyp* out_dev);
/* Deterministic merge of per-rank top-k lists (n_lists x k_each records, e.g. the output of an
 * all-gather): same order as pgp_topk on the union.  Host-side, no context needed. */
PGP_API int pgp_topk_merge(const pgp_hyp* lists, int n_lists, int k_each, int k, pgp_hyp* out);
/* The strictly-improving chain in generation order that Perform_N_steps returns as
 * hypothesisSet (match4pcsBase.cc:1888-1914); its last element is bestHypothesis.
 * Returns the chain length (<= cap) or PGP_E_CAPACITY: for a chain of at most 4096 elements out_host then holds its last cap
 * elements; a longer chain leaves out_host unusable.  Collective on a communicator context, like pgp_topk: the chain over the
 * ranks' batches in rank order (each rank may contribute at most PGP_CHAIN_EXCHANGE_CAP elements). */
PGP_API int pgp_improving_chain(pgp_ctx* ctx, int obj, int64_t index_base, pgp_hyp* out_host, int cap);

/* ---------------------------------------------------------------- K4d: pose-distinct candidates */

/* Greedy non-maximum suppression in pose space: which hypotheses of an object become MCTS candidates when many of the best ones
 * are the same placement with millimetre and sub-degree jitter (congruent sets of different bases agree, LCP is smooth in the
 * pose).  No live reference counterpart: the reference's pose-space clustering (greedyClustering) is commented out
 * (PPE/src/hypothesis_generation/HypothesisSelection.cpp:161) and its only CUDA kernel is a box NMS.  RESTATED, exact contract
 * (oracle/select_port.py restates it in float64):
 *
 *  Pool: m records (pgp_hyp) of one object, 1 <= m <= 4096, processed in the order given (pgp_topk's order is what callers pass).
 *    Records with index < 0 (pgp_topk_dev's padding) are skipped: they neither keep nor suppress.
 *  Greedy rule: record i is kept iff no earlier KEPT record suppresses it; the walk stops once k records are kept.  Kept records
 *    keep their pool order and are copied bit for bit.
 *  A kept record a suppresses a later record b when both tests pass, every step in double from the fp32 entries of the centred
 *  row-major 3x4 T, each operation rounded on its own (no FMA):
 *    translation: dx = (double)a.T[3] - (double)b.T[3], dy (entries 7), dz (entries 11); d2 = (dx*dx + dy*dy) + dz*dz;
 *      passes when d2 <= max_dist * max_dist (one rounded product).  In the centred frame this is the distance between the
 *      points where the model's search centroid lands.
 *    rotation: for S in {I} and the object's symmetries, G = R_b S entry by entry ((R_b[r][0] S[0][c] + R_b[r][1] S[1][c]) +
 *      R_b[r][2] S[2][c]) (for S = I, G = R_b promoted to double; the identity is not multiplied in); tr = sum R_a[r][c] G[r][c]
 *      left to right in row-major order; passes when tr >= 1.0 + 2.0 * cos_angle for some S.
 *  NaN follows the IEEE comparisons: a record with a NaN entry in T never suppresses and is never suppressed (it is kept when
 *  reached, and suppresses nothing).
 *  Camera-frame output row j = pgp_centred_to_pose(obj, kept[j].T), bitwise (same double expression and order). */
#define PGP_MAX_SYMMETRIES 23
/* Discrete symmetries of model slot obj: n row-major 3x3 rotations R9 (n x 9 doubles) in the centred model frame; the identity is
 * implied.  n = 0 clears the set.  A property of the model, like pgp_set_mesh: pgp_set_model leaves it alone.  The matrices need not
 * be orthonormal (the contract is the arithmetic above).  PGP_E_INVALID: obj out of range, n < 0 or n > PGP_MAX_SYMMETRIES, a
 * NULL R9 with n > 0, a non-finite entry. */
PGP_API int pgp_set_symmetries(pgp_ctx* ctx, int obj, const double* R9, int n);
/* Many pools at once on device data, asynchronous on the context's stream, in two launches whatever n_lists is.  On the host:
 * objs (n_lists model slots), pool_offsets (n_lists + 1, non-decreasing from 0, each list 1 .. 4096 records) and k (1 .. 4096), so
 * every launch size is known and nothing is read back.  In device memory (of the context's device, or managed):
 *   pool_dev  the concatenated pools (pool_offsets[n_lists] records);
 *   out_dev   n_lists x k records: list l's kept records at l x k, the slots after them index = -1 and zero elsewhere (as pgp_topk_dev pads);
 *   poses16_dev (NULL allowed) n_lists x k row-major 4x4 doubles, the kept records' camera-frame poses, the rows after them the
 *     identity: with pose_offsets = {0, k, 2k, ...} they go straight to pgp_refine_batch_dev (a padding row is finite, refines to
 *     something finite and is ignored by its record's index);
 *   n_kept_dev (NULL allowed) one int32 per list.
 * The call returns once the work is queued; once the context's scratch has grown to the call's size (one 2 MB suppression mask per
 * 4096-pool) it makes no host synchronisation.  Returned at once with nothing queued and every output untouched: n_lists < 0, bad
 * offsets or list sizes, k outside 1 .. 4096, max_dist not finite or < 0, cos_angle NaN, a NULL objs / pool_dev / out_dev with
 * lists, an obj out of range (PGP_E_INVALID) or without a model (PGP_E_NO_MODEL), no scene when poses16_dev is requested
 * (PGP_E_NO_SCENE), a device argument that is not device or managed memory of the context's device.  No value is refused on the
 * device (there is no status word).  n_lists = 0 is a no-op. */
PGP_API int pgp_distinct_dev(pgp_ctx* ctx, const int32_t* objs, const int64_t* pool_offsets, int n_lists, const pgp_hyp* pool_dev, int k,
                             double max_dist, double cos_angle, pgp_hyp* out_dev, double* poses16_dev, int32_t* n_kept_dev);
/* The host convenience: the pool is pgp_topk(obj, m, PGP_INDEX_AUTO), K4d runs on it, out_host (room for k records) receives the
 * kept ones; returns their number.  On a communicator context the call is COLLECTIVE because pgp_topk is: every rank selects from
 * the same merged pool, so the answer does not depend on the number of GPUs (greedy suppression over the global top m depends on
 * that list alone).  PGP_E_INVALID: m or k outside 1 .. 4096, max_dist not finite or < 0, cos_angle NaN, out_host NULL; the
 * refusals of pgp_topk. */
PGP_API int pgp_topk_distinct(pgp_ctx* ctx, int obj, int m, int k, double max_dist, double cos_angle, pgp_hyp* out_host);

/* ---------------------------------------------------------------- K2: PCS generation ------- */

PGP_API void pgp_pcs_default_opts(pgp_pcs_opts* o);
/* All ordered pairs (i,j),(j,i) of the centred SEARCH model with | |q_i - q_j| - dist | <= eps:
 * MatchSuper4PCS::ExtractPairs (S4/algorithms/super4pcs.cc:193-236) with the shipped options,
 * i.e. the filter of S4/pairCreationFunctor.h:167-253 / brute-force spec S4/algorithms/4pcs.cc:109-192.
 * pairs_host: cap x 2 int32 (may be NULL to only count).  Returns the number of ordered pairs
 * through *n_pairs (which may exceed cap; only cap are written). */
PGP_API int pgp_extract_pairs(pgp_ctx* ctx, int obj, float dist, float eps, int32_t* pairs_host, int64_t cap, int64_t* n_pairs);
/* Congruent quads for one base (scene ids b[4], invariants inv1/inv2): the join of
 * MatchSuper4PCS::FindCongruentQuadrilaterals (S4/algorithms/super4pcs.cc:78-187).
 * pairs1/pairs2: ordered model pairs for base edges (b0,b1) and (b2,b3). quads_host: cap x 4. */
PGP_API int pgp_find_quads(pgp_ctx* ctx, int obj, const int32_t* base4, float inv1, float inv2, float eps,
                           const int32_t* pairs1_host, int64_t n1, const int32_t* pairs2_host, int64_t n2,
                           int32_t* quads_host, int64_t cap, int64_t* n_quads);
/* Congruent quads for one base in operMode 2 (V4PCS): ExtractCongruentSet (match4pcsBase.cc:1929-2039) with its six
 * ExtractPairs calls and FindCongruentQuadrilateralsV4PCS (:978-1044) -- every ordered 4-tuple of search-cloud points whose
 * six pairwise distances match the base's within eps (the pair filter of S4/pairCreationFunctor.h:167-253).  base4: scene
 * ids.  quads_host: cap x 4, sorted by (v1, v2, v3, v4) (the reference's order is an unordered_set iteration: compare as sets). */
PGP_API int pgp_find_quads_v4pcs(pgp_ctx* ctx, int obj, const int32_t* base4, float eps, int32_t* quads_host, int64_t cap, int64_t* n_quads);
/* Rigid transform of one (base, quad): ComputeRigidTransformFromCongruentPair
 * (match4pcsBase.cc:1411-1488) + ComputeRigidTransformation (:1504-1614).  n quads of the same
 * base; T_host: n x 12 centred; ok_host: n flags (0 = rejected: degenerate or non-orthogonal). */
PGP_API int pgp_rigid_from_quads(pgp_ctx* ctx, int obj, const int32_t* base4, const int32_t* quads_host, int64_t n,
                                 float* T_host, uint8_t* ok_host);
/* Full device-side generator: bases from the scene (SelectQuadrilateral, match4pcsBase.cc:507-580),
 * pairs, quads, transforms -- written straight into the device buffer that pgp_score_generated
 * scores, no host round trip.  Returns the number of hypotheses generated through *n_hyp. */
PGP_API int pgp_generate_pcs(pgp_ctx* ctx, int obj, const pgp_pcs_opts* opts, uint64_t seed, int64_t max_hyp, int64_t* n_hyp);
/* The same for bases [base_lo, base_hi) of the opts->n_bases the request draws -- the unit bases shard by across GPUs (per-base
 * independence of Perform_N_steps, match4pcsBase.cc:1855-1877).  Every random draw is keyed by (seed, GLOBAL base index), so the
 * hypotheses of a base do not depend on which GPU generates it. */
PGP_API int pgp_generate_pcs_range(pgp_ctx* ctx, int obj, const pgp_pcs_opts* opts, uint64_t seed, int base_lo, int base_hi, int64_t max_hyp,
                                   int64_t* n_hyp);
/* Scores the hypotheses pgp_generate_pcs left on the device. */
PGP_API int pgp_score_generated(pgp_ctx* ctx, int obj, int mode);
/* Copies generated transforms / their scores to the host (n x 12, n). */
PGP_API int pgp_get_generated(pgp_ctx* ctx, int obj, float* T_host, uint32_t* counts_host, float* scores_host, int64_t cap);

/* PPF map of object `obj`'s SEARCH cloud (the PPFMap argument of getProbableTransformsSuper4PCS, S4/super4pcs_test.cc:39-43,
 * loaded from PPFMap.txt by Objects::readPPFMap, PPE/src/data_layer/Objects.cpp:31-49): n_keys rows, row k = key
 * keys4[4k..4k+3] (computePPF bins, match4pcsBase.cc:582-598) -> pairs[2 offsets[k] .. 2 offsets[k+1]) of search-cloud
 * indices.  Call after pgp_set_model. */
PGP_API int pgp_set_ppf_map(pgp_ctx* ctx, int obj, const int32_t* keys4, const int64_t* offsets, const int32_t* pairs, int64_t n_keys);
/* Builds that map on the device from the search cloud itself (all ordered pairs i != j) -- the offline generator the
 * reference does not ship -- and installs it. */
PGP_API int pgp_build_ppf_map(pgp_ctx* ctx, int obj);
/* Copies the installed map out (any pointer may be NULL); *n_keys / *n_pairs receive the sizes.  Rows are in key order. */
PGP_API int pgp_get_ppf_map(pgp_ctx* ctx, int obj, int32_t* keys4, int64_t cap_keys, int64_t* offsets, int32_t* pairs, int64_t cap_pairs,
                            int64_t* n_keys, int64_t* n_pairs);
/* computePPF (match4pcsBase.cc:582-598) of n scene index pairs: keys4 n x 4.  Parity hook. */
PGP_API int pgp_scene_ppf_keys(pgp_ctx* ctx, const int32_t* pairs, int64_t n, int32_t* keys4);
/* The engine seed the StoCS sampler gives std::default_random_engine for base `base`, attempt `attempt` of a generation
 * seeded with `seed` (the reference seeds from the wall clock, match4pcsBase.cc:611). */
PGP_API uint32_t pgp_stocs_engine_seed(uint64_t seed, int base, int attempt);

/* The bases the last pgp_generate_pcs call drew from the scene (baseSet of Perform_N_steps, match4pcsBase.cc:1838-1853):
 * ids cap x 4 scene indices in the pairing TryQuadrilateral chose (:415-464), inv cap x 2 invariants, ok cap flags
 * (0 = no admissible base was found for that draw).  Returns the number of bases written. */
PGP_API int pgp_get_bases(pgp_ctx* ctx, int obj, int32_t* ids, float* inv, uint8_t* ok, int cap);

/* ---------------------------------------------------------------- multi-GPU (SURVEY.md 8e) - */

/* Hypotheses (pgp_score_lcp* with a rank-specific index_base) or bases (pgp_generate_pcs_range) shard across the GPUs of one
 * box; scene grid and models are replicated (every rank makes the same pgp_set_scene / pgp_set_model calls); the only exchange
 * on the path is the all-gather of the selection records inside pgp_topk / pgp_improving_chain.  The reference is one thread
 * (match4pcsBase.cc:1855-1877 per base, :1888-1901 per hypothesis, PPE/src/data_layer/SceneCfg.cpp:379-390 per object): these
 * calls have no counterpart there; they keep its results.  NCCL is loaded with dlopen on first use.
 *
 * One process per GPU: rank 0 calls pgp_comm_unique_id, the PGP_COMM_ID_BYTES bytes reach the other ranks over any host channel,
 * then every rank calls pgp_comm_init (collective; ncclCommInitRank on the context's device). */
#define PGP_COMM_ID_BYTES 128
#define PGP_CHAIN_EXCHANGE_CAP 255
PGP_API int pgp_comm_unique_id(void* id128);
PGP_API int pgp_comm_init(pgp_ctx* ctx, const void* id128, int rank, int world);
/* One process, n contexts on n different devices (ncclCommInitAll); ctxs[i] becomes rank i. */
PGP_API int pgp_comm_init_all(pgp_ctx** ctxs, int n);
PGP_API int pgp_comm_rank(const pgp_ctx* ctx);
PGP_API int pgp_comm_world(const pgp_ctx* ctx);
PGP_API int pgp_comm_destroy(pgp_ctx* ctx);
/* After pgp_generate_pcs_range on every rank (collective): exchanges the per-rank hypothesis counts, applies the request's global
 * cap max_hyp in rank order (<= 0: no cap) -- the cut pgp_generate_pcs makes on one GPU -- and reports the global index of this
 * rank's first hypothesis and the global total (either pointer may be NULL). */
PGP_API int pgp_comm_sync_generated(pgp_ctx* ctx, int obj, int64_t max_hyp, int64_t* index_base, int64_t* n_total);
/* The cut pgp_comm_sync_generated applies, as a pure host function (no context, no GPU): counts[r] = hypotheses rank r generated;
 * on return *keep = how many of its own this rank keeps under the global cap max_hyp (<= 0: no cap), *index_base = global index of
 * its first hypothesis, *n_total = hypotheses of the whole request.  Same prefix the single-GPU generator keeps
 * (S4/algorithms/match4pcsBase.cc:1855-1877 appends base by base). */
PGP_API int pgp_generated_cap_split(const int64_t* counts, int world, int64_t max_hyp, int rank, int64_t* keep, int64_t* index_base, int64_t* n_total);

/* The merge behind the collective pgp_topk / pgp_improving_chain, as a pure host function (no context): `wire` = world blocks of
 * (k + 1) records as the all-gather delivers them -- per rank a header {index = the rank's batch size, count = valid records}
 * and k records.  kind 0: global top-k by (score desc, index asc); kind 1: the strictly improving chain over the ranks in order
 * (mode = the pgp_lcp_mode the batch was scored in).  auto_base != 0: records carry shard-local indices (PGP_INDEX_AUTO).
 * Returns the number of records written (<= cap) or PGP_E_CAPACITY. */
PGP_API int pgp_exchange_merge(const pgp_hyp* wire, int world, int k, int kind, int mode, int auto_base, pgp_hyp* out, int cap);

/* One process, n devices: a group owns one context per device and a communicator over them.  Replicated state is set on every
 * device, work is sharded, results are merged -- the calls below mirror their single-context namesakes.  (What SURVEY.md 8(b)
 * sketches as pgp_create(n_devices, device_ids).) */
typedef struct pgp_group pgp_group;
PGP_API pgp_group* pgp_group_create(int n_devices, const int* device_ids /* NULL: 0 .. n-1 */);
PGP_API void pgp_group_destroy(pgp_group* g);
PGP_API int pgp_group_size(const pgp_group* g);
PGP_API pgp_ctx* pgp_group_ctx(pgp_group* g, int i);          /* device i's context, for the per-device calls (pgp_registered_points ...) */
PGP_API const char* pgp_group_last_error(const pgp_group* g);
PGP_API int pgp_group_set_scene(pgp_group* g, const float* xyz_host, const float* nrm_host, int n, float delta);
PGP_API int pgp_group_set_scene_prior_image(pgp_group* g, const uint16_t* img_host, int rows, int cols, const float* K9);
PGP_API int pgp_group_set_scene_priors(pgp_group* g, const float* prior_host);
PGP_API int pgp_group_set_model(pgp_group* g, int obj, const float* search_xyz, const float* search_nrm, int nq, const float* val_xyz,
                                const float* val_nrm, int nv);
PGP_API int pgp_group_set_ppf_map(pgp_group* g, int obj, const int32_t* keys4, const int64_t* offsets, const int32_t* pairs, int64_t n_keys);
PGP_API int pgp_group_build_ppf_map(pgp_group* g, int obj);
/* bases split across the devices: device i generates -- and pgp_group_score_generated scores -- bases [i B / n, (i+1) B / n) */
PGP_API int pgp_group_generate_pcs(pgp_group* g, int obj, const pgp_pcs_opts* opts, uint64_t seed, int64_t max_hyp, int64_t* n_hyp);
PGP_API int pgp_group_score_generated(pgp_group* g, int obj, int mode);
/* hypotheses split across the devices: device i scores [i n / n_dev, (i+1) n / n_dev) */
PGP_API int pgp_group_score_lcp(pgp_group* g, int obj, const float* T_host, int64_t n, int mode, uint32_t* counts_host, float* scores_host);
/* K4 on every device -> one grouped ncclAllGather -> merge: the global answers, independent of the device count */
PGP_API int pgp_group_topk(pgp_group* g, int obj, int k, pgp_hyp* out_host);
PGP_API int pgp_group_improving_chain(pgp_group* g, int obj, pgp_hyp* out_host, int cap);
/* pgp_set_symmetries on every device; pgp_topk_distinct over pgp_group_topk's merged pool (run on device 0): the same answer as one
 * context on the concatenated batch. */
PGP_API int pgp_group_set_symmetries(pgp_group* g, int obj, const double* R9, int n);
PGP_API int pgp_group_topk_distinct(pgp_group* g, int obj, int m, int k, double max_dist, double cos_angle, pgp_hyp* out_host);

/* Random 32-byte-sector gather micro-benchmark (SURVEY.md 8d: the denominator of K3's moved-bytes roofline): every thread chases
 * `loads_per_thread` pseudo-random 32-byte sectors of a `footprint_bytes` buffer (L2-resident when below ~100 MB), four
 * independent chains per thread.  Returns the sustained sector traffic in GB/s through *gbps.  No reference counterpart. */
PGP_API int pgp_bench_sector_gather(pgp_ctx* ctx, int64_t footprint_bytes, int loads_per_thread, float* gbps);

/* ---- host-callable copies of two exact-arithmetic helpers of the kernels (no GPU needed; tests/test_host_arithmetic.py) ---------
 * pgp_host_chain_sum_equal: the float chain acc = c; (m - 1) x acc = fl(acc + c) -- std::accumulate over m equal weights in
 * SelectQuadrilateralStoCS's normalisation (S4/algorithms/match4pcsBase.cc:652-657) -- in O(binades) steps, bit-identical to the chain.
 * pgp_host_max_eigvec4: eigenvector of the largest eigenvalue of the symmetric 4x4 matrix of Horn's quaternion fit (the rigid fit
 * of trimmed ICP, replaces PCL's TrimmedICP -> SVD) from its characteristic polynomial; 0 = nearly double top eigenvalue, the kernel
 * then diagonalises with Jacobi. */
PGP_API float pgp_host_chain_sum_equal(float c, long long m);
PGP_API int pgp_host_max_eigvec4(const double* N16_rowmajor, double* q4);
/* pgp_host_solve_plane6: x6 = H^+ g6, the truncated, scaled pseudo-inverse solve of pgp_tricp_plane's fit (H36 row-major,
 * symmetric positive semi-definite); returns the number of eigenvalues kept. */
PGP_API int pgp_host_solve_plane6(const double* H36_rowmajor, const double* g6, double* x6);

/* ---------------------------------------------------------------- K5: trimmed ICP ---------- */

/* Trimmed ICP of k poses of object `obj` against the segment (source) with the model's
 * VALIDATION cloud as target: UCTState::performTrICP (PPE/src/hypothesis_verification/mcts/
 * UCTState.cpp:121-204) / utilities::performTrICP (PPE/src/misc/utilities.cpp:651-680) ->
 * pcl::recognition::TrimmedICP::align.  poses: k x 16 doubles, row-major camera-frame
 * model->scene poses, refined in place.  seg_xyz: ns x 3 camera frame.  trim: kept fraction
 * (0.5 at the MCTS call site), ratio: new-to-old energy ratio (0.99), max_iter: safety cap
 * (values below 1 act as 1).  iters_out / energy_out (k each) may be NULL.
 * PGP_E_INVALID, before anything runs and with the poses untouched: trim or ratio not > 0 (NaN
 * included), a NaN or infinite segment coordinate or pose entry.  k = 0 is a no-op.
 * n_keep = min(ns, (int)|trim * ns|) in fp32; n_keep < 3 leaves every pose as given with
 * iters_out = 0, energy_out = 0.  Ties at the trim threshold are kept in the Morton order of the
 * segment over its bounding cube.  A finite pose whose squared distances overflow fp32 (e.g. a
 * translation of 1e20): every such query takes model point 0 at FLT_MAX; if the trimmed energy is
 * then not finite the pose stops after that iteration, is returned exactly as given, and reports
 * energy_out = +Inf (iters_out = 1 when it overflows from the start).  Other poses of the batch are
 * unaffected: each pose's result does not depend on the rest of the batch. */
PGP_API int pgp_tricp(pgp_ctx* ctx, int obj, const float* seg_xyz_host, int ns, double* poses16_host, int k,
                      float trim, float ratio, int max_iter, int* iters_out, float* energy_out);

/* Trimmed point-to-plane ICP: utilities::pointToPlaneICP (PPE/src/misc/utilities.cpp:709-739) -> PCL's
 * TransformationEstimationPointToPlaneLLS, restated (PCL is not vendored: parity unpinned).  Arguments, refusals and result
 * conventions are those of pgp_tricp, and so are the start transform, the queries, the nearest neighbours, the trim (the
 * n_keep smallest POINT-TO-POINT squared distances, ties in Morton order), the stop rule and the final inversion.  Per kept pair,
 * in double: q = the validation point as given, n = its unit validation normal (zero where pgp_set_model zeroed it), p' = the
 * fp32 query, r = ((dx nx + dy ny) + dz nz) with d = p' - q, a = [p' x n, n].  Sums over the kept set: E = sum r^2,
 * H = sum a a^T, g = -sum a r; energy_out = (float)E, the point-to-plane trimmed energy.  When it is finite:
 * x = H^+ g with Jacobi scaling s_j = 1/sqrt(H_jj) (0 where H_jj <= 0), M = S H S = V L V^T by cyclic Jacobi in double (stop
 * when the off-diagonal norm is <= 1e-15 |M|_F, or after 30 sweeps), eigenvalues <= 1e-9 lambda_max dropped (all when
 * lambda_max <= 0), x = S V L^+ V^T S g; x = (alpha, beta, gamma, tx, ty, tz), dR = Rz(gamma) Ry(beta) Rx(alpha), and the
 * transform becomes fp32(dR R, dR t + (tx, ty, tz)), computed in double from the fp32 transform.  A kept set that constrains
 * only some directions (one plane: rank 3) moves the pose in those alone, with the minimum-norm update; normals that are all
 * zero leave it in place, and the loop stops at the second ratio test.  A non-finite energy (overflow or NaN) returns the pose
 * as given with energy_out = +Inf.
 * PGP_E_INVALID in addition: the model slot was set with val_nrm == NULL. */
PGP_API int pgp_tricp_plane(pgp_ctx* ctx, int obj, const float* seg_xyz_host, int ns, double* poses16_host, int k,
                            float trim, float ratio, int max_iter, int* iters_out, float* energy_out);

/* ---------------------------------------------------------------- K6: MCTS node helpers ---- */

/* Explained-point removal of UCTState::performTrICP (PPE/src/hypothesis_verification/mcts/UCTState.cpp:149-174): segment
 * points closer than `threshold` (pointRemovalThreshold, 8 mm) to object `obj`'s VALIDATION cloud placed at each of the
 * n_placed poses (row-major 4x4 doubles; the reference transforms the current object's model by the poses of the objects
 * already placed, :150-155) are flagged.  explained: ns flags (1 = removed).  Returns the number of points that REMAIN. */
PGP_API int pgp_remove_explained(pgp_ctx* ctx, int obj, const float* seg_xyz_host, int ns, const double* placed_poses16, int n_placed,
                                 float threshold, uint8_t* explained);
/* One MCTS expansion's refinement (UCTState::performTrICP, :121-204) for k candidate poses of object `obj` at once:
 * explained-point removal, then pgp_tricp on the unexplained segment.  n_unexplained may be NULL.
 * The input checks of pgp_tricp apply (k = 0 is refused here); when fewer than 3 points remain the poses stay as given
 * with iters_out = 0, energy_out = 0. */
PGP_API int pgp_mcts_tricp(pgp_ctx* ctx, int obj, const float* seg_xyz_host, int ns, const double* placed_poses16, int n_placed,
                           float threshold, double* poses16_host, int k, float trim, float ratio, int max_iter, int* iters_out,
                           float* energy_out, int* n_unexplained);

/* Many refinements in one call: the items of a frame (one per object) or of an expansion batch or rollouts (one per MCTS node
 * or step), each with its own object, segment and placed set.  The arrays go up once, the batch runs as the device pipeline of
 * pgp_refine_batch_dev (explained-point removal over every item with placed objects in one launch, the survivors' count, n_keep
 * and Morton order per item on the device, the trimmed ICP of every pose of every item in one K5 launch: one cluster of two CTAs
 * per pose, the item's source, target grid and scratch rows read from a per-item descriptor), and the results come back with
 * one synchronisation.
 *
 * Item i refines rows [pose_offsets[i], pose_offsets[i + 1]) of poses16 (row-major 4x4 model->camera doubles, in place),
 * iters_out and energy_out; k_i = 0 is allowed.  Its segment is points [seg_offsets[seg], seg_offsets[seg + 1]) of seg_xyz
 * (camera frame, x 3); every segment goes up once however many items use it.  Its placed set is rows [placed_lo, placed_lo +
 * n_placed) of placed16 (row-major 4x4 doubles); items may share rows.  n_unexplained_out: one entry per item, the points left
 * after the removal (the segment size when n_placed = 0).  iters_out, energy_out and n_unexplained_out may be NULL.
 *
 * Each item's poses, iterations, energies and n_unexplained are bitwise those of the single calls on the same context:
 *   PGP_ICP_POINT, n_placed > 0: pgp_mcts_tricp(obj, segment, placed rows, threshold, its poses, trim, ratio, max_iter);
 *   PGP_ICP_POINT, n_placed = 0: pgp_tricp on the whole segment;
 *   PGP_ICP_PLANE, n_placed > 0: pgp_remove_explained, the survivors in their original order, pgp_tricp_plane;
 *   PGP_ICP_PLANE, n_placed = 0: pgp_tricp_plane on the whole segment.
 * At the edges both metrics follow pgp_mcts_tricp: when no point survives, or n_keep < 3, the poses stay as given with
 * iters_out = 0 and energy_out = 0; a pose whose result is not finite is returned as given with energy_out = +Inf.  No result
 * depends on item order, on the other items or on earlier calls.
 *
 * PGP_E_INVALID, before anything runs and with every output untouched:
 *   - metric not PGP_ICP_POINT / PGP_ICP_PLANE; n_items, n_segs or n_placed_rows < 0; a NULL array that has entries;
 *   - seg_offsets or pose_offsets not non-decreasing from 0 (NULL reads as {0} when n_segs / n_items is 0);
 *   - an item's seg outside [0, n_segs) or an empty segment; n_placed < 0 or placed rows outside [0, n_placed_rows);
 *   - a segment coordinate, placed-pose entry or pose entry that is NaN or infinite;
 *   - trim or ratio not > 0, threshold not >= 0 (NaN included);
 *   - PGP_ICP_PLANE on a model slot set without validation normals;
 *   - more than PGP_REFINE_MAX_POINTS segment points or PGP_REFINE_MAX_POSES poses in all; or scratch above PGP_REFINE_MAX_PAIRS,
 *     counted in int64 as the sum over items of (k_i + (n_placed_i > 0)) x segment size -- the d2 / nn rows of the poses
 *     (k_i x n_unexplained_i, bounded by the segment size since n_unexplained is not known before the call) and the flags.
 * PGP_E_NO_MODEL: an item's slot has no model.  n_items = 0 is a valid no-op. */
typedef struct pgp_refine_item {
  int32_t obj;        /* model slot (pgp_set_model): its validation cloud is the ICP target and the explained cloud */
  int32_t seg;        /* segment index: points seg_offsets[seg] .. seg_offsets[seg + 1] of seg_xyz */
  int32_t placed_lo;  /* first row of placed16 */
  int32_t n_placed;   /* number of placed poses (0: nothing is explained) */
} pgp_refine_item;

#define PGP_ICP_POINT 0   /* pgp_tricp's fit */
#define PGP_ICP_PLANE 1   /* pgp_tricp_plane's fit */
#define PGP_REFINE_MAX_POINTS (1ll << 30)
#define PGP_REFINE_MAX_POSES (1ll << 20)
#define PGP_REFINE_MAX_PAIRS (1ll << 30)

PGP_API int pgp_refine_batch(pgp_ctx* ctx, int metric,
                             const float* seg_xyz, const int64_t* seg_offsets, int n_segs,
                             const double* placed16, int64_t n_placed_rows,
                             const pgp_refine_item* items, const int64_t* pose_offsets, int n_items,
                             double* poses16, float threshold, float trim, float ratio, int max_iter,
                             int* iters_out, float* energy_out, int* n_unexplained_out);

/* pgp_refine_batch with the bulk data in device memory, asynchronous on the context's stream (pgp_set_stream): the form for a
 * caller whose segments, placed poses or candidate poses already live on the GPU, or that queues the refinement behind other
 * work.  pgp_refine_batch itself uploads its arguments, runs this pipeline and downloads the results.
 *
 * Arguments are those of pgp_refine_batch.  In device memory (of the context's device, or managed): seg_xyz_dev, placed16_dev,
 * poses16_dev (refined in place), iters_dev, energy_dev and n_unexplained_dev (each may be NULL) and status_dev (one int32).
 * On the host: seg_offsets, items and pose_offsets, so every launch size is known without reading anything back.  The call
 * returns once the work is queued, and the host arrays may be reused at once.  Once the context's scratch has grown to the
 * batch's size (a first call of that size), it makes no host synchronisation and no device-to-host copy; a call of a larger
 * size grows the scratch, and cudaFree / cudaMalloc synchronise the device.
 *
 * Results: each item's poses, iterations, energies and n_unexplained are bitwise what pgp_refine_batch gives on the same inputs
 * (so bitwise the single calls listed there), with the same edge cases.  The work is a fixed number of launches whatever the
 * number of items: ingest (conversion, finiteness, start transforms), explained points, item preparation (survivor count,
 * n_keep, Morton order), one K5 launch over every pose, and the final inversion.
 *
 * Returned at once, with nothing queued and every output untouched: every refusal of pgp_refine_batch that the host can decide
 * (all but the value checks), status_dev == NULL, and a device argument that cudaPointerGetAttributes does not report as device
 * or managed memory of the context's device.
 * On the device: a NaN or infinite segment coordinate, placed-pose entry or pose entry sets *status_dev = PGP_E_INVALID and no
 * output is written; otherwise *status_dev = PGP_OK.  Every call sets *status_dev afresh (n_items = 0 included). */
PGP_API int pgp_refine_batch_dev(pgp_ctx* ctx, int metric,
                                 const float* seg_xyz_dev, const int64_t* seg_offsets, int n_segs,
                                 const double* placed16_dev, int64_t n_placed_rows,
                                 const pgp_refine_item* items, const int64_t* pose_offsets, int n_items,
                                 double* poses16_dev, float threshold, float trim, float ratio, int max_iter,
                                 int* iters_dev, float* energy_dev, int* n_unexplained_dev, int32_t* status_dev);

/* ---------------------------------------------------------------- K7: segment preparation -- */

/* The step in front of the path, for one object of one RGB-D frame: depth decode (utilities::readDepthImage,
 * PPE/src/misc/utilities.cpp:47-61: ((d << 13) | (d >> 3)) / 10000), class mask (GTSegmentation::compute2dSegment,
 * PPE/src/segmentation/Segmentation.cpp:187-207), back-projection of the pixels with 0.1 < depth < 2.0
 * (utilities::convert3dUnOrganizedRGB, utilities.cpp:210-228), then -- restated, PCL being un-vendored -- `leaf` voxel
 * centroids (pcl::VoxelGrid, Segmentation.cpp:226-229), pcl::MovingLeastSquares as the reference configures it (:231-238:
 * polynomial fit of order 2 over the neighbours within normal_radius, the point projected onto the fitted surface, its normal;
 * points with fewer than 3 neighbours vanish), removal of the projected points with fewer than min_neighbors within
 * outlier_radius and normals turned to the camera (pcl::RadiusOutlierRemoval + flipNormalTowardsViewpoint,
 * PPE/src/hypothesis_generation/ObjectPoseCandidateSet.cpp:28-51).  pgp_set_option("k7_mls", 0) selects plain PCA normals on the
 * un-projected centroids instead (round 1's stand-in).
 * depth_raw: rows x cols uint16 as stored in frame-*.depth.png; class_mask: rows x cols uint8; K9 row-major intrinsics.
 * xyz_out / nrm_out: cap x 3 camera-frame points / unit normals, ready for pgp_set_scene.  Returns the number of points.
 * A centroid q is a neighbour of p when ((dx*dx + dy*dy) + dz*dz) <= r*r, in double from the fp32 coordinates, with r the fp32
 * radius promoted to double.  A 6x6 polynomial system whose Cholesky pivot falls to 1e-10 of its diagonal or below (neighbours
 * on one or two lines) is not solved: the point stays on the PCA plane with the plane's normal.
 * PGP_E_INVALID, before anything runs and with every output untouched: a NULL pointer, rows or cols < 1, rows x cols > 2^30, cap < 0,
 * a NaN or infinite K9 entry, fx or fy = 0, leaf not finite and > 0, a radius not > 0, a radius above 16 x leaf, or a leaf so
 * small that a voxel index could exceed 2^30 (coordinates bounded by depth < 2 m over the frame: max(2, 2 |v - cx| / |fx|,
 * 2 |u - cy| / |fy|) / leaf > 2^30).  PGP_E_TOO_LARGE: the voxel table over the segment's extent needs more than 2.5e8 cells.
 * PGP_E_CAPACITY: more than cap points survive; xyz_out and nrm_out are then not written. */
PGP_API int pgp_prepare_segment(pgp_ctx* ctx, const uint16_t* depth_raw, const uint8_t* class_mask, int rows, int cols, int class_id,
                                const float* K9, float leaf, float normal_radius, float outlier_radius, int min_neighbors,
                                float* xyz_out, float* nrm_out, int cap, int* n_valid_pixels);

/* ---------------------------------------------------------------- K8: rendered-depth cost --- */

/* The render + compare step of an MCTS node evaluation (UCTState::render followed by UCTState::computeCost,
 * PPE/src/hypothesis_verification/mcts/UCTState.cpp:93-116; renderer depth_sim/src/renderScene.cpp:36-84).  RESTATED, PARITY
 * UNPINNED: the reference renders with OpenGL (a pcl::simulation fork) and the body of computeCost is not available, so K8 has
 * its own exact contract and returns exact per-object pixel counts from which a per-pixel depth-agreement cost is composed on
 * the host.  The contract, in order (oracle/render_port.py restates it line by line):
 *  1. pose -> fp32 3x4 (as K6); camera-frame vertex (X, Y, Z) per row ((m0 x + m1 y) + m2 z) + m3, unfused fp32.
 *  2. sx = ((fx X) / Z) + cx, sy = ((fy Y) / Z) + cy, fp32, each operation rounded.  Pixel (row r, col c) samples the point
 *     (c, r), the convention of K7's back-projection.
 *  3. vertices snap to 1/256 px: rint(s * 256) to int64, ties to even.  A triangle is dropped whole (no clipping) when a vertex has
 *     a non-finite X, Y or Z, Z <= 0.1f (fp32 compare), or |sx| or |sy| > 2^20 px (or NaN), or when its snapped area is 0.  No
 *     back-face culling.
 *  4. edge function E(a, b, p) = (b.x - a.x)(p.y - a.y) - (b.y - a.y)(p.x - a.x) in int64 on snapped coordinates (exact).  The
 *     triangle (v0, v1, v2) is reoriented (v1 <-> v2) so that its area A = E(v0, v1, v2) > 0; E_0 = E(v1, v2, p),
 *     E_1 = E(v2, v0, p), E_2 = E(v0, v1, p).  p is covered when every E_i > 0, or == 0 on an edge a -> b that owns it:
 *     dy < 0, or dy == 0 && dx > 0 (top-left rule; a shared edge or vertex covers each sample exactly once).
 *  5. depth = (float)((double)A / (((double)E_0 iz_0 + (double)E_1 iz_1) + (double)E_2 iz_2)), iz_i = 1.0 / (double)Z_i, double,
 *     unfused, A = E_0 + E_1 + E_2 exact in int64.
 *  6. per pixel the minimum of the 64-bit key (float_bits(depth) << 32) | slot wins (slot = position in the state; equal depths go
 *     to the smaller slot).  Independent of triangle order.
 *  7. per front pixel of a slot: rendered += 1.  Observed o = K7's decode; if (double)o > 0.1 && (double)o < 2.0 exactly one of
 *     agree (fabsf(r - o) <= tau), in_front (o - r > tau: the object would hide a surface the camera sees), behind (r - o > tau:
 *     the object is occluded) += 1.  on_segment += 1 where class_mask == the mesh's class_id.  Pixels without a valid observation:
 *     rendered - agree - in_front - behind.
 * Image sides are limited to 1 .. 16384 px, meshes to 2^24 vertices and 2^24 triangles. */

/* Triangle mesh of object slot `obj` (model frame: the frame pgp_tricp's poses map from).  vert_xyz: nv x 3, tri3: nt x 3 vertex
 * indices, class_id: the object's label in the class mask (-1: none).  Independent of pgp_set_model.  Replaces a previous mesh.
 * PGP_E_INVALID: nv < 3, nt < 1, a non-finite vertex, an index outside [0, nv). */
PGP_API int pgp_set_mesh(pgp_ctx* ctx, int obj, const float* vert_xyz, int nv, const int32_t* tri3, int nt, int class_id);

/* Observed frame: depth_raw as stored in frame-*.depth.png (decoded exactly as pgp_prepare_segment does), class_mask (NULL: none;
 * on_segment then stays 0), K9 row-major intrinsics (fx = K[0], fy = K[4], cx = K[2], cy = K[5], as K7).  class_pixels_out
 * (256 entries, NULL allowed): pixels of each label with valid depth (all 0 without a mask).  PGP_E_INVALID: rows or cols
 * outside 1 .. 16384, a non-finite K9 entry, fx <= 0 or fy <= 0. */
PGP_API int pgp_set_depth_observation(pgp_ctx* ctx, const uint16_t* depth_raw, const uint8_t* class_mask, int rows, int cols,
                                      const float* K9, int64_t* class_pixels_out);

/* One state rendered in full: depth_out rows x cols fp32 metres (0 = nothing), slot_out rows x cols (-1 = nothing; NULL allowed).
 * PGP_E_TOO_LARGE: the state covers more than 2^31 - 1 (triangle, tile) entries; depth_out and slot_out then hold an empty frame. */
PGP_API int pgp_render_depth(pgp_ctx* ctx, const int32_t* obj_ids, const double* poses16, int n, float* depth_out, int32_t* slot_out);

typedef struct pgp_depth_counts { int32_t rendered, agree, in_front, behind, on_segment; } pgp_depth_counts;
/* n_states states in CSR form: state s places obj_ids[state_offsets[s] .. state_offsets[s+1]) at the matching poses16 (row-major 4x4
 * model->camera doubles).  out: one record per placed object (state_offsets[n_states] records), counted over the pixels where that
 * object is the front surface.  Each state's records equal that state evaluated alone.
 * PGP_E_INVALID before anything runs, outputs untouched: no observation set, state_offsets not non-decreasing from 0, more than
 * PGP_MAX_OBJECTS objects in a state, an object id outside [0, PGP_MAX_OBJECTS), a non-finite pose entry, tau < 0 or not finite.
 * PGP_E_NO_MODEL: an object without a mesh.  n_states = 0 and empty states are valid. */
PGP_API int pgp_depth_cost(pgp_ctx* ctx, const int64_t* state_offsets, int n_states, const int32_t* obj_ids, const double* poses16,
                           float tau, pgp_depth_counts* out);

/* pgp_depth_cost with the poses and counts in device memory, asynchronous on the context's stream (pgp_set_stream): the form for an
 * MCTS driver whose refined poses are already on the GPU (pgp_refine_batch_dev), so that refinement, rendering and cost run as one
 * stream of work.  pgp_depth_cost and pgp_render_depth run this pipeline themselves: they upload, run it, download and
 * synchronise once.
 *
 * Arguments are those of pgp_depth_cost.  On the host: state_offsets and obj_ids (the tree structure; with them every mesh and
 * every chunk of the work is known without reading anything back).  In device memory (of the context's device, or managed):
 * poses16_dev (one row-major 4x4 double per record), out_dev (one pgp_depth_counts per record) and status_dev (one int32).  The
 * call returns once the work is queued, and the host arrays may be reused at once.  Once the context's scratch has grown to the
 * call's size (a first call of that size), it makes no host synchronisation and no device-to-host copy; a call of a larger size
 * grows the scratch, and cudaFree / cudaMalloc synchronise the device.
 *
 * Results: bitwise those of pgp_depth_cost on the same inputs.  The states are rasterized in chunks cut on the host by triangles,
 * vertices and (state, tile) bins; each chunk reserves min(2^25, its triangles x the image's 16 x 16 tiles) (triangle, tile) entries.
 *
 * Returned at once, with nothing queued and every output untouched: every refusal of pgp_depth_cost that the host can decide (all
 * but the pose values), status_dev == NULL, and a device argument that cudaPointerGetAttributes does not report as device or
 * managed memory of the context's device.
 * On the device, every call sets *status_dev afresh (n_states = 0 included):
 *   PGP_OK;
 *   PGP_E_INVALID: a pose entry is NaN or infinite;
 *   PGP_E_CAPACITY: a chunk needs more (triangle, tile) entries than it reserved (pgp_depth_cost evaluates such states in
 *     smaller chunks).
 * On either error out_dev is not written. */
PGP_API int pgp_depth_cost_dev(pgp_ctx* ctx, const int64_t* state_offsets, int n_states, const int32_t* obj_ids,
                               const double* poses16_dev, float tau, pgp_depth_counts* out_dev, int32_t* status_dev);

/* n_states states in CSR form, as pgp_depth_cost_dev, rendered into device memory on the context's stream: the form for a caller that
 * composes its own per-pixel cost on the GPU from the rendered frames.  depth_dev: n_states x rows x cols fp32 metres, state s at
 * offset s x rows x cols (0 = nothing); slot_dev: the same layout in int32 (-1 = nothing), or NULL.  Frame s is bitwise
 * pgp_render_depth of state s alone; an empty state gives an empty frame.  Offsets are 64-bit: n_states x rows x cols may exceed 2^31.
 *
 * Structure, asynchrony, device memory and refusals are those of pgp_depth_cost_dev (tau aside): the call is queued and returns,
 * and once the scratch has grown to the call's size it makes no host synchronisation and no device-to-host copy.  Returned at once,
 * with nothing queued and every frame untouched: every refusal the host can decide, status_dev == NULL, and a depth_dev, slot_dev,
 * poses16_dev or status_dev that is not device or managed memory of the context's device.  *status_dev, set afresh by every call
 * (n_states = 0 included):
 *   PGP_OK: every frame is written;
 *   PGP_E_INVALID: a pose entry is NaN or infinite; no frame is written;
 *   PGP_E_CAPACITY: a chunk needs more (triangle, tile) entries than it reserved; the frames' contents are then unspecified, and
 *     pgp_render_depth renders those states (it re-cuts the chunks). */
PGP_API int pgp_render_depth_dev(pgp_ctx* ctx, const int64_t* state_offsets, int n_states, const int32_t* obj_ids,
                                 const double* poses16_dev, float* depth_dev, int32_t* slot_dev, int32_t* status_dev);

/* pgp_set_depth_observation on device data (of the context's device, or managed): depth_raw_dev rows x cols uint16 in the stored
 * encoding, class_mask_dev rows x cols uint8 or NULL, K9 on the host, class_pixels_dev 256 x int64 or NULL (zeroed, then the pixels
 * of each label with valid depth; all 0 without a mask).  Queued on the context's stream with no host synchronisation: the raw depth
 * is decoded into the context's frame and the mask copied into the context's buffer, so the caller's buffers are read only by work
 * ordered at this call, and every call queued after it on the stream sees this observation.  Refusals: those of
 * pgp_set_depth_observation, and a device argument that is not device or managed memory of the context's device. */
PGP_API int pgp_set_depth_observation_dev(pgp_ctx* ctx, const uint16_t* depth_raw_dev, const uint8_t* class_mask_dev, int rows,
                                          int cols, const float* K9, int64_t* class_pixels_dev);

#define PGP_MAX_OBJECTS 64
#define PGP_MAX_CELLS (1ll << 29)

#ifdef __cplusplus
}
#endif
#endif /* PGP_H_ */
