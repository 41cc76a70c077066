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
 * tuning): out8 = {cells whose 512 sub-voxels are all OUT, all IN, mixed; sub-voxels OUT, IN, AMBIG; words of
 * AMBIG candidate lists; entries of the nearest-candidate lists (0 until a WEIGHTED call built them)}. */
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
 *                           serialise streams)
 *   "k3_warps_count", "k3_warps_weighted" = 16 | 24 | 32   warps per CTA of the scoring kernel (defaults 32 / 24) */
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
 * xyz_out / nrm_out: cap x 3 camera-frame points / unit normals, ready for pgp_set_scene.  Returns the number of points. */
PGP_API int pgp_prepare_segment(pgp_ctx* ctx, const uint16_t* depth_raw, const uint8_t* class_mask, int rows, int cols, int class_id,
                                const float* K9, float leaf, float normal_radius, float outlier_radius, int min_neighbors,
                                float* xyz_out, float* nrm_out, int cap, int* n_valid_pixels);

#define PGP_MAX_OBJECTS 64
#define PGP_MAX_CELLS (1ll << 29)

#ifdef __cplusplus
}
#endif
#endif /* PGP_H_ */
