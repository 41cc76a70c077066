// Internal declarations shared by the translation units of libpgp.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "pgp.h"

#define PGP_WORK_BYTES (512 << 10)   // pgp_ctx::work, allocated once in pgp_create (k4_select.cu static_asserts that its layout fits)
#define VREC_EPS_STEP (0.6f / 254.0f)   // K1c cone records: code c in 1..254 bounds |n_i - n_rep| by c * VREC_EPS_STEP
#define PGP_WARPS_PER_CTA 8
#define PGP_THREADS (32 * PGP_WARPS_PER_CTA)

// Device buffer that only ever grows (cudaMalloc is not on any steady-state path).
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return static_cast<T*>(p); }
};

// Pinned staging for the one host -> device upload of a call's host-built tables (K5 and K8 device pipelines): PGP_STAGES buffers
// used in turn, each reused once its last copy has run, so that a call queues without waiting unless PGP_STAGES calls are still
// queued.  The buffers grow together, so that one call of a size readies every later call of that size.
constexpr int PGP_STAGES = 4;
struct StagingRing {
  struct Stage { void* host = nullptr; size_t cap = 0; cudaEvent_t copied = nullptr; };
  Stage stage[PGP_STAGES];
  unsigned next = 0;
  // the next buffer, at least `bytes` long and free to be written
  cudaError_t acquire(size_t bytes, Stage** out) {
    cudaError_t e = cudaSuccess;
    if (stage[0].cap < bytes) {
      const size_t cap = bytes + bytes / 4 + 256;
      for (Stage& g : stage) {
        if (!g.copied && (e = cudaEventCreateWithFlags(&g.copied, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventSynchronize(g.copied)) != cudaSuccess) return e;
        if (g.host) cudaFreeHost(g.host);
        g.host = nullptr; g.cap = 0;
        if ((e = cudaMallocHost(&g.host, cap)) != cudaSuccess) return e;
        g.cap = cap;
      }
    }
    Stage& g = stage[next++ % PGP_STAGES];
    if ((e = cudaEventSynchronize(g.copied)) != cudaSuccess) return e;
    *out = &g;
    return cudaSuccess;
  }
  // queues the copy of the buffer's first `bytes` to dev on st, and marks the buffer busy until it has run
  static cudaError_t upload(Stage* g, void* dev, size_t bytes, cudaStream_t st) {
    cudaError_t e = cudaMemcpyAsync(dev, g->host, bytes, cudaMemcpyHostToDevice, st);
    return e != cudaSuccess ? e : cudaEventRecord(g->copied, st);
  }
  void release() {
    for (Stage& g : stage) {
      if (g.host) cudaFreeHost(g.host);
      if (g.copied) cudaEventDestroy(g.copied);
      g = Stage{};
    }
  }
};

// Scene voxel grid ("K1").  Cell edge h = delta * (1 + 2^-8) so that every scene point that can
// pass the fp32 test d2 <= delta^2 lies in the 27 cells around the query's cell (DESIGN.md).
// Two empty apron cells on every side: a query in cells 1..dim-2 never indexes out of range.
struct GridParams {
  float lo[3];        // origin of cell (0,0,0)
  float inv_h;        // 1 / h
  float h;
  int dim[3];
  int64_t n_cells;
  float r2;           // fl(fl(delta) * fl(delta)), the reference's sq_eps (match4pcsBase.cc:1710)
  // fine tri-state classification (K1b): every cell whose 27-neighbourhood is occupied owns a
  // block of 8x8x8 sub-voxels, 2 bits each: 0 = no scene point can be within delta of ANY query that
  // lands in the voxel, 1 = some scene point is within delta of EVERY such query, 2 = undecided.
  int fine;           // sub-voxels per cell edge (8), 0 = not built
  float inv_hf;       // fine * inv_h  (exact: power-of-two scaling)
  float hf;           // h / fine
  float inflate;      // how far outside its ideal box a voxel's queries may lie (rounding of the fast path)
  float pos_bound;    // the fast (FMA) transform path is valid for hypotheses whose intermediates stay below this
  float dlo2, dhi2;   // (delta (1 -+ 1e-5))^2: certainly-inside / certainly-outside thresholds
  int n_blocks;
};

struct Scene {
  int n = 0;
  float delta = 0.f;
  float cP[3] = {0, 0, 0};
  GridParams g{};
  DevBuf xyz_raw;      // n x float3, camera frame (for the prior projection)
  DevBuf nrm_raw;      // n x float3 as given (original order)
  bool has_nrm = false;
  DevBuf unsorted;     // n x float4 centred, original order (staging of the build)
  DevBuf cursor;       // (n_cells + 1) x u32 scatter cursors
  int64_t bitmap_words = 0;
  DevBuf pts;          // n x float4 sorted by cell: x,y,z centred, w = original index (as int bits)
  DevBuf aux;          // n x float4 sorted by cell: unit normal, prior
  DevBuf cell_start;   // (n_cells + 1) x u32
  DevBuf cell_of;      // n x u32 (scratch: cell id per original point)
  DevBuf bitmap;       // ceil(n_cells/32) x u32: dilated occupancy (any point in the 27 cells)
  DevBuf bmrank;       // per bitmap word: {bits, number of set bits in all earlier words} -> block id of a cell
  DevBuf block_cell;   // n_blocks x u32: cell of block b
  DevBuf codes;        // n_blocks x 32 words: 512 2-bit voxel states, voxel v = (sz*8+sy)*8+sx at bits 2(v&15) of word v>>4
  DevBuf near_cnt;     // build scratch: n_blocks x 512 u16 candidate counts
  DevBuf hdr;          // build scratch: n_blocks x 8 u32: {.., #ambig voxels at [5], #overflow records at [6], ..}
  DevBuf region;       // build scratch: region sizes / bases
  DevBuf hdrw;         // n_blocks x 32 u32: global rank of the first AMBIG voxel of each label word
  DevBuf aslot;        // per AMBIG voxel (rank order), 32 bytes: {x0, y0, z0, n} {x1, y1, z1, first overflow record}, candidate 0 closest to the voxel centre
  DevBuf aovf;         // float4 copies {x, y, z, original index} of the AMBIG voxels' candidates beyond the second
  int64_t n_ovf_records = 0;   // records in aovf
  int64_t n_ambig_voxels = 0;
  DevBuf wvox;         // K1c build scratch: n_blocks x 512 u32 counts / offsets
  DevBuf wbase;        // K1c build scratch: n_blocks u32: first wlists entry of the block's region
  DevBuf wcnt;         // K1c: n_blocks x 512 bytes: candidate count of every voxel (0 for OUT voxels)
  DevBuf wword;        // K1c: n_blocks x 32 u32: first wlists entry of the 16 voxels of each label word
  DevBuf wlists;       // K1c: ORIGINAL INDEX (u32) of the nearest-neighbour candidates of every non-OUT voxel (the points are read from `unsorted`)
  DevBuf vrec;         // K1c: n_blocks x 512 u32: per voxel (code << 24 | representative candidate): how far the candidates' normals spread (k1_fine.cu)
  int64_t n_wlist_entries = 0;
  DevBuf dist;         // K1d: f32 per sub-cell (dist_r per cell edge), lower bound of the distance from any point of the sub-cell to the nearest scene point
  DevBuf dist_tmp;     // K1d build scratch
  int dist_r = 1;
  DevBuf aux_orig;     // n x float4 in ORIGINAL order: unit normal, prior (the K1c records carry original indices)
  bool wlists_ready = false, wlists_tried = false;
  DevBuf prior;        // n x f32 in ORIGINAL order
  DevBuf scratch;      // scan scratch etc.
  int64_t n_occupied = 0;
  int64_t n_mixed = 0;
  bool priors_binary = true;   // every prior is exactly 0 or 1 -> weighted sums are order-free
  bool ready = false;
};

struct Model {
  int nq = 0, nv = 0;
  float cQ[3] = {0, 0, 0};
  float val_rinf = 0.f;  // max |coordinate| of the centred validation cloud
  DevBuf search;       // nq x float4 centred (w = 0)
  DevBuf search_nrm;   // nq x float4 unit normal
  DevBuf search_unit;  // nq x float4: search cloud in the unit cube (PairCreationFunctor::synch3DContent, pairCreationFunctor.h:102-138)
  float unit_ratio = 1.f;      // _ratio
  float unit_center[3] = {0, 0, 0};   // _gcenter
  float search_diameter = 0.f; // P_diameter_ estimate (match4pcsBase.cc:274-283)
  DevBuf val;          // nv x float4 centred, in a cache-friendly order; w = original index bits
  DevBuf val_nrm;      // nv x float4 unit normal, same order
  DevBuf val_groups;   // ceil(nv/32) x float4: bounding sphere {centre, radius} of each run of 32 points of `val` (K3 group cull)
  DevBuf val_orig;     // nv x float4 centred, ORIGINAL order (weighted mode with general priors, TrICP target)
  DevBuf val_nrm_orig;
  bool val_has_nrm = false;   // pgp_set_model was given validation normals (the point-to-plane fit needs them)
  // model-space grid for TrICP (K5): nearest validation-model point of any query
  DevBuf val_raw;        // nv x float4, model frame as given (un-centred): the TrICP target
  float val_raw_lo[3] = {0, 0, 0}, val_raw_hi[3] = {0, 0, 0};
  DevBuf tgrid_pts, tgrid_start;
  float tg_lo[3] = {0, 0, 0}, tg_g = 1.f; int tg_dim[3] = {1, 1, 1};
  bool tgrid_ready = false;
  bool ready = false;
  // generated hypotheses (K2)
  DevBuf gen_T, gen_counts, gen_scores;
  int64_t n_gen = 0;
  int64_t gen_index_base = -1;  // global index of the first generated hypothesis (bases sharded over ranks: pgp_comm_sync_generated); -1 = not known yet
  int n_gen_bases = 0;
  bool gen_scored = false;
  // PPF map of the SEARCH cloud (operMode 1 / StoCS): sorted packed keys -> pair lists, + presence bitset
  DevBuf ppf_keys, ppf_offsets, ppf_pairs, ppf_bits;
  int n_ppf_keys = 0;
  int64_t n_ppf_pairs = 0;
  std::vector<uint32_t> h_ppf_keys, h_ppf_offsets;
  std::vector<int32_t> h_ppf_pairs;
};

struct LastBatch {
  const float* T = nullptr;         // device
  const uint32_t* counts = nullptr; // device
  const float* scores = nullptr;    // device
  int64_t n = 0;
  int mode = 0;
  int obj = -1;
};

struct PendingBatch {            // pgp_score_lcp_begin ... pgp_score_lcp_end
  bool active = false, streamed = false;
  int obj = -1, mode = 0;
  int64_t n = 0;
  uint32_t* counts = nullptr;    // host
  float* scores = nullptr;       // host
};
// The host-buffer scoring API keeps TWO batches in flight (upload of batch i+1 under the scoring of batch i, download of batch i
// under the scoring of batch i+1): each has its own device residency, upload counter and events.
struct BatchSlot {
  DevBuf T, counts, scores;      // device residency of the batch
  PendingBatch pending;
  uint32_t* marks = nullptr;     // pinned, 16 words: [0..4] chunk boundaries, [6] zero, [7] zero, [8] abort flag read back
  cudaEvent_t ev_start = nullptr, ev_first = nullptr, ev_scored = nullptr, ev_done = nullptr;   // queued so far | first chunk up | K3 done | downloads done
};
#define PGP_BATCH_SLOTS 2

struct pgp_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;      // host -> device of the host-buffer API
  cudaStream_t back_stream = nullptr;      // device -> host of the host-buffer API (PCIe is full duplex: its own stream)
  Scene scene;
  std::vector<Model> models;
  LastBatch last;
  BatchSlot batch[PGP_BATCH_SLOTS];        // host-buffer API: batches in flight (pgp_score_lcp_begin / _end)
  int batch_head = 0, batch_tail = 0;      // next slot to begin / to end (counters, slot = value % PGP_BATCH_SLOTS)
  DevBuf work;                                   // counters / select scratch
  DevBuf topk_out;
  void* pinned = nullptr; size_t pinned_cap = 0;
  int64_t launches = 0;
  void* comm = nullptr;                    // pgp_comm.cu: NCCL communicator, exchange stream and slots (pgp_comm_release)
  void* k2_scratch = nullptr;              // k2_pcs.cu: the generator's device scratch (k2_release)
  void* k5_scratch = nullptr;              // k5_tricp.cu (k5_release)
  void* k6_scratch = nullptr;              // k6_explained.cu (k6_release)
  void* k7_scratch = nullptr;              // k7_segment.cu (k7_release)
  void* k8_scratch = nullptr;              // k8_render.cu: meshes, observation, rasterizer scratch (k8_release)
  void* k4d_scratch = nullptr;             // k4d_distinct.cu: symmetries, suppression mask, staging (k4d_release)
  int k7_mls = 1;                          // segment preparation: 1 = MLS polynomial projection + normals (what the reference runs), 0 = PCA normals on the centroids
  int stream_upload = 1;  // pgp_score_lcp: overlap the batch upload with the scoring launch (0: upload first; use under profilers)
  int tail_split = 4;     // K3 fine kernel: model chunks per hypothesis in the last wave (1 = off)
  int group_cull = 1;     // K3 fine kernel: drop groups of 32 model points whose bounding sphere cannot reach the scene (0 = off, test hook)
  int force_coarse = 0;   // test hook: score on the 27-cell path even when the fine grid exists
  std::string err;
};

int pgp_fail(pgp_ctx* ctx, int code, const char* fmt, ...);
#define PGP_CUDA(ctx, expr)                                                                     \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess)                                                                     \
      return pgp_fail(ctx, PGP_E_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
  } while (0)

// k1_grid.cu
int k1_build_grid(pgp_ctx* ctx);
int k1_project_priors(pgp_ctx* ctx, const uint16_t* img_dev, int rows, int cols, const float* K9);
int k1_refresh_sorted_priors(pgp_ctx* ctx);
int k1_fill_priors(pgp_ctx* ctx, float v);
int k1_build_fine(pgp_ctx* ctx);
int k1_build_wlists(pgp_ctx* ctx);
int k1_fine_stats(pgp_ctx* ctx, int64_t* out8);
int pgp_scan_exclusive_u32(pgp_ctx* ctx, uint32_t* data, int64_t n, uint32_t* scratch);
// k3_lcp.cu
int k3_score(pgp_ctx* ctx, const Model& m, const float* T_dev, int64_t n, int mode, uint32_t* counts_dev, float* scores_dev, uint32_t* ready_dev = nullptr);
bool k3_streams_upload(pgp_ctx* ctx, int mode);
int k3_nearest(pgp_ctx* ctx, const Model& m, const float* T_dev, int32_t* idx_dev, int gate);
// k4_select.cu
constexpr int K4_MAX_K = 4096;   // largest k of a selection, and the most chain candidates one launch can sort
int k4_topk(pgp_ctx* ctx, const LastBatch& b, int k, int64_t index_base, pgp_hyp* out_host, int* n_out);
int k4_topk_dev(pgp_ctx* ctx, const LastBatch& b, int k, int64_t index_base, pgp_hyp* out_dev);
int k4_chain(pgp_ctx* ctx, const LastBatch& b, int64_t index_base, pgp_hyp* out_host, int cap, int* n_out);
int k4_select_dev(pgp_ctx* ctx, const LastBatch& b, int k, int64_t index_base, int mode, pgp_hyp* hdr_dev, pgp_hyp* out_dev);
// k4d_distinct.cu (arguments checked by the C ABI in pgp_api.cu)
void k4d_set_symmetries(pgp_ctx* ctx, int obj, const double* R9, int n);
// pgp_distinct_dev after its checks: descriptors up from pinned staging, the mask and the scan queued on ctx->stream
int k4d_distinct_dev(pgp_ctx* ctx, const int32_t* objs, const int64_t* pool_offsets, int n_lists, const pgp_hyp* pool_dev, int k,
                     double max_dist, double cos_angle, pgp_hyp* out_dev, double* poses16_dev, int32_t* n_kept_dev);
// one list from host memory: pool up, run, kept records down, one synchronisation; returns the number kept
int k4d_distinct_host(pgp_ctx* ctx, int obj, const pgp_hyp* pool_host, int m, int k, double max_dist, double cos_angle, pgp_hyp* out_host);
void k4d_release(pgp_ctx* ctx);
// pgp_comm.cu
void pgp_comm_release(pgp_ctx* ctx);
bool pgp_comm_active(const pgp_ctx* ctx);
extern "C" int pgp_comm_improving_chain(pgp_ctx* ctx, int obj, int64_t index_base, pgp_hyp* out_host, int cap);
// k2_pcs.cu
int k2_extract_pairs(pgp_ctx* ctx, const Model& m, float dist, float eps, int32_t* pairs_host, int64_t cap, int64_t* n_pairs);
int k2_find_quads(pgp_ctx* ctx, const Model& m, const int32_t* base4, float inv1, float inv2, float eps,
                  const int32_t* p1, int64_t n1, const int32_t* p2, int64_t n2, int32_t* quads_host, int64_t cap, int64_t* n_quads);
int k2_find_quads_v4pcs(pgp_ctx* ctx, const Model& m, const int32_t* base4, float eps, int32_t* quads_host, int64_t cap, int64_t* n_quads);
int k2_rigid_from_quads(pgp_ctx* ctx, const Model& m, const int32_t* base4, const int32_t* quads_host, int64_t n, float* T_host, uint8_t* ok_host);
int k2_generate(pgp_ctx* ctx, Model& m, const pgp_pcs_opts* o, uint64_t seed, int base_lo, int base_hi, int64_t max_hyp, int64_t* n_hyp);
int k2_set_ppf_map(pgp_ctx* ctx, Model& m, const int32_t* keys4, const int64_t* offsets, const int32_t* pairs, int64_t n_keys);
int k2_build_ppf_map(pgp_ctx* ctx, Model& m);
int k2_scene_ppf_keys(pgp_ctx* ctx, const int32_t* pairs_host, int64_t n, int32_t* keys4_host);
uint32_t k2_stocs_engine_seed(uint64_t seed, int base, int attempt);
int k2_get_bases(pgp_ctx* ctx, const Model& m, int n_bases, int32_t* ids_host, float* inv_host, uint8_t* ok_host);
void k2_release(pgp_ctx* ctx);
void k5_release(pgp_ctx* ctx);
void k6_release(pgp_ctx* ctx);
void k7_release(pgp_ctx* ctx);
// k5_tricp.cu
// plane: the point-to-plane fit (pgp_tricp_plane) instead of the point-to-point one (pgp_tricp)
int k5_tricp(pgp_ctx* ctx, Model& m, const float* seg_xyz_host, int ns, double* poses16_host, int k, float trim, float ratio,
             int max_iter, int* iters_out, float* energy_out, bool plane);
// pgp_refine_batch after its argument checks: uploads the host arrays, runs k5_refine_batch_dev, downloads, synchronises once
int k5_refine_batch(pgp_ctx* ctx, bool plane, const float* seg_xyz, const int64_t* seg_offsets, int n_segs, const double* placed16, int64_t n_placed_rows,
                    const pgp_refine_item* items, const int64_t* pose_offsets, int n_items, double* poses16, float threshold, float trim,
                    float ratio, int max_iter, int* iters_out, float* energy_out, int* n_unexplained_out);
// pgp_refine_batch_dev after its argument checks: the whole batch queued on ctx->stream (seg_xyz, placed16, poses16 and the outputs
// in device memory, the structure on the host); *status_dev = PGP_OK, or PGP_E_INVALID with no output written when a value is
// not finite
int k5_refine_batch_dev(pgp_ctx* ctx, bool plane, const float* seg_xyz, const int64_t* seg_offsets, int n_segs, const double* placed16,
                        int64_t n_placed_rows, const pgp_refine_item* items, const int64_t* pose_offsets, int n_items, double* poses16,
                        float threshold, float trim, float ratio, int max_iter, int* iters_out, float* energy_out, int* n_unexplained_out,
                        int32_t* status_dev);

// ---------------------------------------------------------------------------------------------
// fp32 arithmetic in the reference's association, every operation individually rounded
// (SURVEY.md 7 "Hard parts"; the library is also compiled with -fmad=false).
__device__ __forceinline__ float xf_row(float m0, float m1, float m2, float m3, float x, float y, float z) {
  // (mat * p.homogeneous()).head<3>()  S4/algorithms/match4pcsBase.cc:1717 :  ((m0 x + m1 y) + m2 z) + m3
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m0, x), __fmul_rn(m1, y)), __fmul_rn(m2, z)), m3);
}
__device__ __forceinline__ float sqdist3(float ax, float ay, float az, float bx, float by, float bz) {
  // (q - p).squaredNorm()  S4/accelerators/kdtree.h:423 :  dx^2 + (dy^2 + dz^2)
  float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz)));
}
__device__ __forceinline__ float dot3_tree(float a0, float a1, float a2, float b0, float b1, float b2) {
  // 3-element lazy product / dot: a0 b0 + (a1 b1 + a2 b2)   match4pcsBase.cc:1755-1756
  return __fadd_rn(__fmul_rn(a0, b0), __fadd_rn(__fmul_rn(a1, b1), __fmul_rn(a2, b2)));
}
// cell coordinate of a centred coordinate; the SAME function bins scene points and queries, and
// it is monotone, which is what the 27-cell completeness argument needs.
__device__ __forceinline__ float cell_coord(float x, float lo, float inv_h) { return __fmul_rn(__fsub_rn(x, lo), inv_h); }
// utilities::convertToMatrix (Isometry3d -> Matrix4f): the top 3x4 of a row-major 4x4 double pose, each entry rounded to fp32
// (K6 placed poses, K8 rendered poses)
__host__ __device__ inline void pose16_to_f32x12(const double* pose16, float* T12) {
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) T12[4 * r + c] = (float)pose16[4 * r + c];
}
// utilities::readDepthImage (PPE/src/misc/utilities.cpp:47-61): ((d << 13) | (d >> 3)) as u16, / 10000 (K7 segments, K8 observations)
__device__ __forceinline__ float decode_depth(uint16_t raw) {
  const uint16_t d = (uint16_t)((raw << 13) | (raw >> 3));
  return __fdiv_rn((float)d, 10000.0f);
}
// utilities::convert3dUnOrganizedRGB's depth > 0.1 && depth < 2.0: a float compared with double literals
__device__ __forceinline__ bool depth_valid(float d) { return (double)d > 0.1 && (double)d < 2.0; }
// k6_explained.cu
int k6_remove_explained(pgp_ctx* ctx, Model& m, const float* seg_xyz_host, int ns, const double* placed16_host, int n_placed, float threshold,
                        uint8_t* flags_host, int* n_unexplained);
// One segment of a batch flagged against a model placed at rows [placed_lo, placed_lo + n_placed) of the placed transforms
// (pgp_refine_batch): its flags start at flag_lo, its blocks of K6_T points at block_lo.
constexpr int K6_T = 256;
struct K6Dev { const float4* model; int nv, ns, n_placed; int64_t seg_lo, placed_lo, flag_lo, block_lo; };
// The flags of every job in one launch on ctx->stream, bit for bit those of k6_remove_explained: seg4 is every segment point
// (w = 0), T12 every placed row (pose16_to_f32x12), n_blocks the sum over the jobs of ceil(ns / K6_T).
int k6_mark_batch_dev(pgp_ctx* ctx, const float4* seg4, const K6Dev* jobs_dev, int n_jobs, int64_t n_blocks, const float* T12, float threshold,
                      uint8_t* flags_dev);
// the points with flag 0, in their original order (extract.setNegative(true), UCTState.cpp:170-174); returns their number
int k6_compact(const float* seg_xyz_host, int ns, const uint8_t* flags, float* out_xyz);
// k7_segment.cu
int k7_prepare_segment(pgp_ctx* ctx, const uint16_t* depth_host, const uint8_t* mask_host, int rows, int cols, int cls, const float* K9, float leaf,
                       float normal_r, float outlier_r, int min_nb, float* xyz_host, float* nrm_host, int cap, int* n_out, int* n_raw_out);
// k8_render.cu (arguments checked by the C ABI in pgp_api.cu)
int k8_set_mesh(pgp_ctx* ctx, int obj, const float* vert_xyz, int nv, const int32_t* tri3, int nt, int class_id);
bool k8_has_mesh(pgp_ctx* ctx, int obj);
bool k8_has_observation(pgp_ctx* ctx);
int k8_set_observation(pgp_ctx* ctx, const uint16_t* depth_raw, const uint8_t* class_mask, int rows, int cols, const float* K9, int64_t* class_pixels_out);
// the host forms: the poses up, the device pipeline, the results down, one synchronisation (one more, and a second run, when a
// chunk's (triangle, tile) pairs exceeded its reservation)
int k8_render(pgp_ctx* ctx, const int32_t* obj_ids, const double* poses16, int n, float* depth_out, int32_t* slot_out);
int k8_depth_cost(pgp_ctx* ctx, const int64_t* state_offsets, int n_states, const int32_t* obj_ids, const double* poses16, float tau, pgp_depth_counts* out);
// pgp_depth_cost_dev after its checks: the pipeline queued on ctx->stream; *status_dev = PGP_OK, PGP_E_INVALID (a pose entry not
// finite) or PGP_E_CAPACITY (a chunk's pairs exceeded its reservation), out_dev written only on PGP_OK
int k8_depth_cost_dev(pgp_ctx* ctx, const int64_t* state_offsets, int n_states, const int32_t* obj_ids, const double* poses16_dev, float tau,
                      pgp_depth_counts* out_dev, int32_t* status_dev);
// pgp_render_depth_dev after its checks: the same pipeline in render mode, state s's frame to depth_dev / slot_dev + s x rows x cols;
// the status as k8_depth_cost_dev, the frames cleared and written only while it is PGP_OK
int k8_render_dev(pgp_ctx* ctx, const int64_t* state_offsets, int n_states, const int32_t* obj_ids, const double* poses16_dev, float* depth_dev,
                  int32_t* slot_dev, int32_t* status_dev);
// pgp_set_depth_observation_dev after its checks: decode, mask copy and histogram queued on ctx->stream, no synchronisation
int k8_set_observation_dev(pgp_ctx* ctx, const uint16_t* depth_raw_dev, const uint8_t* class_mask_dev, int rows, int cols, const float* K9,
                           int64_t* class_pixels_dev);
void k8_release(pgp_ctx* ctx);
