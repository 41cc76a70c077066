// K4d -- pose-distinct candidates: greedy non-maximum suppression in pose space over pools of scored hypotheses.
//
// The reference's only CUDA kernel is a box NMS (rcnn_detection_package/lib/nms/nms_kernel.cu); its pose-space analogue,
// greedyClustering, is dead code (HypothesisSelection.cpp:161).  K4d has its own exact contract (include/pgp.h, pgp_distinct_dev;
// oracle/select_port.py restates it in float64):
//   record i of a pool is kept iff no earlier kept record suppresses it, until k are kept; records with index < 0 are skipped;
//   a suppresses b iff ((dx*dx + dy*dy) + dz*dz) <= max_dist^2 on the translations and, for S = I or one of the object's
//   symmetries, sum_rc R_a[r][c] (R_b S)[r][c] >= 1 + 2 cos_angle, every operation in double and rounded on its own.
//
// Two launches whatever the number of lists:
//   k4d_mask  one 64 x 64 tile of one list's upper triangle per CTA step (persistent grid over every list's tiles): bit j of word
//             cb of row i says "i suppresses j" (j > i).  The translation test runs first; rotations only for the pairs it passes.
//   k4d_scan  one warp per list: the greedy walk over the mask, 64 records per step.  Each lane keeps two of the 64 "removed"
//             words of a 4096-pool in registers and ORs in the row of every kept record.  The same warp writes the kept records,
//             their camera-frame poses, the padding slots and the count.
// The per-list descriptors and the symmetry matrices go up in one copy from pinned staging; the mask lives in context scratch
// that only grows, so a call of a size already seen makes no host synchronisation.
#include <algorithm>
#include <vector>

#include "pgp_internal.cuh"

namespace {

constexpr int TB = 64;             // tile edge and threads per k4d_mask CTA
constexpr int SCAN_WARPS = 4;      // lists per k4d_scan CTA
constexpr int MAX_SYM = PGP_MAX_SYMMETRIES;

struct ListDesc {
  int64_t pool_lo;     // first record of the list in the pool
  int64_t mask_lo;     // first mask word (m x nw words, row-major)
  int64_t tile_lo;     // first tile of the list in the flat tile order
  int64_t out_lo;      // first output slot (list x k)
  int m, nw;           // records, words per mask row (ceil(m / 64))
  int sym_lo, n_sym;   // the object's symmetries: matrices [sym_lo, sym_lo + n_sym) of the call's table
  float cQ[3];         // the object's search centroid (camera-frame poses)
  int pad;
};

struct MaskParams {
  const ListDesc* lists;
  int n_lists;
  int64_t n_tiles;
  const pgp_hyp* pool;
  const double* syms;        // 9 doubles per matrix, row-major
  double max_d2, min_tr;     // max_dist * max_dist, 1 + 2 cos_angle
  unsigned long long* mask;
};

struct ScanParams {
  const ListDesc* lists;
  int n_lists, k;
  const pgp_hyp* pool;
  const unsigned long long* mask;
  pgp_hyp* out;
  double* poses16;           // may be null
  int32_t* n_kept;           // may be null
  float cP[3];
};

__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }

// trace(R_a^T G), summed left to right in row-major order; a and g hold 9 doubles
__device__ __forceinline__ double frob_dot(const double* a, const double* g) {
  double tr = dmul(a[0], g[0]);
#pragma unroll
  for (int e = 1; e < 9; ++e) tr = dadd(tr, dmul(a[e], g[e]));
  return tr;
}

__global__ void __launch_bounds__(TB) k4d_mask(const MaskParams p) {
  __shared__ float s_T[TB][12];
  __shared__ double s_S[MAX_SYM * 9];
  const int t = threadIdx.x;
  for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    // the list of this tile: the last one whose first tile is <= tile
    int lo = 0, hi = p.n_lists - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (p.lists[mid].tile_lo <= tile) lo = mid; else hi = mid - 1; }
    const ListDesc L = p.lists[lo];
    // (rb, cb), cb >= rb, in row-major order over the upper triangle of nw x nw tiles
    int u = (int)(tile - L.tile_lo), rb = 0;
    while (u >= L.nw - rb) { u -= L.nw - rb; ++rb; }
    const int cb = rb + u;
    __syncthreads();                                   // the previous tile's readers are done with s_T / s_S
    const int jc = cb * TB + t;
    if (jc < L.m) {
      const float* T = p.pool[L.pool_lo + jc].T;
#pragma unroll
      for (int e = 0; e < 12; ++e) s_T[t][e] = T[e];
    }
    for (int e = t; e < L.n_sym * 9; e += TB) s_S[e] = p.syms[(int64_t)L.sym_lo * 9 + e];
    __syncthreads();
    const int i = rb * TB + t;
    if (i >= L.m) continue;
    float a[12];
    const float* Ta = p.pool[L.pool_lo + i].T;
#pragma unroll
    for (int e = 0; e < 12; ++e) a[e] = Ta[e];
    double Ra[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) Ra[3 * r + c] = (double)a[4 * r + c];
    const int jn = min(TB, L.m - cb * TB);
    unsigned long long word = 0ull;
    for (int c = 0; c < jn; ++c) {
      const int j = cb * TB + c;
      if (j <= i) continue;
      const float* b = s_T[c];
      const double dx = __dsub_rn((double)a[3], (double)b[3]);
      const double dy = __dsub_rn((double)a[7], (double)b[7]);
      const double dz = __dsub_rn((double)a[11], (double)b[11]);
      const double d2 = dadd(dadd(dmul(dx, dx), dmul(dy, dy)), dmul(dz, dz));
      if (!(d2 <= p.max_d2)) continue;
      double Rb[9];
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) Rb[3 * r + cc] = (double)b[4 * r + cc];
      bool hit = frob_dot(Ra, Rb) >= p.min_tr;
      for (int s = 0; s < L.n_sym && !hit; ++s) {
        const double* S = s_S + 9 * s;
        double G[9];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int cc = 0; cc < 3; ++cc)
            G[3 * r + cc] = dadd(dadd(dmul(Rb[3 * r], S[cc]), dmul(Rb[3 * r + 1], S[3 + cc])), dmul(Rb[3 * r + 2], S[6 + cc]));
        hit = frob_dot(Ra, G) >= p.min_tr;
      }
      if (hit) word |= 1ull << c;
    }
    p.mask[L.mask_lo + (int64_t)i * L.nw + cb] = word;
  }
}

// Record r copied by lanes 0..15 (4 bytes each), and its camera-frame pose by lanes 0..15 (one entry each): rotation unchanged,
// translation ((t_c + c_P) - R_0 c_Q,0) - ... in pgp_centred_to_pose's order.
__device__ __forceinline__ void write_kept(const ScanParams& p, const ListDesc& L, const pgp_hyp* rec, int64_t slot, int lane) {
  if (lane < 16) reinterpret_cast<uint32_t*>(p.out + slot)[lane] = reinterpret_cast<const uint32_t*>(rec)[lane];
  if (p.poses16 && lane < 16) {
    const int r = lane >> 2, c = lane & 3;
    double v;
    if (r == 3) v = c == 3 ? 1.0 : 0.0;
    else if (c < 3) v = (double)rec->T[4 * r + c];
    else {
      const float cP = r == 0 ? p.cP[0] : (r == 1 ? p.cP[1] : p.cP[2]);     // no dynamic index into the parameter block
      v = dadd((double)rec->T[4 * r + 3], (double)cP);
#pragma unroll
      for (int q = 0; q < 3; ++q) v = __dsub_rn(v, dmul((double)rec->T[4 * r + q], (double)L.cQ[q]));
    }
    p.poses16[16 * slot + lane] = v;
  }
}

__global__ void __launch_bounds__(32 * SCAN_WARPS) k4d_scan(const ScanParams p) {
  const int lane = threadIdx.x & 31;
  const int l = blockIdx.x * SCAN_WARPS + (threadIdx.x >> 5);
  if (l >= p.n_lists) return;
  const ListDesc L = p.lists[l];
  const pgp_hyp* pool = p.pool + L.pool_lo;
  const unsigned long long* mask = p.mask + L.mask_lo;
  unsigned long long rem0 = 0ull, rem1 = 0ull;     // removed words lane and lane + 32
  int kept = 0;
  for (int b = 0; b < L.nw && kept < p.k; ++b) {
    const int i0 = b * 64 + lane, i1 = i0 + 32;
    const unsigned v0 = __ballot_sync(0xffffffffu, i0 < L.m && pool[i0].index >= 0);
    const unsigned v1 = __ballot_sync(0xffffffffu, i1 < L.m && pool[i1].index >= 0);
    const unsigned long long removed = __shfl_sync(0xffffffffu, (b >> 5) ? rem1 : rem0, b & 31);
    unsigned long long cand = (((unsigned long long)v1 << 32) | v0) & ~removed;
    while (cand && kept < p.k) {
      const int bit = __ffsll((long long)cand) - 1;
      const int i = b * 64 + bit;
      write_kept(p, L, pool + i, L.out_lo + kept, lane);
      ++kept;
      const unsigned long long* row = mask + (int64_t)i * L.nw;
      if (lane >= b && lane < L.nw) rem0 |= row[lane];
      if (lane + 32 >= b && lane + 32 < L.nw) rem1 |= row[lane + 32];
      cand &= ~row[b];
      cand &= ~(1ull << bit);
    }
  }
  // padding: index -1 and zeros, identity poses
  for (int s = kept; s < p.k; ++s) {
    const int64_t slot = L.out_lo + s;
    if (lane < 16) reinterpret_cast<uint32_t*>(p.out + slot)[lane] = lane < 2 ? 0xffffffffu : 0u;
    if (p.poses16 && lane < 16) p.poses16[16 * slot + lane] = (lane % 5 == 0) ? 1.0 : 0.0;
  }
  if (p.n_kept && lane == 0) p.n_kept[l] = kept;
}

struct K4dScratch {
  DevBuf tables, mask, pool, out, n_kept;
  StagingRing staging;
  int mask_grid = 0;
  // per model slot: the symmetries of pgp_set_symmetries, row-major 3x3 doubles
  std::vector<double> sym[PGP_MAX_OBJECTS];
};
K4dScratch& scratch_of(pgp_ctx* ctx) {
  if (!ctx->k4d_scratch) ctx->k4d_scratch = new K4dScratch();
  return *static_cast<K4dScratch*>(ctx->k4d_scratch);
}

}  // namespace

void k4d_set_symmetries(pgp_ctx* ctx, int obj, const double* R9, int n) {
  scratch_of(ctx).sym[obj].assign(R9, R9 + (size_t)9 * n);
}

int k4d_distinct_dev(pgp_ctx* ctx, const int32_t* objs, const int64_t* pool_offsets, int n_lists, const pgp_hyp* pool_dev, int k,
                     double max_dist, double cos_angle, pgp_hyp* out_dev, double* poses16_dev, int32_t* n_kept_dev) {
  if (n_lists == 0) return PGP_OK;
  K4dScratch& sc = scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  // host tables: descriptors, then each distinct object's symmetries once
  int sym_lo_of[PGP_MAX_OBJECTS];
  std::fill(sym_lo_of, sym_lo_of + PGP_MAX_OBJECTS, -1);
  int n_mat = 0;
  for (int l = 0; l < n_lists; ++l)
    if (sym_lo_of[objs[l]] < 0) { sym_lo_of[objs[l]] = n_mat; n_mat += (int)(sc.sym[objs[l]].size() / 9); }
  const size_t o_sym = (size_t)n_lists * sizeof(ListDesc), blob = o_sym + (size_t)std::max(n_mat, 1) * 9 * sizeof(double);
  int64_t mask_words = 0, n_tiles = 0;
  for (int l = 0; l < n_lists; ++l) {
    const int64_t m = pool_offsets[l + 1] - pool_offsets[l], nw = (m + 63) / 64;
    mask_words += m * nw;
    n_tiles += nw * (nw + 1) / 2;
  }
  // every reservation before the first queued operation (a growing buffer's cudaFree synchronises the device)
  PGP_CUDA(ctx, sc.tables.reserve(blob));
  PGP_CUDA(ctx, sc.mask.reserve((size_t)mask_words * 8));
  if (!sc.mask_grid) {
    int per_sm = 0;
    PGP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k4d_mask, TB, 0));
    sc.mask_grid = std::max(per_sm, 1) * ctx->sm_count;
  }
  StagingRing::Stage* sg = nullptr;
  PGP_CUDA(ctx, sc.staging.acquire(blob, &sg));
  char* h = static_cast<char*>(sg->host);
  ListDesc* desc = reinterpret_cast<ListDesc*>(h);
  double* syms = reinterpret_cast<double*>(h + o_sym);
  int64_t mask_lo = 0, tile_lo = 0;
  for (int l = 0; l < n_lists; ++l) {
    const int obj = objs[l];
    const int m = (int)(pool_offsets[l + 1] - pool_offsets[l]), nw = (m + 63) / 64;
    ListDesc d{};
    d.pool_lo = pool_offsets[l]; d.mask_lo = mask_lo; d.tile_lo = tile_lo; d.out_lo = (int64_t)l * k;
    d.m = m; d.nw = nw;
    d.sym_lo = sym_lo_of[obj]; d.n_sym = (int)(sc.sym[obj].size() / 9);
    for (int c = 0; c < 3; ++c) d.cQ[c] = ctx->models[obj].cQ[c];
    desc[l] = d;
    mask_lo += (int64_t)m * nw;
    tile_lo += (int64_t)nw * (nw + 1) / 2;
  }
  for (int obj = 0; obj < PGP_MAX_OBJECTS; ++obj)
    if (sym_lo_of[obj] >= 0 && !sc.sym[obj].empty()) std::copy(sc.sym[obj].begin(), sc.sym[obj].end(), syms + 9 * (size_t)sym_lo_of[obj]);
  PGP_CUDA(ctx, StagingRing::upload(sg, sc.tables.p, blob, st));
  const ListDesc* lists = sc.tables.as<ListDesc>();

  MaskParams mp{};
  mp.lists = lists; mp.n_lists = n_lists; mp.n_tiles = n_tiles; mp.pool = pool_dev;
  mp.syms = reinterpret_cast<const double*>(sc.tables.as<char>() + o_sym);
  mp.max_d2 = max_dist * max_dist;
  mp.min_tr = 1.0 + 2.0 * cos_angle;
  mp.mask = sc.mask.as<unsigned long long>();
  k4d_mask<<<(unsigned)std::min<int64_t>(n_tiles, sc.mask_grid), TB, 0, st>>>(mp);
  ctx->launches++;
  ScanParams spp{};
  spp.lists = lists; spp.n_lists = n_lists; spp.k = k; spp.pool = pool_dev; spp.mask = mp.mask;
  spp.out = out_dev; spp.poses16 = poses16_dev; spp.n_kept = n_kept_dev;
  for (int c = 0; c < 3; ++c) spp.cP[c] = ctx->scene.cP[c];
  k4d_scan<<<(unsigned)((n_lists + SCAN_WARPS - 1) / SCAN_WARPS), 32 * SCAN_WARPS, 0, st>>>(spp);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

// The host form: the pool up, one list, the kept records and their count down, one synchronisation.
int k4d_distinct_host(pgp_ctx* ctx, int obj, const pgp_hyp* pool_host, int m, int k, double max_dist, double cos_angle, pgp_hyp* out_host) {
  K4dScratch& sc = scratch_of(ctx);
  PGP_CUDA(ctx, sc.pool.reserve((size_t)m * sizeof(pgp_hyp)));
  PGP_CUDA(ctx, sc.out.reserve((size_t)k * sizeof(pgp_hyp)));
  PGP_CUDA(ctx, sc.n_kept.reserve(4));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.pool.p, pool_host, (size_t)m * sizeof(pgp_hyp), cudaMemcpyHostToDevice, ctx->stream));
  const int64_t offs[2] = {0, m};
  int rc = k4d_distinct_dev(ctx, &obj, offs, 1, sc.pool.as<pgp_hyp>(), k, max_dist, cos_angle, sc.out.as<pgp_hyp>(), nullptr, sc.n_kept.as<int32_t>());
  if (rc) return rc;
  int32_t n = 0;
  std::vector<pgp_hyp> tmp((size_t)k);
  PGP_CUDA(ctx, cudaMemcpyAsync(&n, sc.n_kept.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(tmp.data(), sc.out.p, (size_t)k * sizeof(pgp_hyp), cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  std::copy(tmp.begin(), tmp.begin() + n, out_host);
  return n;
}

void k4d_release(pgp_ctx* ctx) {
  if (!ctx->k4d_scratch) return;
  K4dScratch* sc = static_cast<K4dScratch*>(ctx->k4d_scratch);
  for (DevBuf* b : {&sc->tables, &sc->mask, &sc->pool, &sc->out, &sc->n_kept}) b->release();
  sc->staging.release();
  delete sc;
  ctx->k4d_scratch = nullptr;
}
