// K8 -- rendered-depth cost of MCTS states: the placed objects' meshes rasterized at their poses and compared with the observed
// depth frame (UCTState::render + UCTState::computeCost, PPE/src/hypothesis_verification/mcts/UCTState.cpp:93-116; renderer
// depth_sim/src/renderScene.cpp:36-84).  RESTATED, PARITY UNPINNED: the reference renders with OpenGL (a pcl::simulation fork)
// and computeCost's formula is not available; K8 follows its own exact contract (include/pgp.h, DESIGN.md 3), restated in numpy
// in oracle/render_port.py and matched bit for bit.
//
// One device pipeline for pgp_depth_cost_dev, pgp_render_depth_dev, pgp_depth_cost and pgp_render_depth, queued on the context's
// stream with no host stop:
//   k8_ingest  per placed object: pose -> fp32 3x4, finiteness (status PGP_E_INVALID)
//   k8_clear   render mode: every frame of the call emptied, only when the status is still PGP_OK
// then per chunk of states, the chunks cut on the host from the mesh sizes alone and queued back to back on the same scratch:
//   k8_vertex  per (state, slot, vertex): transform, project, snap to 1/256 px
//   k8_setup   per triangle: cull, orient, pixel bounding box clipped to the image, count its (state, 16x16 tile) bins; the chunk's
//              and each state's (triangle, tile) pairs summed on the device
//   scan -> k8_list (non-empty bins, their number on the device) -> k8_fill (bin lists, when the chunk's pairs fit the entries
//              reserved for it; otherwise status PGP_E_CAPACITY and the chunk's fill and tiles do nothing)
//   k8_tiles   a persistent grid that takes the non-empty (state, tile) bins in turn: 64-bit (depth bits, slot) z-buffer in shared
//              memory with atomicMin, then either the tile written out to its state's frame (render mode) or the fused comparison
//              with the observation, summed per slot in shared memory and added to the state's records.
// and k8_finish copies the counts out when the status is PGP_OK.  The host forms upload, run the pipeline, download and synchronise
// once; on PGP_E_CAPACITY they re-cut the chunks from the per-state pair counts the device wrote and run again.
// Work scales with triangles and covered tiles; in the cost mode no per-state frame reaches HBM.  Every count is an integer and every
// depth is a deterministic function of one triangle and one sample, so results depend neither on scheduling nor on chunking.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "pgp_internal.cuh"

namespace {

constexpr int TILE = 16;                       // tile side in pixels; k8_tiles runs one thread per pixel of a tile
constexpr int TT = TILE * TILE;
constexpr int T = 256;                         // threads of the per-vertex / per-triangle passes
constexpr int SMALL = 16;                      // a triangle whose box covers at most this many pixels of a tile is rasterized by one thread
constexpr int64_t CHUNK_TRIS = 1 << 21;        // triangles per chunk (a single state above this is its own chunk)
constexpr int64_t CHUNK_VERTS = 1 << 21;
constexpr int64_t CHUNK_KEYS = 1 << 22;        // (state, tile) bins per chunk
constexpr int64_t CHUNK_PAIRS = 1 << 25;       // (triangle, tile) entries reserved for a chunk
constexpr int64_t MAX_PAIRS = (1ll << 31) - 1; // ... and the most a re-run gives one state alone
constexpr float GUARD = 1048576.f;             // 2^20 px

struct Inst {                                  // one placed object of the call
  const float* T;                              // its pose as fp32 3x4 (k8_ingest)
  const float* v;
  const int32_t* t;
  int64_t vbase, tbase;                        // its first vertex / triangle in the call
  int state, slot;                             // state of the call, position in the state
};

struct __align__(16) Tri {                     // a triangle after setup (slot < 0: culled)
  int x[3], y[3];                              // snapped, oriented: A > 0
  int slot, state;                             // state: of the chunk
  short c0, c1, r0, r1;                        // covered pixel box, clipped to the image
  double iz[3];
};
static_assert(sizeof(Tri) == 64, "Tri is one 64-byte record");

__device__ __forceinline__ int find_inst(const Inst* __restrict__ in, int n, int64_t id, bool tri) {
  int lo = 0, hi = n - 1;                      // last instance whose base <= id
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((tri ? in[mid].tbase : in[mid].vbase) <= id) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// every pose to fp32 3x4; a NaN or Inf entry anywhere sets *status = PGP_E_INVALID (PGP_OK was stored before the launch)
__global__ void __launch_bounds__(T) k8_ingest(const double* __restrict__ poses16, int64_t n, float* __restrict__ pose12, int32_t* __restrict__ status) {
  bool ok = true;
  for (int64_t i = blockIdx.x * (int64_t)T + threadIdx.x; i < n; i += (int64_t)gridDim.x * T) {
    double P[16];
    for (int k = 0; k < 16; ++k) { P[k] = poses16[16 * i + k]; ok &= isfinite(P[k]); }
    pose16_to_f32x12(P, pose12 + 12 * i);
  }
  if (!ok) *status = PGP_E_INVALID;
}

// render mode: the call's n frame pixels emptied (depth 0.0f, slot -1: nothing; slot nullptr: no slot frames), queued after k8_ingest
// so that a call whose poses it refused writes no frame; k8_tiles then writes the pixels of every non-empty tile
__global__ void __launch_bounds__(T) k8_clear(size_t n, float* __restrict__ depth, int* __restrict__ slot, const int32_t* __restrict__ status) {
  if (*status != PGP_OK) return;
  for (size_t i = blockIdx.x * (size_t)T + threadIdx.x; i < n; i += (size_t)gridDim.x * T) {
    depth[i] = 0.f;
    if (slot) slot[i] = -1;
  }
}

// vertex v0 + i of the call -> {snapped x, snapped y, Z bits, ok} at i
__global__ void __launch_bounds__(T) k8_vertex(const Inst* __restrict__ inst, int n_inst, int64_t v0, int n_vert, float fx, float fy, float cx,
                                               float cy, int4* __restrict__ out, const int32_t* __restrict__ status) {
  const int v = blockIdx.x * T + threadIdx.x;
  if (v >= n_vert || *status == PGP_E_INVALID) return;
  const Inst& I = inst[find_inst(inst, n_inst, v0 + v, false)];
  const float* p = I.v + 3 * (v0 + v - I.vbase);
  const float* M = I.T;
  const float x = p[0], y = p[1], z = p[2];
  const float X = xf_row(M[0], M[1], M[2], M[3], x, y, z);
  const float Y = xf_row(M[4], M[5], M[6], M[7], x, y, z);
  const float Z = xf_row(M[8], M[9], M[10], M[11], x, y, z);
  bool ok = isfinite(X) && isfinite(Y) && isfinite(Z) && Z > 0.1f;
  const float sx = __fadd_rn(__fdiv_rn(__fmul_rn(fx, X), Z), cx);
  const float sy = __fadd_rn(__fdiv_rn(__fmul_rn(fy, Y), Z), cy);
  ok = ok && fabsf(sx) <= GUARD && fabsf(sy) <= GUARD;
  int4 r = make_int4(0, 0, __float_as_int(Z), 0);
  if (ok) { r.x = (int)__float2ll_rn(__fmul_rn(sx, 256.f)); r.y = (int)__float2ll_rn(__fmul_rn(sy, 256.f)); r.w = 1; }
  out[v] = r;
}

__device__ __forceinline__ long long edge_fn(int ax, int ay, int bx, int by, int px, int py) {
  return (long long)(bx - ax) * (long long)(py - ay) - (long long)(by - ay) * (long long)(px - ax);
}
__device__ __forceinline__ bool owns(long long e, int ax, int ay, int bx, int by) {
  const int dx = bx - ax, dy = by - ay;
  return e > 0 || (e == 0 && (dy < 0 || (dy == 0 && dx > 0)));
}

// triangle t0 + i of the call (chunk: vertices from v0, states from s0) -> record + bin counts, the chunk's pair total and the
// pair count of each state of the call
__global__ void __launch_bounds__(T) k8_setup(const Inst* __restrict__ inst, int n_inst, int64_t v0, int64_t t0, int s0, int n_tri,
                                              const int4* __restrict__ vtx, int rows, int cols, int ntx, int ntiles, Tri* __restrict__ tris,
                                              uint32_t* __restrict__ cnt, unsigned long long* __restrict__ pair_total,
                                              unsigned long long* __restrict__ state_pairs, const int32_t* __restrict__ status) {
  if (*status == PGP_E_INVALID) return;
  const int t = blockIdx.x * T + threadIdx.x;
  uint32_t pairs = 0;
  int state = -1;
  if (t < n_tri) {
    const Inst& I = inst[find_inst(inst, n_inst, t0 + t, true)];
    const int32_t* ix = I.t + 3 * (t0 + t - I.tbase);
    const int4* vb = vtx + (I.vbase - v0);
    int4 a = vb[ix[0]], b = vb[ix[1]], c = vb[ix[2]];
    state = I.state;
    Tri r;
    r.slot = -1;
    if (a.w && b.w && c.w) {
      const long long area = edge_fn(a.x, a.y, b.x, b.y, c.x, c.y);
      if (area < 0) { const int4 s = b; b = c; c = s; }
      const int mnx = min(a.x, min(b.x, c.x)), mxx = max(a.x, max(b.x, c.x));
      const int mny = min(a.y, min(b.y, c.y)), mxy = max(a.y, max(b.y, c.y));
      const int c0 = max((mnx + 255) >> 8, 0), c1 = min(mxx >> 8, cols - 1);      // samples at c * 256 within [mnx, mxx]
      const int r0 = max((mny + 255) >> 8, 0), r1 = min(mxy >> 8, rows - 1);
      if (area != 0 && c0 <= c1 && r0 <= r1) {
        r.x[0] = a.x; r.y[0] = a.y; r.x[1] = b.x; r.y[1] = b.y; r.x[2] = c.x; r.y[2] = c.y;
        r.slot = I.slot; r.state = I.state - s0;
        r.c0 = (short)c0; r.c1 = (short)c1; r.r0 = (short)r0; r.r1 = (short)r1;
        r.iz[0] = __ddiv_rn(1.0, (double)__int_as_float(a.z));
        r.iz[1] = __ddiv_rn(1.0, (double)__int_as_float(b.z));
        r.iz[2] = __ddiv_rn(1.0, (double)__int_as_float(c.z));
        const int tx0 = c0 / TILE, tx1 = c1 / TILE, ty0 = r0 / TILE, ty1 = r1 / TILE;
        uint32_t* base = cnt + (size_t)(I.state - s0) * ntiles;
        for (int ty = ty0; ty <= ty1; ++ty)
          for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(base + ty * ntx + tx, 1u);
        pairs = (uint32_t)((tx1 - tx0 + 1) * (ty1 - ty0 + 1));
      }
    }
    tris[t] = r;
  }
  // a warp's triangles nearly always belong to one state: one atomic per warp then (lane 0 holds the warp's first triangle)
  const uint32_t w = __reduce_add_sync(0xffffffffu, pairs);      // <= 32 x 2^20: no wrap
  const int first = __shfl_sync(0xffffffffu, state, 0);
  const bool one_state = __all_sync(0xffffffffu, pairs == 0 || state == first);
  if ((threadIdx.x & 31) == 0 && w) {
    atomicAdd(pair_total, (unsigned long long)w);
    if (one_state) atomicAdd(state_pairs + first, (unsigned long long)w);
  }
  if (!one_state && pairs) atomicAdd(state_pairs + state, (unsigned long long)pairs);
}

// the bin lists, when the chunk's pairs fit the cap entries of bins; otherwise nothing, and the status becomes PGP_E_CAPACITY
__global__ void __launch_bounds__(T) k8_fill(const Tri* __restrict__ tris, int n_tri, int ntx, int ntiles, uint32_t* __restrict__ cursor,
                                             uint32_t* __restrict__ bins, const unsigned long long* __restrict__ pair_total, int64_t cap,
                                             int32_t* __restrict__ status) {
  const bool over = *pair_total > (unsigned long long)cap;
  if (*status != PGP_OK || over) {
    if (over && blockIdx.x == 0 && threadIdx.x == 0 && *status == PGP_OK) *status = PGP_E_CAPACITY;    // the only writer of this launch
    return;
  }
  const int t = blockIdx.x * T + threadIdx.x;
  if (t >= n_tri) return;
  const Tri& r = tris[t];
  if (r.slot < 0) return;
  uint32_t* base = cursor + (size_t)r.state * ntiles;
  for (int ty = r.r0 / TILE; ty <= r.r1 / TILE; ++ty)
    for (int tx = r.c0 / TILE; tx <= r.c1 / TILE; ++tx) bins[atomicAdd(base + ty * ntx + tx, 1u)] = (uint32_t)t;
}

__global__ void __launch_bounds__(T) k8_list(const uint32_t* __restrict__ off, int n_keys, uint32_t* __restrict__ list, uint32_t* __restrict__ n_list) {
  const int k = blockIdx.x * T + threadIdx.x;
  if (k < n_keys && off[k + 1] != off[k]) list   // != : a count below 2^32 is non-zero mod 2^32 even where the scan wrapped
   [atomicAdd(n_list, 1u)] = (uint32_t)k;
}

// coverage + depth of sample (c, r) for one triangle; keeps the smaller key
__device__ __forceinline__ void shade(const Tri& t, int c, int r, unsigned long long* zpix) {
  const int px = c << 8, py = r << 8;
  const long long e0 = edge_fn(t.x[1], t.y[1], t.x[2], t.y[2], px, py);
  if (!owns(e0, t.x[1], t.y[1], t.x[2], t.y[2])) return;
  const long long e1 = edge_fn(t.x[2], t.y[2], t.x[0], t.y[0], px, py);
  if (!owns(e1, t.x[2], t.y[2], t.x[0], t.y[0])) return;
  const long long e2 = edge_fn(t.x[0], t.y[0], t.x[1], t.y[1], px, py);
  if (!owns(e2, t.x[0], t.y[0], t.x[1], t.y[1])) return;
  const double den = __dadd_rn(__dadd_rn(__dmul_rn((double)e0, t.iz[0]), __dmul_rn((double)e1, t.iz[1])), __dmul_rn((double)e2, t.iz[2]));
  const float d = __double2float_rn(__ddiv_rn((double)(e0 + e1 + e2), den));
  atomicMin(zpix, ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)t.slot);
}

struct Obs {
  const float* depth;                          // decoded
  const uint8_t* mask;                         // nullptr: no class mask
  int rows, cols;
};

// The chunk's counters on the device (K8Scratch::misc): zeroed before the chunk's first launch.
struct ChunkCounters {
  unsigned long long pairs;                    // (triangle, tile) pairs
  uint32_t n_list;                             // non-empty bins
  uint32_t next;                               // the next bin k8_tiles takes
};

// A persistent grid: each CTA takes the next non-empty bin (list position from counters->next) until none is left, and resets its
// z-buffer, queue and accumulators per bin.  RENDER: write the tile into frame key / ntiles of depth_out / slot_out (the chunk's
// first frame; slot_out nullptr: no slot frames);  else: compare with the observation and add the per-slot counts to out.  Nothing
// when the status is not PGP_OK (an earlier refusal, or this chunk's bins did not fit).
template <bool RENDER>
__global__ void __launch_bounds__(TT) k8_tiles(const Tri* __restrict__ tris, const uint32_t* __restrict__ off, const uint32_t* __restrict__ bins,
                                               const uint32_t* __restrict__ list, ChunkCounters* __restrict__ counters, int ntx, int ntiles,
                                               Obs obs, float tau, const int* __restrict__ state_first, const int* __restrict__ rec_cls,
                                               int* __restrict__ out, float* __restrict__ depth_out, int* __restrict__ slot_out,
                                               const int32_t* __restrict__ status) {
  __shared__ unsigned long long z[TT];
  __shared__ uint32_t queue[TT];
  __shared__ int qn;
  __shared__ int acc[RENDER ? 1 : PGP_MAX_OBJECTS * 5];
  __shared__ uint32_t s_key;
  __shared__ int org[2];                       // the tile's first column and row (read from shared memory: kept out of the registers
                                               // that must survive the double divisions' calls, which would spill them)
  volatile int* vorg = org;
  volatile uint32_t* vkey = &s_key;
  const int tid = threadIdx.x;
  if (*status != PGP_OK) return;
  for (;;) {
    __syncthreads();                                                 // the previous bin is done with the shared state
    if (tid == 0) {
      const uint32_t i = atomicAdd(&counters->next, 1u);
      const uint32_t key = i < counters->n_list ? list[i] : ~0u;
      const int tile = (int)(key % (uint32_t)ntiles);
      s_key = key; qn = 0; org[0] = (tile % ntx) * TILE; org[1] = (tile / ntx) * TILE;
    }
    z[tid] = ~0ull;
    if (!RENDER)
      for (int i = tid; i < PGP_MAX_OBJECTS * 5; i += TT) acc[i] = 0;
    __syncthreads();
    const uint32_t key = *vkey;
    if (key == ~0u) return;
    const uint32_t b0 = off[key], b1 = off[key + 1];
    for (uint32_t base = b0; base < b1; base += TT) {
      if (base + tid < b1) {
        const uint32_t id = bins[base + tid];
        const Tri& t = tris[id];
        const int cl = vorg[0], rl = vorg[1];
        const int c0 = max((int)t.c0, cl), c1 = min((int)t.c1, cl + TILE - 1), r0 = max((int)t.r0, rl), r1 = min((int)t.r1, rl + TILE - 1);
        if ((c1 - c0 + 1) * (r1 - r0 + 1) <= SMALL) {
          for (int r = r0; r <= r1; ++r)
            for (int c = c0; c <= c1; ++c) shade(t, c, r, &z[(r - vorg[1]) * TILE + (c - vorg[0])]);
        } else {
          queue[atomicAdd(&qn, 1)] = id;
        }
      }
      __syncthreads();
      const int nq = qn;
      for (int j = 0; j < nq; ++j) {                                 // larger triangles: the whole CTA, one pixel per thread
        const Tri& t = tris[queue[j]];
        const int mc = vorg[0] + (tid % TILE), mr = vorg[1] + (tid / TILE);
        if (mc >= t.c0 && mc <= t.c1 && mr >= t.r0 && mr <= t.r1) shade(t, mc, mr, &z[tid]);
      }
      __syncthreads();
      if (tid == 0) qn = 0;
      __syncthreads();
    }
    const int mc = vorg[0] + (tid % TILE), mr = vorg[1] + (tid / TILE);   // this thread's pixel
    const bool in_img = mr < obs.rows && mc < obs.cols;
    const unsigned long long k = z[tid];
    const size_t p = (size_t)mr * obs.cols + mc;
    if (RENDER) {
      if (in_img) {
        const size_t q = (size_t)(*vkey / (uint32_t)ntiles) * ((size_t)obs.rows * obs.cols) + p;
        depth_out[q] = k == ~0ull ? 0.f : __uint_as_float((unsigned)(k >> 32));
        if (slot_out) slot_out[q] = k == ~0ull ? -1 : (int)(unsigned)k;
      }
      continue;
    }
    const int first = state_first[*vkey / (uint32_t)ntiles];
    if (in_img && k != ~0ull) {
      const int slot = (int)(unsigned)k;
      const float r = __uint_as_float((unsigned)(k >> 32));
      int* a = acc + 5 * slot;
      atomicAdd(a + 0, 1);
      const float o = obs.depth[p];
      if (depth_valid(o)) {
        if (fabsf(__fsub_rn(r, o)) <= tau) atomicAdd(a + 1, 1);
        else if (__fsub_rn(o, r) > tau) atomicAdd(a + 2, 1);
        else atomicAdd(a + 3, 1);                                    // r - o > tau
      }
      if (obs.mask && (int)obs.mask[p] == rec_cls[first + slot]) atomicAdd(a + 4, 1);
    }
    __syncthreads();
    for (int i = tid; i < PGP_MAX_OBJECTS * 5; i += TT)
      if (acc[i]) atomicAdd(out + 5 * (size_t)(first + i / 5) + i % 5, acc[i]);
  }
}

// the call's counts to the caller's buffer, only when every chunk ran (status PGP_OK)
__global__ void __launch_bounds__(T) k8_finish(const int* __restrict__ counts, int64_t n, int* __restrict__ out, const int32_t* __restrict__ status) {
  if (*status != PGP_OK) return;
  for (int64_t i = blockIdx.x * (int64_t)T + threadIdx.x; i < n; i += (int64_t)gridDim.x * T) out[i] = counts[i];
}

// the observation decoded once per frame (K7's decode), and the pixels of each label with valid depth (hist: nullptr = not wanted)
__global__ void __launch_bounds__(T) k8_observe(const uint16_t* __restrict__ raw, const uint8_t* __restrict__ mask, int n, float* __restrict__ depth,
                                                unsigned long long* __restrict__ hist) {
  __shared__ unsigned int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  for (int i = blockIdx.x * T + threadIdx.x; i < n; i += gridDim.x * T) {
    const float d = decode_depth(raw[i]);
    depth[i] = d;
    if (hist && depth_valid(d)) atomicAdd(&h[mask[i]], 1u);
  }
  __syncthreads();
  if (hist && h[threadIdx.x]) atomicAdd(hist + threadIdx.x, (unsigned long long)h[threadIdx.x]);
}

struct Mesh { DevBuf v, t; int nv = 0, nt = 0, cls = -1; };
// Device scratch of K8, owned by the context.  The pipeline adds pose12 (the fp32 poses), tables (the host-built instance, state and
// class tables, uploaded once per call from pinned staging), state_pairs (each state's (triangle, tile) pairs), and the host forms'
// copies of their poses (raw_poses) and status word.
struct K8Scratch {
  Mesh mesh[PGP_MAX_OBJECTS];
  DevBuf raw, depth, mask;                     // observation: as given, decoded, labels
  int rows = 0, cols = 0;
  bool has_obs = false, has_mask = false;
  float fx = 0, fy = 0, cx = 0, cy = 0;
  DevBuf tables, pose12, state_pairs, raw_poses, status, vtx, tris, cnt, cursor, bins, list, misc, out, frame_d, frame_s;
  StagingRing staging;
  int tiles_grid[2] = {0, 0};                  // k8_tiles<false>, <true>: resident CTAs on the whole GPU
};
K8Scratch& k8_scratch_of(pgp_ctx* ctx) {
  if (!ctx->k8_scratch) ctx->k8_scratch = new K8Scratch();
  return *static_cast<K8Scratch*>(ctx->k8_scratch);
}

struct Chunk { int s, e; int64_t cap; };       // states [s, e) and the (triangle, tile) entries reserved for them

int64_t ntiles_of(const K8Scratch& sc) { return (int64_t)((sc.cols + TILE - 1) / TILE) * ((sc.rows + TILE - 1) / TILE); }

// Chunks of whole states (a state's z-test needs all of its objects) by triangles, vertices and bins; with pairs (each state's
// (triangle, tile) pairs, read back after a PGP_E_CAPACITY), also by pairs, each chunk reserving exactly what it needs.
int cut_chunks(pgp_ctx* ctx, const K8Scratch& sc, const int64_t* offs, int n_states, const int32_t* obj_ids, const unsigned long long* pairs,
               std::vector<Chunk>& chunks) {
  const int64_t ntiles = ntiles_of(sc);
  chunks.clear();
  for (int s = 0; s < n_states;) {
    int64_t tris = 0, verts = 0, np = 0;
    int e = s;
    while (e < n_states) {
      int64_t t = 0, v = 0;
      for (int64_t i = offs[e]; i < offs[e + 1]; ++i) { t += sc.mesh[obj_ids[i]].nt; v += sc.mesh[obj_ids[i]].nv; }
      const int64_t p = pairs ? (int64_t)pairs[e] : 0;
      if (e > s && (tris + t > CHUNK_TRIS || verts + v > CHUNK_VERTS || (e - s + 1) * ntiles > CHUNK_KEYS || np + p > CHUNK_PAIRS)) break;
      tris += t; verts += v; np += p; ++e;
    }
    if (np > MAX_PAIRS) return pgp_fail(ctx, PGP_E_TOO_LARGE, "one state covers %lld (triangle, tile) pairs", (long long)np);
    if (offs[e] > offs[s]) chunks.push_back(Chunk{s, e, pairs ? np : std::min<int64_t>(CHUNK_PAIRS, tris * ntiles)});
    s = e;
  }
  return PGP_OK;
}

// The device pipeline of one call, queued on ctx->stream (see the top of the file): the records of offs[0 .. n_states] with their
// poses in device memory (poses16), the given chunks.  *status: PGP_OK, PGP_E_INVALID (a pose entry is not finite; nothing runs)
// or PGP_E_CAPACITY (a chunk's pairs exceeded its reservation; its fill and tiles and those of every later chunk did nothing).
// Counts: summed in sc.out, then copied to out_dev when the status is PGP_OK (out_dev nullptr: left in sc.out).  Render mode
// (frame_d not nullptr): state s's frame to frame_d / frame_s + s x rows x cols (frame_s nullptr: no slot frames), and no counts.
// Makes no host synchronisation once the scratch has grown to the call's size.
int run_pipeline(pgp_ctx* ctx, K8Scratch& sc, const int64_t* offs, int n_states, const int32_t* obj_ids, const double* poses16, float tau,
                 const std::vector<Chunk>& chunks, int* out_dev, float* frame_d, int* frame_s, int32_t* status) {
  cudaStream_t st = ctx->stream;
  const bool render = frame_d != nullptr;
  const int ntx = (sc.cols + TILE - 1) / TILE, ntiles = (int)ntiles_of(sc);
  const int64_t n_rec = n_states > 0 ? offs[n_states] : 0;
  // sizes: every reservation before the first launch (a growing buffer's cudaFree synchronises the device)
  int64_t max_v = 0, max_t = 0, max_keys = 0, max_cap = 0;
  for (const Chunk& c : chunks) {
    int64_t v = 0, t = 0;
    for (int64_t i = offs[c.s]; i < offs[c.e]; ++i) { v += sc.mesh[obj_ids[i]].nv; t += sc.mesh[obj_ids[i]].nt; }
    max_v = std::max(max_v, v); max_t = std::max(max_t, t);
    max_keys = std::max(max_keys, (int64_t)(c.e - c.s) * ntiles); max_cap = std::max(max_cap, c.cap);
  }
  const size_t o_first = (size_t)n_rec * sizeof(Inst), o_cls = o_first + (size_t)n_states * 4, blob = o_cls + (size_t)n_rec * 4;
  const size_t npx = (size_t)sc.rows * sc.cols;
  PGP_CUDA(ctx, sc.pose12.reserve((size_t)n_rec * 48));
  PGP_CUDA(ctx, sc.out.reserve((size_t)n_rec * sizeof(pgp_depth_counts)));
  PGP_CUDA(ctx, sc.state_pairs.reserve((size_t)n_states * 8));
  PGP_CUDA(ctx, sc.tables.reserve(blob));
  PGP_CUDA(ctx, sc.vtx.reserve((size_t)max_v * 16));
  PGP_CUDA(ctx, sc.tris.reserve((size_t)max_t * sizeof(Tri)));
  PGP_CUDA(ctx, sc.cnt.reserve((size_t)(max_keys + 1) * 4));
  PGP_CUDA(ctx, sc.cursor.reserve((size_t)(max_keys + 1) * 4));
  PGP_CUDA(ctx, sc.list.reserve((size_t)max_keys * 4));
  PGP_CUDA(ctx, sc.bins.reserve((size_t)max_cap * 4));
  PGP_CUDA(ctx, sc.misc.reserve(sizeof(ChunkCounters)));
  PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((max_keys + 1) / 2048 + 4096) * 4));
  for (int r = 0; r < 2; ++r)
    if (!sc.tiles_grid[r]) {
      int per_sm = 0;
      PGP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, r ? k8_tiles<true> : k8_tiles<false>, TT, 0));
      sc.tiles_grid[r] = std::max(per_sm, 1) * ctx->sm_count;
    }
  // ingest, then the frames emptied unless a pose was refused
  PGP_CUDA(ctx, cudaMemsetAsync(status, 0, sizeof(int32_t), st));     // PGP_OK
  if (n_rec > 0) {
    k8_ingest<<<(unsigned)std::min<int64_t>((n_rec + T - 1) / T, 4 * ctx->sm_count), T, 0, st>>>(poses16, n_rec, sc.pose12.as<float>(), status);
    ctx->launches++;
  }
  if (render && n_states > 0) {
    const size_t n = (size_t)n_states * npx;
    k8_clear<<<(unsigned)std::min<size_t>((n + T - 1) / T, (size_t)8 * ctx->sm_count), T, 0, st>>>(n, frame_d, frame_s, status);
    ctx->launches++;
  }
  PGP_CUDA(ctx, cudaGetLastError());
  if (n_rec == 0) return PGP_OK;
  PGP_CUDA(ctx, cudaMemsetAsync(sc.out.p, 0, (size_t)n_rec * sizeof(pgp_depth_counts), st));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.state_pairs.p, 0, (size_t)n_states * 8, st));
  // the tables, in one copy from the next pinned buffer: every record's instance, each state's first record, each record's class
  StagingRing::Stage* sg = nullptr;
  PGP_CUDA(ctx, sc.staging.acquire(blob, &sg));
  char* h = static_cast<char*>(sg->host);
  Inst* inst = reinterpret_cast<Inst*>(h);
  int* first = reinterpret_cast<int*>(h + o_first);
  int* cls = reinterpret_cast<int*>(h + o_cls);
  int64_t nvert = 0, ntri = 0;
  for (int q = 0; q < n_states; ++q) {
    first[q] = (int)offs[q];
    for (int64_t i = offs[q]; i < offs[q + 1]; ++i) {
      const Mesh& m = sc.mesh[obj_ids[i]];
      inst[i] = Inst{sc.pose12.as<float>() + 12 * i, m.v.as<float>(), m.t.as<int32_t>(), nvert, ntri, q, (int)(i - offs[q])};
      cls[i] = m.cls;
      nvert += m.nv; ntri += m.nt;
    }
  }
  PGP_CUDA(ctx, StagingRing::upload(sg, sc.tables.p, blob, st));
  const Inst* inst_dev = sc.tables.as<Inst>();
  const int* first_dev = reinterpret_cast<const int*>(sc.tables.as<char>() + o_first);
  const int* cls_dev = reinterpret_cast<const int*>(sc.tables.as<char>() + o_cls);
  ChunkCounters* ctr = sc.misc.as<ChunkCounters>();
  const Obs obs{sc.depth.as<float>(), sc.has_mask ? sc.mask.as<uint8_t>() : nullptr, sc.rows, sc.cols};
  for (const Chunk& c : chunks) {
    const int64_t r0 = offs[c.s], r1 = offs[c.e];
    const Inst& I0 = inst[r0];
    const int64_t v0 = I0.vbase, t0 = I0.tbase;
    const int64_t v1 = r1 < n_rec ? inst[r1].vbase : nvert, t1 = r1 < n_rec ? inst[r1].tbase : ntri;
    const int nv = (int)(v1 - v0), nt = (int)(t1 - t0), n_inst = (int)(r1 - r0), n_keys = (c.e - c.s) * ntiles;
    PGP_CUDA(ctx, cudaMemsetAsync(sc.cnt.p, 0, (size_t)(n_keys + 1) * 4, st));
    PGP_CUDA(ctx, cudaMemsetAsync(ctr, 0, sizeof(ChunkCounters), st));
    k8_vertex<<<(unsigned)((nv + T - 1) / T), T, 0, st>>>(inst_dev + r0, n_inst, v0, nv, sc.fx, sc.fy, sc.cx, sc.cy, sc.vtx.as<int4>(), status);
    k8_setup<<<(unsigned)((nt + T - 1) / T), T, 0, st>>>(inst_dev + r0, n_inst, v0, t0, c.s, nt, sc.vtx.as<int4>(), sc.rows, sc.cols, ntx, ntiles,
                                                         sc.tris.as<Tri>(), sc.cnt.as<uint32_t>(), &ctr->pairs,
                                                         sc.state_pairs.as<unsigned long long>(), status);
    ctx->launches += 2;
    int rc = pgp_scan_exclusive_u32(ctx, sc.cnt.as<uint32_t>(), (int64_t)n_keys + 1, ctx->scene.scratch.as<uint32_t>());
    if (rc) return rc;
    k8_list<<<(unsigned)((n_keys + T - 1) / T), T, 0, st>>>(sc.cnt.as<uint32_t>(), n_keys, sc.list.as<uint32_t>(), &ctr->n_list);
    PGP_CUDA(ctx, cudaMemcpyAsync(sc.cursor.p, sc.cnt.p, (size_t)(n_keys + 1) * 4, cudaMemcpyDeviceToDevice, st));
    k8_fill<<<(unsigned)((nt + T - 1) / T), T, 0, st>>>(sc.tris.as<Tri>(), nt, ntx, ntiles, sc.cursor.as<uint32_t>(), sc.bins.as<uint32_t>(), &ctr->pairs,
                                                        c.cap, status);
    const unsigned grid = (unsigned)std::min<int64_t>(sc.tiles_grid[render], n_keys);
    if (render)
      k8_tiles<true><<<grid, TT, 0, st>>>(sc.tris.as<Tri>(), sc.cnt.as<uint32_t>(), sc.bins.as<uint32_t>(), sc.list.as<uint32_t>(), ctr, ntx, ntiles,
                                          obs, tau, first_dev + c.s, cls_dev, nullptr, frame_d + (size_t)c.s * npx,
                                          frame_s ? frame_s + (size_t)c.s * npx : nullptr, status);
    else
      k8_tiles<false><<<grid, TT, 0, st>>>(sc.tris.as<Tri>(), sc.cnt.as<uint32_t>(), sc.bins.as<uint32_t>(), sc.list.as<uint32_t>(), ctr, ntx, ntiles,
                                           obs, tau, first_dev + c.s, cls_dev, sc.out.as<int>(), nullptr, nullptr, status);
    ctx->launches += 3;
    PGP_CUDA(ctx, cudaGetLastError());
  }
  if (out_dev) {
    const int64_t n = n_rec * 5;
    k8_finish<<<(unsigned)std::min<int64_t>((n + T - 1) / T, 4 * ctx->sm_count), T, 0, st>>>(sc.out.as<int>(), n, out_dev, status);
    ctx->launches++;
    PGP_CUDA(ctx, cudaGetLastError());
  }
  return PGP_OK;
}

// The host forms: the poses up, the pipeline, the results down (fetch: queues their copies), one synchronisation.  When a chunk's
// pairs did not fit, the per-state pair counts come back and the pipeline runs again on chunks cut to fit them.
template <class Fetch>
int run_host(pgp_ctx* ctx, K8Scratch& sc, const int64_t* offs, int n_states, const int32_t* obj_ids, const double* poses16, float tau,
             float* frame_d, int* frame_s, Fetch fetch) {
  cudaStream_t st = ctx->stream;
  const int64_t n_rec = n_states > 0 ? offs[n_states] : 0;
  PGP_CUDA(ctx, sc.raw_poses.reserve((size_t)n_rec * 128));
  PGP_CUDA(ctx, sc.status.reserve(sizeof(int32_t)));
  if (n_rec) PGP_CUDA(ctx, cudaMemcpyAsync(sc.raw_poses.p, poses16, (size_t)n_rec * 128, cudaMemcpyHostToDevice, st));
  std::vector<Chunk> chunks;
  std::vector<unsigned long long> pairs;
  for (int pass = 0;; ++pass) {
    int rc = cut_chunks(ctx, sc, offs, n_states, obj_ids, pass ? pairs.data() : nullptr, chunks);
    if (!rc) rc = run_pipeline(ctx, sc, offs, n_states, obj_ids, sc.raw_poses.as<double>(), tau, chunks, nullptr, frame_d, frame_s, sc.status.as<int32_t>());
    if (rc) return rc;
    int32_t status = PGP_OK;
    PGP_CUDA(ctx, cudaMemcpyAsync(&status, sc.status.p, sizeof(status), cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, fetch());
    PGP_CUDA(ctx, cudaStreamSynchronize(st));
    if (status == PGP_OK) return PGP_OK;
    if (status != PGP_E_CAPACITY || pass) return pgp_fail(ctx, PGP_E_CUDA, "K8: device status %d", status);
    pairs.resize((size_t)n_states);
    PGP_CUDA(ctx, cudaMemcpyAsync(pairs.data(), sc.state_pairs.p, (size_t)n_states * 8, cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaStreamSynchronize(st));
  }
}

// the observation's frame size, intrinsics and mask flag, once its decode and mask are queued
void observed(K8Scratch& sc, int rows, int cols, const float* K9, bool has_mask) {
  sc.rows = rows; sc.cols = cols;
  sc.fx = K9[0]; sc.fy = K9[4]; sc.cx = K9[2]; sc.cy = K9[5];
  sc.has_mask = has_mask;
  sc.has_obs = true;
}

}  // namespace

bool k8_has_mesh(pgp_ctx* ctx, int obj) { return ctx->k8_scratch && k8_scratch_of(ctx).mesh[obj].nt > 0; }
bool k8_has_observation(pgp_ctx* ctx) { return ctx->k8_scratch && k8_scratch_of(ctx).has_obs; }

int k8_set_mesh(pgp_ctx* ctx, int obj, const float* vert_xyz, int nv, const int32_t* tri3, int nt, int class_id) {
  K8Scratch& sc = k8_scratch_of(ctx);
  Mesh& m = sc.mesh[obj];
  m.nt = 0;                                    // no mesh until both uploads are queued
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // a pending call may still read the old buffers
  PGP_CUDA(ctx, m.v.reserve((size_t)nv * 12));
  PGP_CUDA(ctx, m.t.reserve((size_t)nt * 12));
  PGP_CUDA(ctx, cudaMemcpyAsync(m.v.p, vert_xyz, (size_t)nv * 12, cudaMemcpyHostToDevice, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(m.t.p, tri3, (size_t)nt * 12, cudaMemcpyHostToDevice, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  m.nv = nv; m.nt = nt; m.cls = class_id;
  return PGP_OK;
}

int k8_set_observation(pgp_ctx* ctx, const uint16_t* depth_raw, const uint8_t* class_mask, int rows, int cols, const float* K9,
                       int64_t* class_pixels_out) {
  K8Scratch& sc = k8_scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  const int npx = rows * cols;
  sc.has_obs = false;
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  PGP_CUDA(ctx, sc.raw.reserve((size_t)npx * 2));
  PGP_CUDA(ctx, sc.depth.reserve((size_t)npx * 4));
  PGP_CUDA(ctx, sc.misc.reserve(256 * 8));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.raw.p, depth_raw, (size_t)npx * 2, cudaMemcpyHostToDevice, st));
  if (class_mask) {
    PGP_CUDA(ctx, sc.mask.reserve((size_t)npx));
    PGP_CUDA(ctx, cudaMemcpyAsync(sc.mask.p, class_mask, (size_t)npx, cudaMemcpyHostToDevice, st));
  }
  const bool hist_wanted = class_mask && class_pixels_out;
  PGP_CUDA(ctx, cudaMemsetAsync(sc.misc.p, 0, 256 * 8, st));
  k8_observe<<<std::min((npx + T - 1) / T, ctx->sm_count * 4), T, 0, st>>>(sc.raw.as<uint16_t>(), sc.mask.as<uint8_t>(), npx, sc.depth.as<float>(),
                                                                           hist_wanted ? sc.misc.as<unsigned long long>() : nullptr);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  unsigned long long hist[256] = {0};
  if (hist_wanted) PGP_CUDA(ctx, cudaMemcpyAsync(hist, sc.misc.p, sizeof(hist), cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  if (class_pixels_out) for (int i = 0; i < 256; ++i) class_pixels_out[i] = (int64_t)hist[i];
  observed(sc, rows, cols, K9, class_mask != nullptr);
  return PGP_OK;
}

// k8_set_observation on device data, queued on ctx->stream with no synchronisation: the caller's raw depth decoded straight into the
// context's frame and its mask copied into the context's buffer (later calls read them), so the caller's buffers are read only by
// work ordered at this call.  A call queued earlier on the stream still reads the observation it was queued with.
int k8_set_observation_dev(pgp_ctx* ctx, const uint16_t* depth_raw_dev, const uint8_t* class_mask_dev, int rows, int cols, const float* K9,
                           int64_t* class_pixels_dev) {
  K8Scratch& sc = k8_scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  const int npx = rows * cols;
  unsigned long long* hist = reinterpret_cast<unsigned long long*>(class_pixels_dev);
  sc.has_obs = false;
  PGP_CUDA(ctx, sc.depth.reserve((size_t)npx * 4));
  if (class_mask_dev) {
    PGP_CUDA(ctx, sc.mask.reserve((size_t)npx));
    PGP_CUDA(ctx, cudaMemcpyAsync(sc.mask.p, class_mask_dev, (size_t)npx, cudaMemcpyDeviceToDevice, st));
  }
  if (hist) PGP_CUDA(ctx, cudaMemsetAsync(hist, 0, 256 * 8, st));
  k8_observe<<<std::min((npx + T - 1) / T, ctx->sm_count * 4), T, 0, st>>>(depth_raw_dev, sc.mask.as<uint8_t>(), npx, sc.depth.as<float>(),
                                                                           class_mask_dev ? hist : nullptr);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  observed(sc, rows, cols, K9, class_mask_dev != nullptr);
  return PGP_OK;
}

int k8_render(pgp_ctx* ctx, const int32_t* obj_ids, const double* poses16, int n, float* depth_out, int32_t* slot_out) {
  K8Scratch& sc = k8_scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  const size_t npx = (size_t)sc.rows * sc.cols;
  const int64_t offs[2] = {0, n};
  PGP_CUDA(ctx, sc.frame_d.reserve(npx * 4));
  PGP_CUDA(ctx, sc.frame_s.reserve(npx * 4));
  return run_host(ctx, sc, offs, 1, obj_ids, poses16, 0.f, sc.frame_d.as<float>(), sc.frame_s.as<int>(), [&]() {
    cudaError_t e = cudaMemcpyAsync(depth_out, sc.frame_d.p, npx * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && slot_out) e = cudaMemcpyAsync(slot_out, sc.frame_s.p, npx * 4, cudaMemcpyDeviceToHost, st);
    return e;
  });
}

int k8_depth_cost(pgp_ctx* ctx, const int64_t* offs, int n_states, const int32_t* obj_ids, const double* poses16, float tau, pgp_depth_counts* out) {
  K8Scratch& sc = k8_scratch_of(ctx);
  const int64_t n_rec = n_states > 0 ? offs[n_states] : 0;
  if (n_rec == 0) return PGP_OK;
  std::vector<pgp_depth_counts> counts((size_t)n_rec);         // out is written only once the status is PGP_OK
  int rc = run_host(ctx, sc, offs, n_states, obj_ids, poses16, tau, nullptr, nullptr, [&]() {
    return cudaMemcpyAsync(counts.data(), sc.out.p, (size_t)n_rec * sizeof(pgp_depth_counts), cudaMemcpyDeviceToHost, ctx->stream);
  });
  if (rc) return rc;
  memcpy(out, counts.data(), counts.size() * sizeof(pgp_depth_counts));
  return PGP_OK;
}

int k8_depth_cost_dev(pgp_ctx* ctx, const int64_t* offs, int n_states, const int32_t* obj_ids, const double* poses16_dev, float tau,
                      pgp_depth_counts* out_dev, int32_t* status_dev) {
  K8Scratch& sc = k8_scratch_of(ctx);
  std::vector<Chunk> chunks;
  int rc = cut_chunks(ctx, sc, offs, n_states, obj_ids, nullptr, chunks);
  return rc ? rc : run_pipeline(ctx, sc, offs, n_states, obj_ids, poses16_dev, tau, chunks, reinterpret_cast<int*>(out_dev), nullptr, nullptr,
                                status_dev);
}

int k8_render_dev(pgp_ctx* ctx, const int64_t* offs, int n_states, const int32_t* obj_ids, const double* poses16_dev, float* depth_dev,
                  int32_t* slot_dev, int32_t* status_dev) {
  K8Scratch& sc = k8_scratch_of(ctx);
  std::vector<Chunk> chunks;
  int rc = cut_chunks(ctx, sc, offs, n_states, obj_ids, nullptr, chunks);
  return rc ? rc : run_pipeline(ctx, sc, offs, n_states, obj_ids, poses16_dev, 0.f, chunks, nullptr, depth_dev, slot_dev, status_dev);
}

void k8_release(pgp_ctx* ctx) {
  if (!ctx->k8_scratch) return;
  K8Scratch* sc = static_cast<K8Scratch*>(ctx->k8_scratch);
  for (Mesh& m : sc->mesh) { m.v.release(); m.t.release(); }
  for (DevBuf* b : {&sc->raw, &sc->depth, &sc->mask, &sc->tables, &sc->pose12, &sc->state_pairs, &sc->raw_poses, &sc->status, &sc->vtx, &sc->tris,
                    &sc->cnt, &sc->cursor, &sc->bins, &sc->list, &sc->misc, &sc->out, &sc->frame_d, &sc->frame_s})
    b->release();
  sc->staging.release();
  delete sc;
  ctx->k8_scratch = nullptr;
}
