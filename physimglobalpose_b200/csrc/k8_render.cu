// K8 -- rendered-depth cost of MCTS states: the placed objects' meshes rasterized at their poses and compared with the observed
// depth frame (UCTState::render + UCTState::computeCost, PPE/src/hypothesis_verification/mcts/UCTState.cpp:93-116; renderer
// depth_sim/src/renderScene.cpp:36-84).  RESTATED, PARITY UNPINNED: the reference renders with OpenGL (a pcl::simulation fork)
// and computeCost's formula is not available; K8 follows its own exact contract (include/pgp.h, DESIGN.md 3), restated in numpy
// in oracle/render_port.py and matched bit for bit.
//
// Sort-middle tiled rasterizer, per chunk of states:
//   k8_vertex  per (state, slot, vertex): transform, project, snap to 1/256 px
//   k8_setup   per triangle: cull, orient, pixel bounding box clipped to the image, count its (state, 16x16 tile) bins
//   scan -> k8_list (non-empty bins) -> one host sync for the two totals -> k8_fill (bin lists)
//   k8_tiles   one CTA per non-empty (state, tile): 64-bit (depth bits, slot) z-buffer in shared memory with atomicMin, then
//              either the frame written out (pgp_render_depth) or the fused comparison with the observation, summed per slot in
//              shared memory and added to the state's records.
// Work scales with triangles and covered tiles; no per-state frame reaches HBM.  Every count is an integer and every depth is a
// deterministic function of one triangle and one sample, so results do not depend on scheduling.
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
constexpr int64_t CHUNK_PAIRS = 1 << 25;       // (triangle, tile) entries per chunk of more than one state
constexpr int64_t MAX_PAIRS = (1ll << 31) - 1; // ... and of a single state
constexpr float GUARD = 1048576.f;             // 2^20 px

struct Inst {                                  // one placed object of the chunk
  float T[12];
  const float* v;
  const int32_t* t;
  int nv, nt, vbase, tbase;
  int state, slot;                             // chunk-local state, position in the state
};

struct __align__(16) Tri {                     // a triangle after setup (slot < 0: culled)
  int x[3], y[3];                              // snapped, oriented: A > 0
  int slot, state;
  short c0, c1, r0, r1;                        // covered pixel box, clipped to the image
  double iz[3];
};
static_assert(sizeof(Tri) == 64, "Tri is one 64-byte record");

__device__ __forceinline__ int find_inst(const Inst* __restrict__ in, int n, int id, bool tri) {
  int lo = 0, hi = n - 1;                      // last instance whose base <= id
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((tri ? in[mid].tbase : in[mid].vbase) <= id) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// vertex -> {snapped x, snapped y, Z bits, ok}
__global__ void __launch_bounds__(T) k8_vertex(const Inst* __restrict__ inst, int n_inst, int n_vert, float fx, float fy, float cx, float cy,
                                               int4* __restrict__ out) {
  const int v = blockIdx.x * T + threadIdx.x;
  if (v >= n_vert) return;
  const Inst& I = inst[find_inst(inst, n_inst, v, false)];
  const float* p = I.v + 3 * (v - I.vbase);
  const float x = p[0], y = p[1], z = p[2];
  const float X = xf_row(I.T[0], I.T[1], I.T[2], I.T[3], x, y, z);
  const float Y = xf_row(I.T[4], I.T[5], I.T[6], I.T[7], x, y, z);
  const float Z = xf_row(I.T[8], I.T[9], I.T[10], I.T[11], x, y, z);
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

// triangle -> record + bin counts
__global__ void __launch_bounds__(T) k8_setup(const Inst* __restrict__ inst, int n_inst, int n_tri, const int4* __restrict__ vtx, int rows, int cols,
                                              int ntx, int ntiles, Tri* __restrict__ tris, uint32_t* __restrict__ cnt,
                                              unsigned long long* __restrict__ pair_total) {
  const int t = blockIdx.x * T + threadIdx.x;
  uint32_t pairs = 0;
  if (t < n_tri) {
    const Inst& I = inst[find_inst(inst, n_inst, t, true)];
    const int32_t* ix = I.t + 3 * (t - I.tbase);
    int4 a = vtx[I.vbase + ix[0]], b = vtx[I.vbase + ix[1]], c = vtx[I.vbase + ix[2]];
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
        r.slot = I.slot; r.state = I.state;
        r.c0 = (short)c0; r.c1 = (short)c1; r.r0 = (short)r0; r.r1 = (short)r1;
        r.iz[0] = __ddiv_rn(1.0, (double)__int_as_float(a.z));
        r.iz[1] = __ddiv_rn(1.0, (double)__int_as_float(b.z));
        r.iz[2] = __ddiv_rn(1.0, (double)__int_as_float(c.z));
        const int tx0 = c0 / TILE, tx1 = c1 / TILE, ty0 = r0 / TILE, ty1 = r1 / TILE;
        uint32_t* base = cnt + (size_t)I.state * ntiles;
        for (int ty = ty0; ty <= ty1; ++ty)
          for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(base + ty * ntx + tx, 1u);
        pairs = (uint32_t)((tx1 - tx0 + 1) * (ty1 - ty0 + 1));
      }
    }
    tris[t] = r;
  }
  pairs = __reduce_add_sync(0xffffffffu, pairs);      // <= 32 x 2^20: no wrap
  if ((threadIdx.x & 31) == 0 && pairs) atomicAdd(pair_total, (unsigned long long)pairs);
}

__global__ void __launch_bounds__(T) k8_fill(const Tri* __restrict__ tris, int n_tri, int ntx, int ntiles, uint32_t* __restrict__ cursor,
                                             uint32_t* __restrict__ bins) {
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

// RENDER: write the frame (one state);  else: compare with the observation and add the per-slot counts to out
template <bool RENDER>
__global__ void __launch_bounds__(TT) k8_tiles(const Tri* __restrict__ tris, const uint32_t* __restrict__ off, const uint32_t* __restrict__ bins,
                                               const uint32_t* __restrict__ list, int ntx, int ntiles, Obs obs, float tau,
                                               const int* __restrict__ state_first, const int* __restrict__ rec_cls, int* __restrict__ out,
                                               float* __restrict__ depth_out, int* __restrict__ slot_out) {
  __shared__ unsigned long long z[TT];
  __shared__ uint32_t queue[TT];
  __shared__ int qn;
  __shared__ int acc[PGP_MAX_OBJECTS * 5];
  __shared__ int org[2];                       // the tile's first column and row (read from shared memory: kept out of the registers
                                               // that must survive the double divisions' calls, which would spill them)
  volatile int* vorg = org;
  const int tid = threadIdx.x;
  const uint32_t key = list[blockIdx.x];
  z[tid] = ~0ull;
  if (tid == 0) {
    const int tile = (int)(key % (uint32_t)ntiles);
    qn = 0; org[0] = (tile % ntx) * TILE; org[1] = (tile / ntx) * TILE;
  }
  __syncthreads();
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
    for (int j = 0; j < nq; ++j) {                                   // larger triangles: the whole CTA, one pixel per thread
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
      depth_out[p] = k == ~0ull ? 0.f : __uint_as_float((unsigned)(k >> 32));
      if (slot_out) slot_out[p] = k == ~0ull ? -1 : (int)(unsigned)k;
    }
    return;
  }
  const int first = state_first[list[blockIdx.x] / (uint32_t)ntiles];
  for (int i = tid; i < PGP_MAX_OBJECTS * 5; i += TT) acc[i] = 0;
  __syncthreads();
  if (in_img && k != ~0ull) {
    const int slot = (int)(unsigned)k;
    const float r = __uint_as_float((unsigned)(k >> 32));
    int* a = acc + 5 * slot;
    atomicAdd(a + 0, 1);
    const float o = obs.depth[p];
    if (depth_valid(o)) {
      if (fabsf(__fsub_rn(r, o)) <= tau) atomicAdd(a + 1, 1);
      else if (__fsub_rn(o, r) > tau) atomicAdd(a + 2, 1);
      else atomicAdd(a + 3, 1);                                      // r - o > tau
    }
    if (obs.mask && (int)obs.mask[p] == rec_cls[first + slot]) atomicAdd(a + 4, 1);
  }
  __syncthreads();
  for (int i = tid; i < PGP_MAX_OBJECTS * 5; i += TT)
    if (acc[i]) atomicAdd(out + 5 * (size_t)(first + i / 5) + i % 5, acc[i]);
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
struct K8Scratch {
  Mesh mesh[PGP_MAX_OBJECTS];
  DevBuf raw, depth, mask;                     // observation: as given, decoded, labels
  int rows = 0, cols = 0;
  bool has_obs = false, has_mask = false;
  float fx = 0, fy = 0, cx = 0, cy = 0;
  DevBuf inst, state_first, rec_cls, vtx, tris, cnt, cursor, bins, list, misc, out, frame_d, frame_s;
};
K8Scratch& k8_scratch_of(pgp_ctx* ctx) {
  if (!ctx->k8_scratch) ctx->k8_scratch = new K8Scratch();
  return *static_cast<K8Scratch*>(ctx->k8_scratch);
}

constexpr int SPLIT = 1;                       // run_chunk: the chunk has too many (triangle, tile) entries, split it

// States [s, e) of the call: every placed object of them rasterized and compared (or, RENDER, the one state's frame written).
int run_chunk(pgp_ctx* ctx, K8Scratch& sc, bool render, const int64_t* offs, int s, int e, const int32_t* obj_ids, const double* poses16,
              float tau) {
  cudaStream_t st = ctx->stream;
  const int ntx = (sc.cols + TILE - 1) / TILE, nty = (sc.rows + TILE - 1) / TILE, ntiles = ntx * nty;
  const int64_t p0 = offs[s], p1 = offs[e];
  std::vector<Inst> inst;
  std::vector<int> first(e - s);
  int64_t nvert = 0, ntri = 0;
  for (int q = s; q < e; ++q) {
    first[q - s] = (int)offs[q];
    for (int64_t i = offs[q]; i < offs[q + 1]; ++i) {
      const Mesh& m = sc.mesh[obj_ids[i]];
      Inst in;
      pose16_to_f32x12(poses16 + 16 * i, in.T);
      in.v = m.v.as<float>(); in.t = m.t.as<int32_t>();
      in.nv = m.nv; in.nt = m.nt; in.vbase = (int)nvert; in.tbase = (int)ntri;
      in.state = q - s; in.slot = (int)(i - offs[q]);
      inst.push_back(in);
      nvert += m.nv; ntri += m.nt;
    }
  }
  if (p1 == p0) return PGP_OK;
  const int n_inst = (int)inst.size(), n_keys = (e - s) * ntiles;
  PGP_CUDA(ctx, sc.inst.reserve(inst.size() * sizeof(Inst)));
  PGP_CUDA(ctx, sc.state_first.reserve(first.size() * 4));
  PGP_CUDA(ctx, sc.vtx.reserve((size_t)nvert * 16));
  PGP_CUDA(ctx, sc.tris.reserve((size_t)ntri * sizeof(Tri)));
  PGP_CUDA(ctx, sc.cnt.reserve((size_t)(n_keys + 1) * 4));
  PGP_CUDA(ctx, sc.cursor.reserve((size_t)(n_keys + 1) * 4));
  PGP_CUDA(ctx, sc.list.reserve((size_t)n_keys * 4));
  PGP_CUDA(ctx, sc.misc.reserve(16));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.inst.p, inst.data(), inst.size() * sizeof(Inst), cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.state_first.p, first.data(), first.size() * 4, cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.cnt.p, 0, (size_t)(n_keys + 1) * 4, st));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.misc.p, 0, 16, st));
  unsigned long long* pair_total = sc.misc.as<unsigned long long>();
  uint32_t* n_list = sc.misc.as<uint32_t>() + 2;                     // low word of the second u64
  k8_vertex<<<(unsigned)((nvert + T - 1) / T), T, 0, st>>>(sc.inst.as<Inst>(), n_inst, (int)nvert, sc.fx, sc.fy, sc.cx, sc.cy, sc.vtx.as<int4>());
  k8_setup<<<(unsigned)((ntri + T - 1) / T), T, 0, st>>>(sc.inst.as<Inst>(), n_inst, (int)ntri, sc.vtx.as<int4>(), sc.rows, sc.cols, ntx, ntiles,
                                                         sc.tris.as<Tri>(), sc.cnt.as<uint32_t>(), pair_total);
  ctx->launches += 2;
  PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((n_keys + 1) / 2048 + 4096) * 4));
  int rc = pgp_scan_exclusive_u32(ctx, sc.cnt.as<uint32_t>(), (int64_t)n_keys + 1, ctx->scene.scratch.as<uint32_t>());
  if (rc) return rc;
  k8_list<<<(unsigned)((n_keys + T - 1) / T), T, 0, st>>>(sc.cnt.as<uint32_t>(), n_keys, sc.list.as<uint32_t>(), n_list);
  ctx->launches++;
  unsigned long long totals[2] = {0, 0};                             // (triangle, tile) pairs, non-empty bins
  PGP_CUDA(ctx, cudaMemcpyAsync(totals, sc.misc.p, 16, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  const unsigned long long pairs = totals[0];
  const unsigned n_bins = (unsigned)totals[1];
  if ((int64_t)pairs > (e - s > 1 ? CHUNK_PAIRS : MAX_PAIRS)) {
    if (e - s > 1) return SPLIT;
    return pgp_fail(ctx, PGP_E_TOO_LARGE, "one state covers %llu (triangle, tile) pairs", pairs);
  }
  if (pairs == 0) return PGP_OK;
  PGP_CUDA(ctx, sc.bins.reserve((size_t)pairs * 4));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.cursor.p, sc.cnt.p, (size_t)(n_keys + 1) * 4, cudaMemcpyDeviceToDevice, st));
  k8_fill<<<(unsigned)((ntri + T - 1) / T), T, 0, st>>>(sc.tris.as<Tri>(), (int)ntri, ntx, ntiles, sc.cursor.as<uint32_t>(), sc.bins.as<uint32_t>());
  const Obs obs{sc.depth.as<float>(), sc.has_mask ? sc.mask.as<uint8_t>() : nullptr, sc.rows, sc.cols};
  if (render)
    k8_tiles<true><<<n_bins, TT, 0, st>>>(sc.tris.as<Tri>(), sc.cnt.as<uint32_t>(), sc.bins.as<uint32_t>(), sc.list.as<uint32_t>(), ntx, ntiles, obs,
                                          tau, sc.state_first.as<int>(), sc.rec_cls.as<int>(), nullptr, sc.frame_d.as<float>(), sc.frame_s.as<int>());
  else
    k8_tiles<false><<<n_bins, TT, 0, st>>>(sc.tris.as<Tri>(), sc.cnt.as<uint32_t>(), sc.bins.as<uint32_t>(), sc.list.as<uint32_t>(), ntx, ntiles, obs,
                                           tau, sc.state_first.as<int>(), sc.rec_cls.as<int>(), sc.out.as<int>(), nullptr, nullptr);
  ctx->launches += 2;
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

// class id of every placed object (record order), for the on_segment test
int upload_classes(pgp_ctx* ctx, K8Scratch& sc, const int32_t* obj_ids, int64_t n) {
  std::vector<int> cls((size_t)std::max<int64_t>(n, 1));
  for (int64_t i = 0; i < n; ++i) cls[i] = sc.mesh[obj_ids[i]].cls;
  PGP_CUDA(ctx, sc.rec_cls.reserve(cls.size() * 4));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.rec_cls.p, cls.data(), cls.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  return PGP_OK;
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
  sc.rows = rows; sc.cols = cols;
  sc.fx = K9[0]; sc.fy = K9[4]; sc.cx = K9[2]; sc.cy = K9[5];
  sc.has_mask = class_mask != nullptr;
  sc.has_obs = true;
  return PGP_OK;
}

int k8_render(pgp_ctx* ctx, const int32_t* obj_ids, const double* poses16, int n, float* depth_out, int32_t* slot_out) {
  K8Scratch& sc = k8_scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  const size_t npx = (size_t)sc.rows * sc.cols;
  PGP_CUDA(ctx, sc.frame_d.reserve(npx * 4));
  PGP_CUDA(ctx, sc.frame_s.reserve(npx * 4));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.frame_d.p, 0, npx * 4, st));               // 0.0f: nothing
  PGP_CUDA(ctx, cudaMemsetAsync(sc.frame_s.p, 0xff, npx * 4, st));            // -1: nothing
  const int64_t offs[2] = {0, n};
  int rc = upload_classes(ctx, sc, obj_ids, n);
  if (!rc) rc = run_chunk(ctx, sc, true, offs, 0, 1, obj_ids, poses16, 0.f);
  if (rc) return rc;
  PGP_CUDA(ctx, cudaMemcpyAsync(depth_out, sc.frame_d.p, npx * 4, cudaMemcpyDeviceToHost, st));
  if (slot_out) PGP_CUDA(ctx, cudaMemcpyAsync(slot_out, sc.frame_s.p, npx * 4, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  return PGP_OK;
}

int k8_depth_cost(pgp_ctx* ctx, const int64_t* offs, int n_states, const int32_t* obj_ids, const double* poses16, float tau, pgp_depth_counts* out) {
  K8Scratch& sc = k8_scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  const int64_t n_rec = n_states > 0 ? offs[n_states] : 0;
  if (n_rec == 0) return PGP_OK;
  const int64_t ntiles = (int64_t)((sc.cols + TILE - 1) / TILE) * ((sc.rows + TILE - 1) / TILE);
  PGP_CUDA(ctx, sc.out.reserve((size_t)n_rec * sizeof(pgp_depth_counts)));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.out.p, 0, (size_t)n_rec * sizeof(pgp_depth_counts), st));
  int rc = upload_classes(ctx, sc, obj_ids, n_rec);
  if (rc) return rc;
  for (int s = 0; s < n_states;) {
    int64_t tris = 0, verts = 0;
    int e = s;
    while (e < n_states) {                   // whole states only: a state's z-test needs all of its objects
      int64_t t = 0, v = 0;
      for (int64_t i = offs[e]; i < offs[e + 1]; ++i) { t += sc.mesh[obj_ids[i]].nt; v += sc.mesh[obj_ids[i]].nv; }
      if (e > s && (tris + t > CHUNK_TRIS || verts + v > CHUNK_VERTS || (e - s + 1) * ntiles > CHUNK_KEYS)) break;
      tris += t; verts += v; ++e;
    }
    while ((rc = run_chunk(ctx, sc, false, offs, s, e, obj_ids, poses16, tau)) == SPLIT) e = s + (e - s) / 2;
    if (rc) return rc;
    s = e;
  }
  PGP_CUDA(ctx, cudaMemcpyAsync(out, sc.out.p, (size_t)n_rec * sizeof(pgp_depth_counts), cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  return PGP_OK;
}

void k8_release(pgp_ctx* ctx) {
  if (!ctx->k8_scratch) return;
  K8Scratch* sc = static_cast<K8Scratch*>(ctx->k8_scratch);
  for (Mesh& m : sc->mesh) { m.v.release(); m.t.release(); }
  for (DevBuf* b : {&sc->raw, &sc->depth, &sc->mask, &sc->inst, &sc->state_first, &sc->rec_cls, &sc->vtx, &sc->tris, &sc->cnt, &sc->cursor, &sc->bins,
                    &sc->list, &sc->misc, &sc->out, &sc->frame_d, &sc->frame_s})
    b->release();
  delete sc;
  ctx->k8_scratch = nullptr;
}
