// K3 -- LCP scoring of pose hypotheses on the scene voxel grid.
//
// Replaces, per hypothesis, Match4PCSBase::Verify (S4/algorithms/match4pcsBase.cc:1699-1731) and
// Match4PCSBase::WeightedVerify (:1733-1766), i.e. one KdTree::doQueryRestrictedClosestIndex
// (S4/accelerators/kdtree.h:394-459) per validation-model point, and the loop over hypotheses of
// Perform_N_steps (:1888-1901).
//
// Two kernels.  k3_fine_kernel (below, the one that runs) works on the tri-state label structure of K1b/K1c/K1d:
//   persistent CTAs, one per SM; the validation model (kd-leaf order: every aligned run of 32 points is a compact patch), its
//   group spheres and the bitmap+rank table are staged ONCE per CTA into shared memory with 1-D TMA bulk copies (cp.async.bulk
//   -> SASS UBLKCP) on an mbarrier; each warp pulls one hypothesis at a time from a global work counter, keeps its 3x4 transform
//   in registers and runs
//     group cull   one lane per 32-point group: distance-field lower bound at the image of the group's centre vs the (norm-
//                  stretched) group radius + delta -> groups that cannot reach the scene are never looked at,
//     phase 1      128 points per step (uniform control flow): FMA voxel transform, shared-memory bitmap+rank word, ONE 4-byte
//                  gather of the 2-bit label; IN counts, OUT is done, AMBIG (weighted: IN too) goes to a per-warp queue
//                  (warp-ballot compaction),
//     phase 2      whenever 32 are queued, every lane takes one and runs the reference's exact non-fused test against the
//                  voxel's few candidate records.
// k3_lcp_kernel (first in this file) is the plain 27-cell probe the fine structure was derived from: exact fp32 transform, cell,
// one dilated-occupancy bit, then the exact d2 <= delta^2 test over the 9 contiguous x-rows of the 27 cells.  It is the
// fallback when the fine grid cannot be built (margins do not close, absurd densities) and the cross-check of the tests.
// Inlier counts are warp-reduced (REDUX) -- integer, hence order-free and bit-exact.
// All float math that decides a count is the reference's association, non-fused (pgp_internal.cuh).
#include <math.h>

#include "pgp_internal.cuh"

namespace {

constexpr int WARPS = 16;            // warps per CTA
constexpr int THREADS = WARPS * 32;
constexpr int QCAP = 64;             // queue slots per warp

struct LcpParams {
  const float4* model;       // nv x float4 (xyz, w = original index bits)
  const float4* model_nrm;   // nv x float4
  int nv;
  int tile_cap;              // model points per shared-memory tile
  const float* T;            // n x 12
  long long n;
  long long n_bulk;          // fine kernel: hypotheses [0, n_bulk) are one work unit each, the rest are split into `split` model chunks
  uint32_t* ready;           // streamed upload: number of hypotheses whose transforms have arrived (nullptr: all of them)
  unsigned long long ready_timeout_ns;   // how long one wait on `ready` may last before the launch gives up (host re-scores)
  int split;                 // (so that the last wave of the persistent grid ends on quarter-sized units, not whole hypotheses)
  const float4* pts;
  const float4* aux;
  const uint32_t* cell_start;
  const uint32_t* bitmap;
  int bitmap_words;          // words staged in smem (0: read the bitmap from global/L1)
  GridParams g;
  uint32_t* counts;
  float* scores;
  unsigned long long* work;  // one counter per model tile
  int n_tiles;
  // fine tri-state path (K1b)
  const uint2* bmrank;       // per bitmap word {bits, rank prefix}
  const uint32_t* codes;     // n_blocks x 32 words
  int bmrank_words;          // words staged in smem (0: read from global/L1)
  const uint32_t* hdrw;      // n_blocks x 32: global rank of the first AMBIG voxel of each label word (K1b pass B)
  const float4* aslot;       // per AMBIG voxel, 32 bytes: {x0, y0, z0, n} {x1, y1, z1, first overflow record}, closest to the voxel centre first
  const float4* aovf;        // candidates 3 .. n of every AMBIG voxel {x, y, z, original index}
  float model_rinf;          // max |coordinate| of the validation model (bounds the transform's intermediates)
  const unsigned char* wcnt; // K1c: per voxel candidate count (a byte)
  const uint32_t* wword;     // K1c: per label word (16 voxels) the first record
  const uint32_t* wlists;    // K1c: candidates' ORIGINAL indices
  const uint32_t* vrec;      // K1c: per voxel (code << 24 | representative candidate, as a position in the cell-sorted cloud): spread of the candidates' normals
  const float4* pts_orig;    // centred scene points by ORIGINAL index (Scene::unsorted)
  const float4* aux_orig;    // unit normal + prior by ORIGINAL scene index
  const float4* groups;      // bounding sphere {centre, radius} of every aligned run of 32 validation points (pgp_set_model)
  const float* dist;         // K1d: per cell, lower bound of the distance to the nearest scene point (nullptr: no group cull)
  float cull_add;            // delta (1 + 1e-5) + rounding margin: a group is dropped when dist > |A| r + cull_add
  float dist_scale;          // voxel units -> sub-cells of the K1d lattice (dist_r / 8)
  float sub_h2;              // (edge of a K1d sub-cell)^2, shrunk by 1e-4
  int ddx, ddy, ddz;         // K1d lattice dimensions
};

// ---- mbarrier + TMA bulk copy (global -> shared), sm_90+/sm_100a PTX ---------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra D;\n\tbra W;\n\tD:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

struct Xf { float m[12]; };

// The batch may still be being written by the copy engine while the kernel runs (streamed upload, LcpParams::ready), so T is not
// read-only for the kernel's lifetime and must not go through the non-coherent path (ld.global.nc / __ldg): plain cached loads
// (ld.global.ca), issued only after the acquire load of the upload counter has covered hypothesis h.  No line of T is touched
// before its chunk has landed (chunks end on 384-byte boundaries), so L1 can never hold a stale copy.
__device__ __forceinline__ Xf load_xf(const float* T, long long h) {
  const float4* t4 = reinterpret_cast<const float4*>(T + 12 * h);
  const float4 a = __ldca(t4), b = __ldca(t4 + 1), c = __ldca(t4 + 2);
  Xf x;
  x.m[0] = a.x; x.m[1] = a.y; x.m[2] = a.z; x.m[3] = a.w;
  x.m[4] = b.x; x.m[5] = b.y; x.m[6] = b.z; x.m[7] = b.w;
  x.m[8] = c.x; x.m[9] = c.y; x.m[10] = c.z; x.m[11] = c.w;
  return x;
}

__device__ __forceinline__ void apply_xf(const Xf& x, float4 q, float& tx, float& ty, float& tz) {
  tx = xf_row(x.m[0], x.m[1], x.m[2], x.m[3], q.x, q.y, q.z);
  ty = xf_row(x.m[4], x.m[5], x.m[6], x.m[7], q.x, q.y, q.z);
  tz = xf_row(x.m[8], x.m[9], x.m[10], x.m[11], q.x, q.y, q.z);
}

// cell of a query; false when the query is outside the grid (then no scene point is within delta)
__device__ __forceinline__ bool query_cell(const GridParams& g, float tx, float ty, float tz, int& cx, int& cy, int& cz) {
  float ux = cell_coord(tx, g.lo[0], g.inv_h), uy = cell_coord(ty, g.lo[1], g.inv_h), uz = cell_coord(tz, g.lo[2], g.inv_h);
  bool in = (ux >= 1.0f) & (ux < (float)(g.dim[0] - 1)) & (uy >= 1.0f) & (uy < (float)(g.dim[1] - 1)) & (uz >= 1.0f) &
            (uz < (float)(g.dim[2] - 1));
  cx = (int)ux; cy = (int)uy; cz = (int)uz;
  return in;   // NaN compares false
}

// exact existence test over the 27 cells = 9 contiguous x-rows
__device__ __forceinline__ bool exists_within(const LcpParams& p, float tx, float ty, float tz, int cx, int cy, int cz) {
  const int dx = p.g.dim[0], dy = p.g.dim[1];
  const float r2 = p.g.r2;
#pragma unroll 1
  for (int oz = -1; oz <= 1; ++oz) {
    const int rowz = ((cz + oz) * dy + cy) * dx + cx;
    uint32_t s[3], e[3];
#pragma unroll
    for (int oy = -1; oy <= 1; ++oy) {
      s[oy + 1] = __ldg(p.cell_start + rowz + oy * dx - 1);
      e[oy + 1] = __ldg(p.cell_start + rowz + oy * dx + 2);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      for (uint32_t i = s[k]; i < e[k]; ++i) {
        float4 q = __ldg(p.pts + i);
        if (sqdist3(tx, ty, tz, q.x, q.y, q.z) <= r2) return true;
      }
    }
  }
  return false;
}

// nearest in-range scene point: sorted position (or -1).  Acceptance d2 <= best as kdtree.h:424;
// exact ties resolve to the smaller original index (the reference: kd-tree visiting order).
__device__ __forceinline__ int nearest_within(const LcpParams& p, float tx, float ty, float tz, int cx, int cy, int cz) {
  const int dx = p.g.dim[0], dy = p.g.dim[1];
  float best = p.g.r2;
  int best_pos = -1, best_orig = 0x7fffffff;
#pragma unroll 1
  for (int oz = -1; oz <= 1; ++oz) {
    const int rowz = ((cz + oz) * dy + cy) * dx + cx;
    uint32_t s[3], e[3];
#pragma unroll
    for (int oy = -1; oy <= 1; ++oy) {
      s[oy + 1] = __ldg(p.cell_start + rowz + oy * dx - 1);
      e[oy + 1] = __ldg(p.cell_start + rowz + oy * dx + 2);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      for (uint32_t i = s[k]; i < e[k]; ++i) {
        float4 q = __ldg(p.pts + i);
        float d2 = sqdist3(tx, ty, tz, q.x, q.y, q.z);
        int orig = __float_as_int(q.w);
        if (d2 < best || (d2 == best && (best_pos < 0 || orig < best_orig))) { best = d2; best_pos = (int)i; best_orig = orig; }
      }
    }
  }
  return best_pos;
}

// The normal gate of WeightedVerify (match4pcsBase.cc:1755-1758):
//   n_q = R n (tree-order products); angle = float(double(acosf(dot) * 180.f) / pi);
//   min(angle, |180 - angle|) < 30   with NaN (|dot| > 1) never counted.
// The decision is taken on the dot product; only inside a guard band around cos 30 deg is the
// angle evaluated (correctly rounded acos via double), so libm differences cannot matter outside
// a 1-ulp sliver at exactly 30 / 150 degrees.
__device__ __forceinline__ bool normal_gate(const Xf& x, float4 nm, float4 ns) {
  float qx = dot3_tree(x.m[0], x.m[1], x.m[2], nm.x, nm.y, nm.z);
  float qy = dot3_tree(x.m[4], x.m[5], x.m[6], nm.x, nm.y, nm.z);
  float qz = dot3_tree(x.m[8], x.m[9], x.m[10], nm.x, nm.y, nm.z);
  float d = dot3_tree(ns.x, ns.y, ns.z, qx, qy, qz);
  float a = fabsf(d);
  if (!(a <= 1.0f)) return false;                 // acos -> NaN -> both min() operands NaN -> not counted
  const float c30 = 0.8660254f;
  if (a > c30 + 1e-4f) return true;
  if (a < c30 - 1e-4f) return false;
  float ang = (float)((double)__fmul_rn((float)acos((double)d), 180.0f) / 3.14159265358979323846);
  float other = fabsf(__fsub_rn(180.0f, ang));
  float m = other < ang ? other : ang;
  return m < 30.0f;
}

template <int MODE>   // 0 = count, 1 = weighted with binary priors (order-free integer sums)
__global__ void __launch_bounds__(THREADS, 2) k3_lcp_kernel(const __grid_constant__ LcpParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t mbar;
  float4* s_model = reinterpret_cast<float4*>(smem);
  float4* s_nrm = s_model + p.tile_cap;                                   // only MODE 1
  uint32_t* s_bitmap = reinterpret_cast<uint32_t*>(smem + (size_t)p.tile_cap * 16 * (MODE == 1 ? 2 : 1));
  uint16_t* s_queue = reinterpret_cast<uint16_t*>(s_bitmap + p.bitmap_words);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint16_t* q = s_queue + warp * QCAP;
  const uint32_t* bitmap = p.bitmap_words ? s_bitmap : p.bitmap;
  const unsigned lt_mask = (1u << lane) - 1u;

  if (threadIdx.x == 0) mbar_init(&mbar, 1);
  __syncthreads();

  for (int tile = 0; tile < p.n_tiles; ++tile) {
    const int t0 = tile * p.tile_cap;
    const int tn = min(p.tile_cap, p.nv - t0);
    if (threadIdx.x == 0) {
      uint32_t bytes = (uint32_t)tn * 16u;
      uint32_t total = bytes * (MODE == 1 ? 2u : 1u) + (tile == 0 ? (uint32_t)p.bitmap_words * 4u : 0u);
      mbar_expect_tx(&mbar, total);
      tma_bulk_g2s(s_model, p.model + t0, bytes, &mbar);
      if (MODE == 1) tma_bulk_g2s(s_nrm, p.model_nrm + t0, bytes, &mbar);
      if (tile == 0 && p.bitmap_words) tma_bulk_g2s(s_bitmap, p.bitmap, (uint32_t)p.bitmap_words * 4u, &mbar);
    }
    mbar_wait(&mbar, tile & 1);

    for (;;) {
      long long h = 0;
      if (lane == 0) h = (long long)atomicAdd(p.work + tile, 1ull);
      h = __shfl_sync(0xffffffffu, h, 0);
      if (h >= p.n) break;
      const Xf x = load_xf(p.T, h);
      int good = 0;
      int qn = 0;

      auto drain = [&](int take) {   // lanes < take each resolve one queued query
        if (lane < take) {
          int i = q[qn - take + lane];
          float tx, ty, tz;
          int cx, cy, cz;
          apply_xf(x, s_model[i], tx, ty, tz);
          query_cell(p.g, tx, ty, tz, cx, cy, cz);
          if (MODE == 0) {
            good += exists_within(p, tx, ty, tz, cx, cy, cz) ? 1 : 0;
          } else {
            int pos = nearest_within(p, tx, ty, tz, cx, cy, cz);
            if (pos >= 0) {
              float4 ns = __ldg(p.aux + pos);
              if (normal_gate(x, s_nrm[i], ns)) good += (ns.w != 0.f) ? 0x10001 : 0x1;   // hi: prior==1, lo: gated
            }
          }
        }
        qn -= take;
      };

      for (int base = 0; base < tn; base += 32) {
        const int i = base + lane;
        bool cand = false;
        if (i < tn) {
          float tx, ty, tz;
          int cx, cy, cz;
          apply_xf(x, s_model[i], tx, ty, tz);
          if (query_cell(p.g, tx, ty, tz, cx, cy, cz)) {
            int c = (cz * p.g.dim[1] + cy) * p.g.dim[0] + cx;
            cand = (bitmap[c >> 5] >> (c & 31)) & 1u;
          }
        }
        unsigned b = __ballot_sync(0xffffffffu, cand);
        if (cand) q[qn + __popc(b & lt_mask)] = (uint16_t)i;
        qn += __popc(b);
        __syncwarp();
        if (qn >= 32) { drain(32); __syncwarp(); }
      }
      if (qn > 0) { drain(qn); __syncwarp(); }

      if (MODE == 0) {
        int tot = __reduce_add_sync(0xffffffffu, good);
        if (lane == 0) {
          if (p.n_tiles == 1) {
            p.counts[h] = (uint32_t)tot;
            if (p.scores) p.scores[h] = __fdiv_rn((float)tot, (float)p.nv);   // Scalar(good)/Scalar(n) :1730
          } else if (tot) {
            atomicAdd(p.counts + h, (uint32_t)tot);
          }
        }
      } else {
        int tot = __reduce_add_sync(0xffffffffu, good);   // nv < 65536 per tile keeps the halves apart
        if (lane == 0) {
          uint32_t gated = (uint32_t)tot & 0xffffu, w = (uint32_t)tot >> 16;
          if (p.n_tiles == 1) {
            p.counts[h] = gated;
            if (p.scores) p.scores[h] = __fdiv_rn((float)w, (float)p.nv);   // weighted_match / Scalar(n) :1765
          } else {
            if (gated) atomicAdd(p.counts + h, gated);
            if (w && p.scores) atomicAdd(reinterpret_cast<uint32_t*>(p.scores) + h, w);   // integer for now; finalised below
          }
        }
      }
    }
    __syncthreads();   // everyone is done with this tile before it is overwritten
  }
}

// ---------------------------------------------------------------------------------------------
// Count mode on the fine tri-state grid (K1b).  Phase 1 computes the query's SUB-VOXEL directly
// with 9 FMAs (transform pre-scaled to voxel units), looks the cell up in the shared-memory
// bitmap+rank table and fetches the 2-bit label; OUT/IN finish the query, AMBIG queries are queued
// and resolved by the exact, non-fused test of the reference in phase 2.  The labels are
// conservative with respect to the difference between the fast transform and the reference's
// rounding sequence (GridParams::inflate), so counts stay bit-exact.
constexpr int FWARPS = 32;           // warps per CTA, one CTA per SM: 64 registers per thread
constexpr int FUNROLL = 4;           // model points per lane per step (their label gathers are issued together)
constexpr int SQCAP = 64;            // second-level (slow) queue slots per warp, weighted mode: < 32 left over + at most 32 new per drain
constexpr int FQCAP = 32 + 32 * FUNROLL;   // queue slots per warp: < 32 left over + the new ones of one step

struct FineCtx {
  const float4* s_model;
  const float4* s_nrm;       // weighted mode only
  const float4* s_groups;    // bounding spheres of the tile's 32-point groups
  const uint2* table;        // bmrank: shared (SMEM_TABLE) or global
  uint16_t* q;               // per warp: queued model-point indices
  uint32_t* qe;              // count mode: (label word index << 4) | rank of the voxel among the word's AMBIG voxels;
                             // weighted mode: the voxel's address block * 512 + voxel = (label word index << 4) | (voxel & 15)
  unsigned char* qr;         // weighted mode: rank of the voxel among the word's AMBIG voxels | (label == AMBIG) << 4
  uint16_t* sq;              // weighted mode, second-level queue (SQCAP slots per warp) of the queries the cone record could not settle:
  uint32_t* sqe;             //   model point, voxel address,
  unsigned char* sqr;        //   info | gate_known << 5 -- resolved 32 at a time so that the rare, long exact path runs on full warps
  unsigned sa;               // per warp: shared-memory address of 12 floats, the hypothesis' pre-scaled (voxel-unit) matrix -- warp-uniform
                             // data the loops re-read with three LDS.128 where they use it instead of holding 12 registers across
                             // the whole hypothesis (at 64 registers per thread the compiler spilled exactly these to local memory)
  uint16_t* glist;           // per warp: indices (u16: the shared-memory plan decides the L1 carve-out, see k3_fine_smem) of the groups of the current hypothesis that survived the cull (+ FUNROLL pad slots)
  int dummy_group;           // a group of NaN points behind the tile
  int dimx, dimy, dimz;
  unsigned limx, limy, limz;   // last voxel index per axis
  int lane;
  unsigned lt_mask;
  uint32_t dummy_word;       // offset of a zero word in `codes`
};

template <bool SMEM_TABLE>
__device__ __forceinline__ uint2 table_word(const FineCtx& f, int w) {
  if (SMEM_TABLE) return f.table[w];            // LDS.64
  return __ldg(f.table + w);
}

// Branch-free label fetch, split in two so that several queries' gathers can be in flight at once:
// label_slot() gives the word offset into `codes` (a zero dummy word behind the last block for
// queries outside the grid or in cells with an empty neighbourhood) and the bit shift.
template <bool SMEM_TABLE>
__device__ __forceinline__ uint32_t label_slot(const LcpParams& p, const FineCtx& f, int ix, int iy, int iz, uint32_t& shift) {
  // ix, iy, iz are clamped to the grid (voxel_of): a query outside lands in an apron cell (0 or dim-1 on some axis), whose bit is clear
  const int c = ((iz >> 3) * f.dimy + (iy >> 3)) * f.dimx + (ix >> 3);
  const uint2 wr = table_word<SMEM_TABLE>(f, c >> 5);
  const unsigned bit = 1u << (c & 31);
  const unsigned blk = wr.y + __popc(wr.x & (bit - 1u));
  const int v = ((iz & 7) << 6) | ((iy & 7) << 3) | (ix & 7);
  shift = (uint32_t)(v & 15) * 2u;
  return (wr.x & bit) ? blk * 32u + (uint32_t)(v >> 4) : f.dummy_word;
}

// K1c nearest-candidate list of voxel v of block blk: the 16 byte counts of its label word and the word's first entry (two
// independent loads from tables that stay L2-resident: 640 bytes per block), then first entry = word base + the counts of the voxels
// before it
__device__ __forceinline__ const uint32_t* wlist_at(const LcpParams& p, uint32_t blk, int v, uint32_t& cnt) {
  const uint4 cw = __ldg(reinterpret_cast<const uint4*>(p.wcnt + (size_t)blk * 512) + (v >> 4));
  const uint32_t base = __ldg(p.wword + (size_t)blk * 32 + (v >> 4));
  const int wi = (v >> 2) & 3, bi = v & 3;
  const uint32_t mine = wi == 0 ? cw.x : wi == 1 ? cw.y : wi == 2 ? cw.z : cw.w;
  uint32_t before = __dp4a(mine & ((1u << (8 * bi)) - 1u), 0x01010101u, 0u);
  before += (wi > 0 ? __dp4a(cw.x, 0x01010101u, 0u) : 0u) + (wi > 1 ? __dp4a(cw.y, 0x01010101u, 0u) : 0u) + (wi > 2 ? __dp4a(cw.z, 0x01010101u, 0u) : 0u);
  cnt = (mine >> (8 * bi)) & 255u;
  return p.wlists + base + before;
}
template <bool SMEM_TABLE>
__device__ __forceinline__ const uint32_t* wlist_of(const LcpParams& p, const FineCtx& f, int ix, int iy, int iz, uint32_t& cnt) {
  const int c = ((iz >> 3) * f.dimy + (iy >> 3)) * f.dimx + (ix >> 3);
  const uint2 wr = table_word<SMEM_TABLE>(f, c >> 5);
  const unsigned blk = wr.y + __popc(wr.x & ((1u << (c & 31)) - 1u));
  return wlist_at(p, blk, ((iz & 7) << 6) | ((iy & 7) << 3) | (ix & 7), cnt);
}

// one 32-byte slot of K1b's aslot (32-byte aligned) in ONE 256-bit load (sm_100: LDG.256): a single request and a single sector per
// lane.  (The .v8.f32 form of the same load crashes ptxas 12.9 in this file; .v4.u64 compiles to the same instruction.)
__device__ __forceinline__ void load_slot(const float4* __restrict__ slot, float4& a, float4& b) {
  unsigned long long u0, u1, u2, u3;
  asm("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(u0), "=l"(u1), "=l"(u2), "=l"(u3) : "l"(slot));
  a = make_float4(__uint_as_float((uint32_t)u0), __uint_as_float((uint32_t)(u0 >> 32)), __uint_as_float((uint32_t)u1), __uint_as_float((uint32_t)(u1 >> 32)));
  b = make_float4(__uint_as_float((uint32_t)u2), __uint_as_float((uint32_t)(u2 >> 32)), __uint_as_float((uint32_t)u3), __uint_as_float((uint32_t)(u3 >> 32)));
}

// phase 2 (count mode) for one queued query: the reference's exact test against the candidate records of its AMBIG voxel.
// `e` = (label word index << 4) | rank of the voxel among the AMBIG voxels of that word, packed by phase 1.  The voxel's slot holds
// its first two candidates (most lists are 1-3 long and the first, closest to the voxel centre, is the likely hit); the overflow
// records are read only when both miss.
__device__ __forceinline__ int resolve_ambiguous(const LcpParams& p, const Xf& x, const float4 m, uint32_t e) {
  const uint32_t r = __ldg(p.hdrw + (e >> 4)) + (e & 15u);
  float4 s0, s1;
  load_slot(p.aslot + 2 * (size_t)r, s0, s1);
  float tx, ty, tz;
  apply_xf(x, m, tx, ty, tz);
  const float r2 = p.g.r2;
  if (sqdist3(tx, ty, tz, s0.x, s0.y, s0.z) <= r2) return 1;
  if (sqdist3(tx, ty, tz, s1.x, s1.y, s1.z) <= r2) return 1;
  const uint32_t n = __float_as_uint(s0.w);
  if (n <= 2u) return 0;
  const float4* __restrict__ rec = p.aovf + __float_as_uint(s1.w);
  // two records per round (the second load is issued before the first is tested: the chain of dependent loads is what this path
  // waits on)
  for (uint32_t j = 0; j < n - 2u; j += 2) {
    const float4 t0 = __ldg(rec + j);
    const float4 t1 = __ldg(rec + min(j + 1u, n - 3u));
    if (sqdist3(tx, ty, tz, t0.x, t0.y, t0.z) <= r2) return 1;
    if (sqdist3(tx, ty, tz, t1.x, t1.y, t1.z) <= r2) return 1;
  }
  return 0;
}

// nearest in-range scene point among the voxel's K1c candidates (same acceptance / tie rule as
// nearest_within: d2 <= delta^2, exact ties to the smaller original index): original index or -1.
// U candidates per round: their indices are loaded together, then their points (L2-resident cloud in original order).
template <int U>
__device__ __forceinline__ int nearest_in_list(const LcpParams& p, const uint32_t* __restrict__ l, uint32_t cnt, float tx, float ty, float tz) {
  float best = p.g.r2;
  int best_orig = 0x7fffffff;
  for (uint32_t j = 0; j < cnt; j += U) {
    uint32_t id[U];
    float4 sp[U];
#pragma unroll
    for (int u = 0; u < U; ++u) if (u == 0 || j + u < cnt) id[u] = __ldg(l + j + u);
#pragma unroll
    for (int u = 0; u < U; ++u) if (u == 0 || j + u < cnt) sp[u] = __ldg(p.pts_orig + id[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (u == 0 || j + u < cnt) {
        const float d2 = sqdist3(tx, ty, tz, sp[u].x, sp[u].y, sp[u].z);
        const int orig = (int)id[u];
        if (d2 < best || (d2 == best && orig < best_orig)) { best = d2; best_orig = orig; }
      }
    }
  }
  return best_orig == 0x7fffffff ? -1 : best_orig;
}

// Phase 2 of the weighted mode for one queued query (non-OUT voxel `vaddr` = block * 512 + voxel; info = rank among the label
// word's AMBIG voxels | (label == AMBIG) << 4).  The result is 0x10001: gated and prior == 1, 0x1: gated, 0: not counted.
//
// The drain loop (score_hypothesis) first tries to settle the normal gate from the voxel's cone record alone: rep = the
// voxel's representative candidate, |n_i - n_rep| <= eps(code) for every candidate i that can be the nearest in-range point
// of a query of this voxel, equal priors (K1c).  With q = R n_model, every candidate's dot product d_i lies within
// eps |q| of d_rep, and |q| <= |R|_2; the loop evaluates d_rep with the pre-scaled FMA matrix (error < 2e-5 |R|_2 against the
// reference's rounding sequence, margin included) and compares a = |d_rep| with normal_gate's own guard band:
//     a + m < cos30 - 1e-4                      => the reference's gate FAILS for every candidate          -> 0, no search
//     a - m > cos30 + 1e-4  and  a + m < 1      => it PASSES for every candidate (and acos sees no |d| > 1) -> the weight of
//                                                  the (equal) priors, provided a scene point is in range: by construction in
//                                                  IN voxels, by count mode's existence test in AMBIG voxels
// and only the rest comes here: gate_known = 0 -> the exact path below; gate_known & 1 -> the gate passes, only the existence
// test is missing (prior bit in gate_known & 2).
//   exact path, code == 0   all candidates carry bit-identical (normal, prior): the reference's gate on the representative IS the
//                           gate on the nearest point, whichever candidate that is,
//   otherwise               nearest in-range candidate (identity!), its normal, the reference's gate (match4pcsBase.cc:1753-1761).
// Out of line: it is rare and its registers should not weigh on the loop around it.
__device__ __noinline__ int resolve_weighted_slow(const LcpParams& p, const float* __restrict__ T, long long h, const float4 m, const float4 nm,
                                                  uint32_t vaddr, uint32_t info, uint32_t vr, int gate_known) {
  const Xf x = load_xf(T, h);
  const uint32_t e = (vaddr & ~15u) | (info & 15u);
  if (gate_known & 1) return ((info & 16u) && !resolve_ambiguous(p, x, m, e)) ? 0 : ((gate_known & 2) ? 0x10001 : 0x1);
  if ((vr >> 24) == 0u) {
    const float4 ns = __ldg(p.aux + (vr & 0xffffffu));
    if (!normal_gate(x, nm, ns)) return 0;
    return ((info & 16u) && !resolve_ambiguous(p, x, m, e)) ? 0 : ((ns.w != 0.f) ? 0x10001 : 0x1);
  }
  uint32_t cnt;
  const uint32_t* l = wlist_at(p, vaddr >> 9, (int)(vaddr & 511u), cnt);
  float tx, ty, tz;
  apply_xf(x, m, tx, ty, tz);
  const int orig = nearest_in_list<2>(p, l, cnt, tx, ty, tz);
  if (orig < 0) return 0;
  const float4 ns = __ldg(p.aux_orig + orig);
  if (!normal_gate(x, nm, ns)) return 0;
  return (ns.w != 0.f) ? 0x10001 : 0x1;
}

// the per-warp matrix slot (FineCtx::sa): volatile asm so that every use site re-reads it (no value held across the loops)
__device__ __forceinline__ void sa_store(unsigned sa, const float (&a)[12]) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(sa), "f"(a[0]), "f"(a[1]), "f"(a[2]), "f"(a[3]) : "memory");
  asm volatile("st.shared.v4.f32 [%0+16], {%1, %2, %3, %4};" ::"r"(sa), "f"(a[4]), "f"(a[5]), "f"(a[6]), "f"(a[7]) : "memory");
  asm volatile("st.shared.v4.f32 [%0+32], {%1, %2, %3, %4};" ::"r"(sa), "f"(a[8]), "f"(a[9]), "f"(a[10]), "f"(a[11]) : "memory");
}
__device__ __forceinline__ void sa_load(unsigned sa, float (&a)[12]) {
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a[0]), "=f"(a[1]), "=f"(a[2]), "=f"(a[3]) : "r"(sa));
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+16];" : "=f"(a[4]), "=f"(a[5]), "=f"(a[6]), "=f"(a[7]) : "r"(sa));
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+32];" : "=f"(a[8]), "=f"(a[9]), "=f"(a[10]), "=f"(a[11]) : "r"(sa));
}

// one hypothesis, the 32-point groups [g_begin, g_end) of the staged tile (the slots behind the last point hold NaN points, which
// convert to voxel 0 and fail the range test; `dummy_group` is a whole group of them).
// FAST: voxel coordinates from the pre-scaled FMA transform a[]; otherwise the reference's
// rounding sequence followed by the grid's own cell_coord (huge / non-finite matrices).
//
// Group cull (FAST only).  All points of a group lie within r of its centre c, so their images lie within |A| r of T c
// (|A| = spectral norm of the 3x3 part, bounded by the square root of the largest absolute row sum of A^T A: 1 for a rotation).
// dist[cell of T c] is a lower bound of the distance from T c to every scene point (cells outside the grid clamp to the border
// cell: the projection onto the grid box only moves T c closer to the scene).  If that exceeds |A| r + delta + margins, no point
// of the group can have a scene point within delta: the whole group is skipped -- one test instead of 32 label look-ups.
template <bool SMEM_TABLE, bool FAST, int MODE>
__device__ __forceinline__ int score_hypothesis(const LcpParams& p, const FineCtx& f, const float* __restrict__ T, long long h, int g_begin, int g_end) {
  static_assert(FUNROLL == 4, "the survivor list is read four entries at a time");
  const Xf x = load_xf(T, h);
  // the pre-scaled matrix: count mode has the registers for it (63 used, no spill); weighted mode keeps it in the per-warp slot
  constexpr bool SLOT = MODE == 1;
  float areg[12];
  if (FAST) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      areg[4 * r + 0] = x.m[4 * r + 0] * p.g.inv_hf;
      areg[4 * r + 1] = x.m[4 * r + 1] * p.g.inv_hf;
      areg[4 * r + 2] = x.m[4 * r + 2] * p.g.inv_hf;
      areg[4 * r + 3] = (x.m[4 * r + 3] - p.g.lo[r]) * p.g.inv_hf;
    }
    if (SLOT) {
      __syncwarp();                                 // (the previous hypothesis' readers are done)
      if (f.lane == 0) sa_store(f.sa, areg);
      __syncwarp();
    }
  }
  auto get_a = [&](float (&a)[12]) {
    if (SLOT) sa_load(f.sa, a);
    else {
#pragma unroll
      for (int i = 0; i < 12; ++i) a[i] = areg[i];
    }
  };
  auto voxel_of = [&](const float (&a)[12], const float4 m, int& ix, int& iy, int& iz) {
    float ux, uy, uz;
    if (FAST) {
      ux = __fmaf_rn(a[0], m.x, __fmaf_rn(a[1], m.y, __fmaf_rn(a[2], m.z, a[3])));
      uy = __fmaf_rn(a[4], m.x, __fmaf_rn(a[5], m.y, __fmaf_rn(a[6], m.z, a[7])));
      uz = __fmaf_rn(a[8], m.x, __fmaf_rn(a[9], m.y, __fmaf_rn(a[10], m.z, a[11])));
    } else {
      float tx, ty, tz;
      apply_xf(x, m, tx, ty, tz);
      ux = cell_coord(tx, p.g.lo[0], p.g.inv_hf); uy = cell_coord(ty, p.g.lo[1], p.g.inv_hf); uz = cell_coord(tz, p.g.lo[2], p.g.inv_hf);
    }
    // float -> unsigned saturates (negative and NaN -> 0), one min clamps the high side: always a valid voxel of the grid
    ix = (int)min(__float2uint_rz(ux), f.limx); iy = (int)min(__float2uint_rz(uy), f.limy); iz = (int)min(__float2uint_rz(uz), f.limz);
  };
  // ---- survivor list of this hypothesis
  int ns = 0;
  float snorm = 0.f;         // upper bound of the spectral norm of the 3x3 part (group cull; weighted mode: |R n| <= snorm)
  {
    const bool cull = FAST && p.dist != nullptr;
    if (cull || (FAST && MODE == 1)) {
      const float g00 = x.m[0] * x.m[0] + x.m[4] * x.m[4] + x.m[8] * x.m[8], g11 = x.m[1] * x.m[1] + x.m[5] * x.m[5] + x.m[9] * x.m[9],
                  g22 = x.m[2] * x.m[2] + x.m[6] * x.m[6] + x.m[10] * x.m[10];
      const float g01 = fabsf(x.m[0] * x.m[1] + x.m[4] * x.m[5] + x.m[8] * x.m[9]), g02 = fabsf(x.m[0] * x.m[2] + x.m[4] * x.m[6] + x.m[8] * x.m[10]),
                  g12 = fabsf(x.m[1] * x.m[2] + x.m[5] * x.m[6] + x.m[9] * x.m[10]);
      snorm = sqrtf(fmaxf(fmaxf(g00 + g01 + g02, g01 + g11 + g12), g02 + g12 + g22)) * (1.0f + 1e-5f);
    }
    for (int g0 = g_begin; g0 < g_end; g0 += 32) {
      const int g = g0 + f.lane;
      bool keep = g < g_end;
      if (cull && keep) {
        const float4 sp = f.s_groups[g];
        float a[12];
        get_a(a);
        const float ux = __fmaf_rn(a[0], sp.x, __fmaf_rn(a[1], sp.y, __fmaf_rn(a[2], sp.z, a[3]))) * p.dist_scale;
        const float uy = __fmaf_rn(a[4], sp.x, __fmaf_rn(a[5], sp.y, __fmaf_rn(a[6], sp.z, a[7]))) * p.dist_scale;
        const float uz = __fmaf_rn(a[8], sp.x, __fmaf_rn(a[9], sp.y, __fmaf_rn(a[10], sp.z, a[11]))) * p.dist_scale;
        const int cx = min(max(__float2int_rd(ux), 0), p.ddx - 1), cy = min(max(__float2int_rd(uy), 0), p.ddy - 1),
                  cz = min(max(__float2int_rd(uz), 0), p.ddz - 1);
        const float d = __ldg(p.dist + ((size_t)cz * p.ddy + cy) * p.ddx + cx);
        // a centre outside the grid box: the scene lies inside the (convex) box, so |q - s|^2 >= |q - q'|^2 + |q' - s|^2 for the
        // projection q' of q onto the box; (ex, ey, ez) = q - q' in sub-cells
        const float ex = fmaxf(fmaxf(-ux, ux - (float)p.ddx), 0.f), ey = fmaxf(fmaxf(-uy, uy - (float)p.ddy), 0.f), ez = fmaxf(fmaxf(-uz, uz - (float)p.ddz), 0.f);
        const float e2 = (ex * ex + ey * ey + ez * ez) * p.sub_h2;
        const float thr = __fmaf_rn(snorm, sp.w, p.cull_add);
        keep = !(__fmaf_rn(d, d, e2) > thr * thr * (1.0f + 1e-5f));
      }
      const unsigned bb = __ballot_sync(0xffffffffu, keep);
      if (keep) f.glist[ns + __popc(bb & f.lt_mask)] = (uint16_t)g;
      ns += __popc(bb);
    }
    if (f.lane < FUNROLL) f.glist[ns + f.lane] = (uint16_t)f.dummy_group;
    __syncwarp();
  }
  int good = 0, qn = 0;
  constexpr int DRAIN = 32;                         // queued queries resolved per drain
  int sn_q = 0;                                     // entries in the second-level queue (weighted mode)
  auto drain_slow = [&](int take) {
    if (f.lane < take) {
      const int k = sn_q - take + f.lane;
      const int i = f.sq[k];
      const uint32_t r = f.sqr[k], va = f.sqe[k];
      good += resolve_weighted_slow(p, T, h, f.s_model[i], f.s_nrm[i], va, r & 31u, __ldg(p.vrec + va), (int)(r >> 5));
    }
    sn_q -= take;
  };
  const float gate_err = 2e-5f * snorm;             // cone shortcut: error budget of the FMA evaluation of d_rep (see resolve_weighted_slow)
  const float gate_eps = VREC_EPS_STEP * (1.0f + 1e-6f) * snorm;
  auto drain = [&](int take) {
    const int b0 = qn - take;
    int n_new = 0;
    if (f.lane < take) {
      const int i = f.q[b0 + f.lane];
      const float4 m = f.s_model[i];
      if (MODE == 0) {
        const Xf xe = FAST ? load_xf(T, h) : x;     // FAST keeps only a[] live across the loop; the exact matrix is re-read (L1)
        good += resolve_ambiguous(p, xe, m, f.qe[b0 + f.lane]);
      } else {
        const uint32_t va = f.qe[b0 + f.lane], info = f.qr[b0 + f.lane];
        const uint32_t vr = __ldg(p.vrec + va);
        const float4 nm = f.s_nrm[i];
        int known = 0;                              // 0: exact path, 1 | prior << 1: gate passes, -1: settled
        if (FAST && (vr >> 24) != 255u) {
          const float4 sn = __ldg(p.aux + (vr & 0xffffffu));      // (cell-sorted order: neighbouring voxels' representatives share sectors)
          float a[12];
          get_a(a);
          const float qx = __fmaf_rn(a[0], nm.x, __fmaf_rn(a[1], nm.y, a[2] * nm.z)), qy = __fmaf_rn(a[4], nm.x, __fmaf_rn(a[5], nm.y, a[6] * nm.z)),
                      qz = __fmaf_rn(a[8], nm.x, __fmaf_rn(a[9], nm.y, a[10] * nm.z));
          const float ae = fabsf(__fmaf_rn(sn.x, qx, __fmaf_rn(sn.y, qy, sn.z * qz))) * p.g.hf;
          const float mg = __fmaf_rn((float)(vr >> 24), gate_eps, gate_err);
          const float c30 = 0.8660254f;
          bool pass = false;
          if (ae + mg < c30 - 1e-4f) known = -1;
          else if (ae - mg > c30 + 1e-4f) {
            pass = ae + mg < 1.0f;
            if (!pass && snorm <= 1.00002f) {
              // nearly parallel normals under a rigid hypothesis (the common case near the ground truth): |d_i| <= 1 needs the ANGLE
              // of every candidate to clear ~7e-3 rad, which the cosine cannot resolve but the sine can.  theta_i >= theta_rep -
              // 1.05 eps (unit normals: pgp_set_scene / pgp_set_model normalise; chord eps <= 0.6), and theta >= sin theta =
              // |n x q| / (|n| |q|) >= |n x q| / (1.000001 snorm); with theta_i >= 7e-3: |d_i| <= 1.000021 (1 - 2.4e-5) + 2e-7 < 1.
              const float cx = __fmaf_rn(sn.y, qz, -sn.z * qy), cy = __fmaf_rn(sn.z, qx, -sn.x * qz), cz = __fmaf_rn(sn.x, qy, -sn.y * qx);
              const float c2 = __fmaf_rn(cx, cx, __fmaf_rn(cy, cy, cz * cz)) * (p.g.hf * p.g.hf);
              const float rhs = __fmaf_rn(__fmaf_rn((float)(vr >> 24), 1.05f * VREC_EPS_STEP * (1.0f + 1e-6f), 7.1e-3f), 1.00002f, 2e-5f) * snorm;
              pass = c2 > rhs * rhs;
            }
          }
          if (pass) {
            known = 1 | (sn.w != 0.f ? 2 : 0);
            if (!(info & 16u)) { good += (sn.w != 0.f) ? 0x10001 : 0x1; known = -1; }
          }
        }
        // what the cone record could not settle waits in the second-level queue until a full warp of it has gathered: on a
        // warp of the first-level queue only ~2 lanes need the (long, latency-bound) exact path
        const unsigned sb = __ballot_sync(take >= 32 ? 0xffffffffu : ((1u << take) - 1u), known >= 0);      // lanes [0, take) are here
        if (known >= 0) {
          const int slot = sn_q + __popc(sb & f.lt_mask);
          f.sq[slot] = (uint16_t)i; f.sqe[slot] = va; f.sqr[slot] = (unsigned char)(info | ((uint32_t)known << 5));
        }
        n_new = __popc(sb);
      }
    }
    qn -= take;
    if (MODE == 1) {
      sn_q += __shfl_sync(0xffffffffu, n_new, 0);       // (lane 0 always takes part in a non-empty drain)
      __syncwarp();
      if (sn_q >= 32) { drain_slow(32); __syncwarp(); }
    }
  };
  const float4* mp = f.s_model + f.lane;
  for (int k = 0; k < ns; k += FUNROLL) {
    const uint2 gg = *reinterpret_cast<const uint2*>(f.glist + k);
    const uint32_t gb[FUNROLL] = {(gg.x & 0xffffu) << 9, (gg.x >> 16) << 9, (gg.y & 0xffffu) << 9, (gg.y >> 16) << 9};     // byte offsets into the staged model
    uint32_t off[FUNROLL], sh[FUNROLL], code[FUNROLL];
    float a[12];
    if (FAST) get_a(a);
#pragma unroll
    for (int u = 0; u < FUNROLL; ++u) {
      int ix, iy, iz;
      voxel_of(a, *reinterpret_cast<const float4*>(reinterpret_cast<const char*>(mp) + gb[u]), ix, iy, iz);
      off[u] = label_slot<SMEM_TABLE>(p, f, ix, iy, iz, sh[u]);
    }
#pragma unroll
    for (int u = 0; u < FUNROLL; ++u) code[u] = __ldg(p.codes + off[u]);
    // labels: OUT = 00, IN = 01, AMBIG = 10 -> bit 0 counts, bit 1 (count mode) / either bit (weighted: IN voxels need the
    // nearest point's identity too) sends the query to phase 2
    unsigned any = 0;
#pragma unroll
    for (int u = 0; u < FUNROLL; ++u) {
      const uint32_t t = code[u] >> sh[u];
      if (MODE == 0) good += t & 1u;
      any |= t;
    }
    if (__any_sync(0xffffffffu, (any & (MODE == 0 ? 2u : 3u)) != 0u)) {
#pragma unroll
      for (int u = 0; u < FUNROLL; ++u) {
        const uint32_t lab = (code[u] >> sh[u]) & 3u;
        const bool push = MODE == 0 ? lab == 2u : lab != 0u;
        const unsigned bb = __ballot_sync(0xffffffffu, push);
        if (push) {
          const int slot = qn + __popc(bb & f.lt_mask);
          f.q[slot] = (uint16_t)((gb[u] >> 4) + f.lane);
          // rank of this voxel among the AMBIG voxels (high bit of the 2-bit label set) of its label word
          const uint32_t rank = (uint32_t)__popc(code[u] & 0xAAAAAAAAu & ((1u << sh[u]) - 1u));
          if (MODE == 0) f.qe[slot] = (off[u] << 4) | rank;
          else {
            const uint32_t va = (off[u] << 4) | (sh[u] >> 1);
            f.qe[slot] = va; f.qr[slot] = (unsigned char)(rank | ((lab & 2u) << 3));
          }
        }
        qn += __popc(bb);
      }
      __syncwarp();
      while (qn >= DRAIN) { drain(DRAIN); __syncwarp(); }
    }
  }
  while (qn > 0) { drain(min(qn, DRAIN)); __syncwarp(); }
  if (MODE == 1 && sn_q > 0) { drain_slow(sn_q); __syncwarp(); }
  return __reduce_add_sync(0xffffffffu, good);
}

template <bool SMEM_TABLE, int MODE>   // MODE 0 = count (Verify), 1 = weighted with binary priors (WeightedVerify)
__global__ void __launch_bounds__(FWARPS * 32, 1) k3_fine_kernel(const __grid_constant__ LcpParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t mbar;
  __shared__ __align__(16) float s_xf[FWARPS * 12];   // FineCtx::sa
  // shared-memory plan (k3_fine_smem on the host): model tile + one NaN group | normals (weighted) | bmrank | group spheres | survivor lists | queues
  const int cap_groups = p.tile_cap >> 5;
  float4* s_model = reinterpret_cast<float4*>(smem);
  float4* s_nrm = s_model + p.tile_cap + 32;                              // only MODE 1
  uint2* s_bmrank = reinterpret_cast<uint2*>(s_nrm + (MODE == 1 ? p.tile_cap : 0));
  float4* s_groups = reinterpret_cast<float4*>(s_bmrank + p.bmrank_words);
  uint16_t* s_glist = reinterpret_cast<uint16_t*>(s_groups + cap_groups);
  uint16_t* s_queue = reinterpret_cast<uint16_t*>(s_glist + FWARPS * (cap_groups + FUNROLL));
  uint32_t* s_qe = reinterpret_cast<uint32_t*>(s_queue + FWARPS * FQCAP);
  unsigned char* s_qr = reinterpret_cast<unsigned char*>(s_qe + FWARPS * FQCAP);  // weighted mode only, like the three below
  uint32_t* s_sqe = reinterpret_cast<uint32_t*>(s_qr + FWARPS * FQCAP);           // (FQCAP is a multiple of 4: aligned)
  uint16_t* s_sq = reinterpret_cast<uint16_t*>(s_sqe + FWARPS * SQCAP);
  unsigned char* s_sqr = reinterpret_cast<unsigned char*>(s_sq + FWARPS * SQCAP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  FineCtx f;
  f.sa = (unsigned)__cvta_generic_to_shared(s_xf + (threadIdx.x >> 5) * 12);
  f.s_model = s_model;
  f.s_nrm = s_nrm;
  f.s_groups = s_groups;
  f.table = SMEM_TABLE ? s_bmrank : p.bmrank;
  f.q = s_queue + warp * FQCAP;
  f.qe = s_qe + warp * FQCAP;
  f.qr = s_qr + warp * FQCAP;
  f.sq = s_sq + warp * SQCAP; f.sqe = s_sqe + warp * SQCAP; f.sqr = s_sqr + warp * SQCAP;
  f.glist = s_glist + warp * (cap_groups + FUNROLL);
  f.dimx = p.g.dim[0]; f.dimy = p.g.dim[1]; f.dimz = p.g.dim[2];
  f.limx = (unsigned)p.g.dim[0] * 8u - 1u; f.limy = (unsigned)p.g.dim[1] * 8u - 1u; f.limz = (unsigned)p.g.dim[2] * 8u - 1u;
  f.lane = lane; f.lt_mask = (1u << lane) - 1u;
  f.dummy_word = (uint32_t)p.g.n_blocks * 32u;

  if (threadIdx.x == 0) mbar_init(&mbar, 1);
  __syncthreads();

  for (int tile = 0; tile < p.n_tiles; ++tile) {
    const int t0 = tile * p.tile_cap;
    const int tn = min(p.tile_cap, p.nv - t0);
    const int ng = (tn + 31) >> 5;                 // groups of this tile; group `ng` is the NaN dummy
    f.dummy_group = ng;
    if (threadIdx.x == 0) {
      uint32_t bytes = (uint32_t)tn * 16u;
      uint32_t bm = (SMEM_TABLE && tile == 0) ? (uint32_t)p.bmrank_words * 8u : 0u;
      mbar_expect_tx(&mbar, bytes * (MODE == 1 ? 2u : 1u) + bm + (uint32_t)ng * 16u);
      tma_bulk_g2s(s_model, p.model + t0, bytes, &mbar);
      if (MODE == 1) tma_bulk_g2s(s_nrm, p.model_nrm + t0, bytes, &mbar);
      if (bm) tma_bulk_g2s(s_bmrank, p.bmrank, bm, &mbar);
      tma_bulk_g2s(s_groups, p.groups + (t0 >> 5), (uint32_t)ng * 16u, &mbar);
    }
    // pad slots: NaN points (their voxel converts to 0 and fails the range test); disjoint from the bulk copy's bytes
    for (int i = tn + (int)threadIdx.x; i < ng * 32 + 32; i += FWARPS * 32) s_model[i] = make_float4(__int_as_float(0x7fc00000), 0.f, 0.f, 0.f);
    mbar_wait(&mbar, tile & 1);
    __syncthreads();

    const long long n_units = p.n_bulk + (p.n - p.n_bulk) * p.split;
    const int chunk = (ng + p.split - 1) / p.split;
    for (;;) {
      long long h = 0;
      if (lane == 0) h = (long long)atomicAdd(p.work + tile, 1ull);
      h = __shfl_sync(0xffffffffu, h, 0);
      if (h >= n_units) break;
      int m_begin = 0, m_end = ng;
      const bool whole = h < p.n_bulk;
      if (!whole) {
        const long long u = h - p.n_bulk;
        h = p.n_bulk + u / p.split;
        m_begin = (int)(u % p.split) * chunk;
        m_end = min(ng, m_begin + chunk);
      }
      if (p.ready) {
        // the transforms are still being uploaded chunk by chunk on another stream (pgp_score_lcp); the counter is written by
        // the copy engine after each chunk, chunks end on 384-byte boundaries so no cache line of T spans two of them
        // ready[0] = hypotheses uploaded, ready[1] = abort flag.  A wait that exceeds ready_timeout_ns (20 ms + the time one chunk
        // needs at a pessimistic 1 GB/s, set by the host from the chunk size; the copy stream is not making progress:
        // a profiler serialising streams, a wedged DMA engine) raises the flag; every other wait then falls through at once, the
        // launch ends with garbage and the host re-scores the batch un-streamed (pgp_score_lcp).  The device never hangs.
        // The counter is read with ld.acquire.sys (the writer is the copy engine), which orders the loads of T behind it.
        unsigned long long t_start = 0;
        for (;;) {
          uint32_t have, stop;
          asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(have) : "l"(p.ready) : "memory");
          if ((long long)have > h) break;
          asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(stop) : "l"(p.ready + 1) : "memory");
          if (stop) break;
          unsigned long long now;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
          if (!t_start) t_start = now;
          else if (now - t_start > p.ready_timeout_ns) { atomicExch(p.ready + 1, 1u); __threadfence(); break; }
          __nanosleep(200);
        }
      }
      // bound on the transform's intermediates: decides whether the FMA fast path's error budget holds
      float bound = 0.f;
      {
        const Xf x = load_xf(p.T, h);
#pragma unroll
        for (int r = 0; r < 3; ++r)
          bound = fmaxf(bound, (fabsf(x.m[4 * r]) + fabsf(x.m[4 * r + 1]) + fabsf(x.m[4 * r + 2])) * p.model_rinf + fabsf(x.m[4 * r + 3]));
      }
      const bool fast = bound <= p.g.pos_bound;     // false for NaN / huge matrices: those take the reference's arithmetic
      const int tot = m_begin >= m_end ? 0 : fast ? score_hypothesis<SMEM_TABLE, true, MODE>(p, f, p.T, h, m_begin, m_end) : score_hypothesis<SMEM_TABLE, false, MODE>(p, f, p.T, h, m_begin, m_end);
      if (lane == 0) {
        if (MODE == 0) {
          if (p.n_tiles == 1 && whole) {
            p.counts[h] = (uint32_t)tot;
            if (p.scores) p.scores[h] = __fdiv_rn((float)tot, (float)p.nv);
          } else if (tot) {
            atomicAdd(p.counts + h, (uint32_t)tot);
          }
        } else {
          const uint32_t gated = (uint32_t)tot & 0xffffu, w = (uint32_t)tot >> 16;   // tile <= 8192 points keeps the halves apart
          if (p.n_tiles == 1 && whole) {
            p.counts[h] = gated;
            if (p.scores) p.scores[h] = __fdiv_rn((float)w, (float)p.nv);           // weighted_match / Scalar(n) :1765
          } else {
            if (gated) atomicAdd(p.counts + h, gated);
            if (w && p.scores) atomicAdd(reinterpret_cast<uint32_t*>(p.scores) + h, w);   // integer until k3_finalise
          }
        }
      }
    }
    __syncthreads();
  }
}

// multi-tile epilogue: counts -> scores
__global__ void k3_finalise(const uint32_t* __restrict__ counts, float* __restrict__ scores, long long n, int nv, int mode) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t v = mode == 0 ? counts[i] : reinterpret_cast<const uint32_t*>(scores)[i];
  scores[i] = __fdiv_rn((float)v, (float)nv);
}

// WeightedVerify with arbitrary priors: the reference adds the priors of the gated matches in
// model-point order in fp32 (weighted_match += ..., :1759), which is not associative, so the sum is
// formed in exactly that order: per 32-point step the lanes' contributions are folded in lane order.
// One warp per hypothesis, model read from global in ORIGINAL order.  Also the kernel behind
// pgp_registered_points / pgp_nearest_in_range (idx_out != nullptr, one hypothesis).
template <bool LISTS>   // LISTS: OUT label cull + K1c candidate lists instead of the 27-cell search
__global__ void __launch_bounds__(256) k3_weighted_ordered(const LcpParams p, int32_t* __restrict__ idx_out, int gate) {
  const int lane = threadIdx.x & 31;
  const long long h = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (h >= p.n) return;
  const Xf x = load_xf(p.T, h);
  FineCtx f;
  f.table = p.bmrank;
  f.dimx = p.g.dim[0]; f.dimy = p.g.dim[1];
  f.limx = (unsigned)p.g.dim[0] * 8u - 1u; f.limy = (unsigned)p.g.dim[1] * 8u - 1u; f.limz = (unsigned)p.g.dim[2] * 8u - 1u;
  f.dummy_word = (uint32_t)p.g.n_blocks * 32u;
  float acc = 0.f;
  int gated = 0;
  for (int base = 0; base < p.nv; base += 32) {
    const int i = base + lane;
    float w = 0.f;
    bool hit = false;
    int orig = -1;
    if (i < p.nv) {
      float tx, ty, tz;
      int cx, cy, cz;
      apply_xf(x, __ldg(p.model + i), tx, ty, tz);
      if (LISTS) {
        // the reference's own rounding sequence, then the grid's cell_coord: exactly the non-FAST voxel of the fine kernel
        const int ix = (int)min(__float2uint_rz(cell_coord(tx, p.g.lo[0], p.g.inv_hf)), f.limx), iy = (int)min(__float2uint_rz(cell_coord(ty, p.g.lo[1], p.g.inv_hf)), f.limy),
                  iz = (int)min(__float2uint_rz(cell_coord(tz, p.g.lo[2], p.g.inv_hf)), f.limz);
        uint32_t sh;
        const uint32_t off = label_slot<false>(p, f, ix, iy, iz, sh);
        if ((__ldg(p.codes + off) >> sh) & 3u) {
          uint32_t cnt;
          const uint32_t* l = wlist_of<false>(p, f, ix, iy, iz, cnt);
          const int o = nearest_in_list<1>(p, l, cnt, tx, ty, tz);
          if (o >= 0) {
            float4 ns = __ldg(p.aux_orig + o);
            if (!gate || normal_gate(x, __ldg(p.model_nrm + i), ns)) {
              hit = true; w = ns.w; orig = o;
            }
          }
        }
      } else if (query_cell(p.g, tx, ty, tz, cx, cy, cz)) {
        int pos = nearest_within(p, tx, ty, tz, cx, cy, cz);
        if (pos >= 0) {
          float4 ns = __ldg(p.aux + pos);
          if (!gate || normal_gate(x, __ldg(p.model_nrm + i), ns)) {
            hit = true; w = ns.w; orig = __float_as_int(__ldg(p.pts + pos).w);
          }
        }
      }
      if (idx_out) idx_out[i] = orig;
    }
    unsigned b = __ballot_sync(0xffffffffu, hit);
    gated += __popc(b);
    while (b) {
      int l = __ffs(b) - 1;
      b &= b - 1;
      acc = __fadd_rn(acc, __shfl_sync(0xffffffffu, w, l));
    }
  }
  if (lane == 0 && p.counts) {
    p.counts[h] = (uint32_t)gated;
    if (p.scores) p.scores[h] = __fdiv_rn(acc, (float)p.nv);
  }
}

}  // namespace

static LcpParams make_params(pgp_ctx* ctx, const Model& m, const float* T, int64_t n, uint32_t* counts, float* scores) {
  const Scene& s = ctx->scene;
  LcpParams p{};
  p.nv = m.nv;
  p.T = T; p.n = n;
  p.pts = s.pts.as<float4>(); p.aux = s.aux.as<float4>();
  p.cell_start = s.cell_start.as<uint32_t>(); p.bitmap = s.bitmap.as<uint32_t>();
  p.g = s.g;
  p.counts = counts; p.scores = scores;
  return p;
}

// true when k3_score will run k3_fine_kernel for this mode (the only kernel that can consume a batch while it is still being uploaded)
bool k3_streams_upload(pgp_ctx* ctx, int mode) {
  const Scene& s = ctx->scene;
  if (s.g.fine != 8 || ctx->force_coarse) return false;
  if (mode == PGP_LCP_WEIGHTED) return s.wlists_ready && s.priors_binary;
  return true;
}

int k3_score(pgp_ctx* ctx, const Model& m, const float* T_dev, int64_t n, int mode, uint32_t* counts_dev, float* scores_dev, uint32_t* ready_dev) {
  if (n == 0) return PGP_OK;
  Scene& s = ctx->scene;
  LcpParams p = make_params(ctx, m, T_dev, n, counts_dev, scores_dev);
  cudaStream_t st = ctx->stream;

  if (ready_dev && !k3_streams_upload(ctx, mode)) return pgp_fail(ctx, PGP_E_INVALID, "streamed upload needs the fine-grid kernel");
  if (mode == PGP_LCP_WEIGHTED && !s.priors_binary) {
    p.model = m.val_orig.as<float4>(); p.model_nrm = m.val_nrm_orig.as<float4>();
    const int T = 256;
    long long blocks = (n * 32 + T - 1) / T;
    if (s.g.fine == 8 && !ctx->force_coarse && !s.wlists_tried) { int rc = k1_build_wlists(ctx); if (rc) return rc; }
    if (s.g.fine == 8 && !ctx->force_coarse && s.wlists_ready) {
      p.bmrank = s.bmrank.as<uint2>(); p.codes = s.codes.as<uint32_t>();
      p.wcnt = s.wcnt.as<unsigned char>(); p.wword = s.wword.as<uint32_t>(); p.wlists = s.wlists.as<uint32_t>(); p.vrec = s.vrec.as<uint32_t>(); p.pts_orig = s.unsorted.as<float4>(); p.aux_orig = s.aux_orig.as<float4>();
      k3_weighted_ordered<true><<<(unsigned)blocks, T, 0, st>>>(p, nullptr, 1);
    } else {
      k3_weighted_ordered<false><<<(unsigned)blocks, T, 0, st>>>(p, nullptr, 1);
    }
    ctx->launches++;
    PGP_CUDA(ctx, cudaGetLastError());
    return PGP_OK;
  }

  p.model = m.val.as<float4>(); p.model_nrm = m.val_nrm.as<float4>();
  PGP_CUDA(ctx, ctx->work.reserve(4096));
  p.work = reinterpret_cast<unsigned long long*>(ctx->work.as<char>() + 1024);

  if (mode == PGP_LCP_WEIGHTED && s.g.fine == 8 && !ctx->force_coarse && !s.wlists_tried) {
    int rc = k1_build_wlists(ctx);      // K1c, once per scene, on the first weighted call
    if (rc) return rc;
  }
  const bool fine_ok = s.g.fine == 8 && !ctx->force_coarse && (mode == PGP_LCP_COUNT || s.wlists_ready);
  if (fine_ok) {
    // shared-memory plan of k3_fine_kernel: model tile + one NaN group | normals (weighted) | bmrank | group spheres | survivor lists | queues
    const size_t smem_max = 216 * 1024;       // of the 227 KB a CTA may take; the kernel has 8 bytes of static shared memory
    auto smem_need = [&](int cap, size_t table) {
      return (size_t)(cap + 32) * 16 + (mode == PGP_LCP_WEIGHTED ? (size_t)cap * 16 : 0) + table + (size_t)(cap >> 5) * 16 +
             (size_t)(FWARPS * ((cap >> 5) + FUNROLL)) * 2 + (size_t)FWARPS * (mode == PGP_LCP_WEIGHTED ? FQCAP * 7 + SQCAP * 7 : FQCAP * 6);
    };
    size_t bm = (size_t)s.bitmap_words * 8;
    int tile_cap = std::min((m.nv + 127) & ~127, 8192);
    if (smem_need(std::min(tile_cap, 2048), bm) > smem_max) bm = 0;          // table too big for smem: read it through L1
    // weighted mode gathers three more tables and is faster with the 96 KB left to the L1 than with the table staged (measured)
    if (mode == PGP_LCP_WEIGHTED) bm = 0;
    while (tile_cap > 128 && smem_need(tile_cap, bm) > smem_max) tile_cap -= 128;
    p.tile_cap = tile_cap;
    p.n_tiles = (m.nv + tile_cap - 1) / tile_cap;
    if (p.n_tiles > 256) return pgp_fail(ctx, PGP_E_INVALID, "validation model too large (%d points)", m.nv);
    p.bmrank = s.bmrank.as<uint2>(); p.codes = s.codes.as<uint32_t>();
    p.hdrw = s.hdrw.as<uint32_t>(); p.aslot = s.aslot.as<float4>(); p.aovf = s.aovf.as<float4>();
    p.wcnt = s.wcnt.as<unsigned char>(); p.wword = s.wword.as<uint32_t>(); p.wlists = s.wlists.as<uint32_t>(); p.vrec = s.vrec.as<uint32_t>(); p.pts_orig = s.unsorted.as<float4>(); p.aux_orig = s.aux_orig.as<float4>();
    p.bmrank_words = (int)(bm / 8);
    p.model_rinf = m.val_rinf;
    p.ready = ready_dev;
    p.ready_timeout_ns = 20000000ull + (unsigned long long)(n / 4 + 1) * 48ull;      // 20 ms + one of the four chunks at 1 GB/s (1 ns per byte)
    p.groups = m.val_groups.as<float4>();
    p.dist = ctx->group_cull ? s.dist.as<float>() : nullptr;
    p.cull_add = s.delta * (1.0f + 1e-5f) + 4.0f * s.g.inflate;
    p.dist_scale = (float)s.dist_r * 0.125f;
    p.sub_h2 = (s.g.h / (float)s.dist_r) * (s.g.h / (float)s.dist_r) * (1.0f - 1e-4f);
    p.ddx = s.g.dim[0] * s.dist_r; p.ddy = s.g.dim[1] * s.dist_r; p.ddz = s.g.dim[2] * s.dist_r;
    const size_t smem = smem_need(tile_cap, bm);
    PGP_CUDA(ctx, cudaMemsetAsync(p.work, 0, 8 * (size_t)p.n_tiles, st));
    int grid = (int)std::min<long long>((n + FWARPS - 1) / FWARPS, ctx->sm_count);
    // the last two hypotheses' worth of work per warp is handed out in quarter-model units (shorter tail of the persistent grid)
    p.split = (ctx->tail_split > 1 && n > 4ll * grid * FWARPS && tile_cap >= 4 * 32 * FUNROLL) ? ctx->tail_split : 1;
    p.n_bulk = p.split > 1 ? n - 2ll * grid * FWARPS : n;
    const long long zero_from = p.n_tiles > 1 ? 0 : p.n_bulk;       // hypotheses whose sums are accumulated with atomics
    if (zero_from < n) {
      PGP_CUDA(ctx, cudaMemsetAsync(counts_dev + zero_from, 0, (size_t)(n - zero_from) * 4, st));
      if (mode == PGP_LCP_WEIGHTED && scores_dev) PGP_CUDA(ctx, cudaMemsetAsync(scores_dev + zero_from, 0, (size_t)(n - zero_from) * 4, st));
    }
    auto launch = [&](auto kern) -> int {
      PGP_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      kern<<<grid, FWARPS * 32, smem, st>>>(p);
      return PGP_OK;
    };
    const int rc = mode == PGP_LCP_WEIGHTED ? launch(k3_fine_kernel<false, 1>) : bm ? launch(k3_fine_kernel<true, 0>) : launch(k3_fine_kernel<false, 0>);
    if (rc) return rc;
    ctx->launches++;
    if (zero_from < n && scores_dev) {
      k3_finalise<<<(unsigned)((n - zero_from + 255) / 256), 256, 0, st>>>(counts_dev + zero_from, scores_dev + zero_from, n - zero_from, m.nv, mode);
      ctx->launches++;
    }
    PGP_CUDA(ctx, cudaGetLastError());
    return PGP_OK;
  }

  const int per_pt = mode == PGP_LCP_WEIGHTED ? 32 : 16;
  // shared memory plan: model tile + bitmap (if it fits) + queues
  const size_t smem_max = 100 * 1024;     // two CTAs per SM
  const size_t qbytes = (size_t)WARPS * QCAP * 2;
  size_t bm_bytes = (size_t)s.bitmap_words * 4;
  int tile_cap = (m.nv + 3) & ~3;
  if (tile_cap > 8192) tile_cap = 8192;                    // queue entries are u16; one mbarrier tx < 1 MiB
  if ((size_t)tile_cap * per_pt + qbytes + bm_bytes > smem_max) {
    // try to keep the bitmap; shrink the tile first, drop the bitmap only if it alone is too big
    if (bm_bytes + qbytes + 1024 * (size_t)per_pt <= smem_max) {
      tile_cap = (int)((smem_max - bm_bytes - qbytes) / per_pt) & ~3;
    } else {
      bm_bytes = 0;
      if ((size_t)tile_cap * per_pt + qbytes > smem_max) tile_cap = (int)((smem_max - qbytes) / per_pt) & ~3;
    }
  }
  p.tile_cap = tile_cap;
  p.bitmap_words = (int)(bm_bytes / 4);
  p.n_tiles = (m.nv + tile_cap - 1) / tile_cap;
  const size_t smem = (size_t)tile_cap * per_pt + bm_bytes + qbytes;

  if (p.n_tiles > 256) return pgp_fail(ctx, PGP_E_INVALID, "validation model too large (%d points)", m.nv);
  PGP_CUDA(ctx, cudaMemsetAsync(p.work, 0, 8 * (size_t)p.n_tiles, st));
  if (p.n_tiles > 1) {
    PGP_CUDA(ctx, cudaMemsetAsync(counts_dev, 0, (size_t)n * 4, st));
    if (scores_dev) PGP_CUDA(ctx, cudaMemsetAsync(scores_dev, 0, (size_t)n * 4, st));
  }
  long long want = (n + WARPS - 1) / WARPS;
  int grid = (int)std::min<long long>(want, 2ll * ctx->sm_count);
  if (mode == PGP_LCP_COUNT) {
    PGP_CUDA(ctx, cudaFuncSetAttribute(k3_lcp_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k3_lcp_kernel<0><<<grid, THREADS, smem, st>>>(p);
  } else {
    PGP_CUDA(ctx, cudaFuncSetAttribute(k3_lcp_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k3_lcp_kernel<1><<<grid, THREADS, smem, st>>>(p);
  }
  ctx->launches++;
  if (p.n_tiles > 1 && scores_dev) {
    k3_finalise<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(counts_dev, scores_dev, n, m.nv, mode);
    ctx->launches++;
  }
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

// one hypothesis, per-point nearest in-range scene index in ORIGINAL model order (gate: apply the normal gate)
int k3_nearest(pgp_ctx* ctx, const Model& m, const float* T_dev, int32_t* idx_dev, int gate) {
  LcpParams p = make_params(ctx, m, T_dev, 1, nullptr, nullptr);
  p.model = m.val_orig.as<float4>(); p.model_nrm = m.val_nrm_orig.as<float4>();
  k3_weighted_ordered<false><<<1, 32, 0, ctx->stream>>>(p, idx_dev, gate);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}
