// K2 / K2b -- congruent-set (4PCS / Super4PCS) hypothesis generation on the device.
//
//   base selection   Match4PCSBase::SelectQuadrilateral / SelectRandomTriangle / TryQuadrilateral
//                    S4/algorithms/match4pcsBase.cc:507-580, 377-410, 415-464, distSegmentToSegment :81-148
//   pair extraction  MatchSuper4PCS::ExtractPairs  S4/algorithms/super4pcs.cc:193-236; the accepting filter is
//                    PairCreationFunctor::process  S4/pairCreationFunctor.h:167-253 (= brute force of 4pcs.cc:109-192)
//   quad join        MatchSuper4PCS::FindCongruentQuadrilaterals  S4/algorithms/super4pcs.cc:78-187 with
//                    IndexedNormalSet<Point,3,7>  S4/accelerators/normalset.h:71-151, normalset.hpp:114-214
//   transforms       ComputeRigidTransformFromCongruentPair :1411-1488 + ComputeRigidTransformation :1504-1614
//   driver           Perform_N_steps :1831-1877 (bases -> quads -> transforms; the verification loop is K3/K4)
//
// The hierarchical sphere rasterisation of the reference's pair extraction is only a candidate
// generator for the exact filter, so an all-pairs sweep (2k points -> 2M distance evaluations)
// yields the same pair SET.  The quad join reproduces the reference's quantisation (power-of-two
// position grid in unit-cube coordinates, 7^3 direction grid, rasterised cone) so that the quad set
// is the reference's, not merely a superset.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "pgp_internal.cuh"

namespace {

constexpr int NG = 7;                        // direction grid cells per axis (normalset: _ngSize)
__host__ __device__ inline uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull; x = (x ^ (x >> 27)) * 0x94D049BB133111EBull; return x ^ (x >> 31);
}

// ------------------------------------------------------------------------------- pair extraction
// thread i owns the pairs (j, i), j < i.  FILL = false: count;  true: write (j,i),(i,j) at the scanned offset.
template <bool FILL>
__global__ void __launch_bounds__(256) k2_pairs(const float4* __restrict__ Q, int nq, float dist, float eps, uint32_t* __restrict__ cnt,
                                                int2* __restrict__ out, long long cap) {
  __shared__ float4 tile[256];
  const int i = blockIdx.x * 256 + threadIdx.x;
  const float4 qi = i < nq ? Q[i] : make_float4(0, 0, 0, 0);
  const double d = (double)dist, e = (double)eps;      // pair_distance / pair_distance_epsilon are doubles (pairCreationFunctor.h:38-39)
  uint32_t n = 0;
  long long w = FILL && i < nq ? 2ll * cnt[i] : 0;
  const int jmax = min(nq, (int)(blockIdx.x + 1) * 256);
  for (int j0 = 0; j0 < jmax; j0 += 256) {
    __syncthreads();
    if (j0 + (int)threadIdx.x < nq) tile[threadIdx.x] = Q[j0 + threadIdx.x];
    __syncthreads();
    const int m = i < nq ? min(256, i - j0) : 0;        // only j < i
    for (int t = 0; t < m; ++t) {
      const float4 p = tile[t];
      const float dx = __fsub_rn(qi.x, p.x), dy = __fsub_rn(qi.y, p.y), dz = __fsub_rn(qi.z, p.z);
      const float dd = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz))));   // (q - p).norm()
      if (fabs((double)dd - d) > e) continue;           // std::abs(distance - pair_distance) > pair_distance_epsilon
      if (FILL) {
        if (w + 1 < cap) { out[w] = make_int2(j0 + t, i); out[w + 1] = make_int2(i, j0 + t); }
        w += 2;
      }
      ++n;
    }
  }
  if (!FILL && i < nq) cnt[i] = n;
}

struct BaseOut { int id[4]; float inv1, inv2; int ok; float d1, d2, cos_alpha; };

// largest c with off[c] <= k   (off ascending, off[0] = 0, k < off[n])
__device__ __forceinline__ int segment_of(const uint32_t* __restrict__ off, int n, uint32_t k) {
  int lo = 0, hi = n;
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (__ldg(off + mid) <= k) lo = mid; else hi = mid; }
  return lo;
}

// batched pair extraction: combo c = 2 base + edge; blockIdx.y = combo
template <bool FILL>
__global__ void __launch_bounds__(256) k2b_pairs(const float4* __restrict__ Q, int nq, const BaseOut* __restrict__ bases, float eps,
                                                 uint32_t* __restrict__ cnt, int2* __restrict__ out) {
  __shared__ float4 tile[256];
  const int c = blockIdx.y;
  const BaseOut bo = bases[c >> 1];
  if (!bo.ok) return;                                   // uniform over the CTA
  const float dist = (c & 1) ? bo.d2 : bo.d1;
  const int i = blockIdx.x * 256 + threadIdx.x;
  const float4 qi = i < nq ? Q[i] : make_float4(0, 0, 0, 0);
  const double d = (double)dist, e = (double)eps;
  uint32_t n = 0;
  long long w = FILL && i < nq ? 2ll * cnt[(size_t)c * nq + i] : 0;
  const int jmax = min(nq, (int)(blockIdx.x + 1) * 256);
  for (int j0 = 0; j0 < jmax; j0 += 256) {
    __syncthreads();
    if (j0 + (int)threadIdx.x < nq) tile[threadIdx.x] = Q[j0 + threadIdx.x];
    __syncthreads();
    const int m = i < nq ? min(256, i - j0) : 0;
    for (int t = 0; t < m; ++t) {
      const float4 p = tile[t];
      const float dx = __fsub_rn(qi.x, p.x), dy = __fsub_rn(qi.y, p.y), dz = __fsub_rn(qi.z, p.z);
      const float dd = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz))));
      if (fabs((double)dd - d) > e) continue;
      if (FILL) { out[w] = make_int2(j0 + t, i); out[w + 1] = make_int2(i, j0 + t); w += 2; }
      ++n;
    }
  }
  if (!FILL && i < nq) cnt[(size_t)c * nq + i] = n;
}
__global__ void k2b_combo_offsets(const uint32_t* __restrict__ scan, int nq, int ncombo, uint32_t* __restrict__ coff) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c <= ncombo) coff[c] = 2u * scan[(size_t)c * nq];
}

// Which of a base's congruent quads survive the per-base cap (max_sampled_csets, match4pcsBase.cc:1858-1869; the reference draws
// with rand()): a Bernoulli selection on a counter-based hash of (seed, GLOBAL base index, the quad's four model points) -- a
// property of the quad itself, independent of the order in which the join happens to enumerate it, of the chunking and of the GPU.
__device__ __forceinline__ bool quad_selected(uint64_t sb, int a1, int a2, int b1, int b2, unsigned long long thr) {
  const uint64_t hq = mix64(sb ^ mix64(((uint64_t)(uint32_t)a1 << 32) | (uint32_t)a2) ^ (((uint64_t)(uint32_t)b1 << 32) | (uint32_t)b2));
  return (hq >> 11) <= thr;
}

// ------------------------------------------------------------------------------- quad join
struct JoinParams {
  const float4* Qn;      // model points in the unit cube (worldToUnit, pairCreationFunctor.h:76-80)
  const float4* Q;       // centred model points
  const int2* A; long long n1;
  const int2* B; long long n2;
  float inv1, inv2, cos_alpha, thr2;
  float cell;            // 1 / egSize
  int eg;                // position grid cells per axis (power of two)
  uint32_t n_buckets;    // power of two (per base)
  // batched mode (bases != nullptr): A == B == all pair lists of the chunk back to back, combo c = 2 base + edge
  // owns [coff[c], coff[c+1]); even combos are the A side, odd ones the B side; base b's buckets start at b * n_buckets
  const BaseOut* bases; const uint32_t* coff; int ncombo;
  // batched mode: per base of the chunk, the cone's sample directions before the rotation onto the query direction --
  // 64 x {sin(alpha) cos(theta_t), sin(alpha) sin(theta_t)} (k2_cone_table): they depend on the base's alpha only, and every
  // pair of the base would otherwise re-evaluate the same ~44 sinf / cosf
  const float2* cone_tab;
};

// per-pair join context; false when pair k is not on the wanted side
__device__ __forceinline__ bool join_ctx(const JoinParams& p, long long k, int side, float& inv1, float& inv2, float& cos_alpha, uint32_t& bkt_base) {
  if (!p.bases) { inv1 = p.inv1; inv2 = p.inv2; cos_alpha = p.cos_alpha; bkt_base = 0; return true; }
  const int c = segment_of(p.coff, p.ncombo, (uint32_t)k);
  if ((c & 1) != side) return false;
  const BaseOut& bo = p.bases[c >> 1];
  inv1 = bo.inv1; inv2 = bo.inv2; cos_alpha = bo.cos_alpha; bkt_base = (uint32_t)(c >> 1) * p.n_buckets;
  return true;
}

__device__ __forceinline__ int pos_cell(const JoinParams& p, float x, float y, float z) {
  // coordinatesPos = p / _epsilon ; index = int(x) + int(y) g + int(z) g^2   (accelerators/utils.h:141-148)
  const int cx = (int)__fdiv_rn(x, p.cell), cy = (int)__fdiv_rn(y, p.cell), cz = (int)__fdiv_rn(z, p.cell);
  return cx + (cy + cz * p.eg) * p.eg;
}
__device__ __forceinline__ int dir_cell(float x, float y, float z) {
  // coordinatesNormal = (n/2 + 1/2) / _nepsilon, _nepsilon = 1/7 + 0.00001   (normalset.h:96,108-112)
  const float ne = 1.0f / 7.0f + 0.00001f;
  // (n / 2: the division by two is exact, so is the product with 0.5)
  const int cx = (int)__fdiv_rn(__fadd_rn(__fmul_rn(x, 0.5f), 0.5f), ne);
  const int cy = (int)__fdiv_rn(__fadd_rn(__fmul_rn(y, 0.5f), 0.5f), ne);
  const int cz = (int)__fdiv_rn(__fadd_rn(__fmul_rn(z, 0.5f), 0.5f), ne);
  return cx + (cy + cz * NG) * NG;
}
__device__ __forceinline__ void normalize3(float& x, float& y, float& z) {
  const float s = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
  const float l = __fsqrt_rn(s);
  x = __fdiv_rn(x, l); y = __fdiv_rn(y, l); z = __fdiv_rn(z, l);
}

// A side: bucket + direction cell of every pair of the first edge
__global__ void k2_join_keys(JoinParams p, uint32_t* __restrict__ bucket_of, uint32_t* __restrict__ key_of, uint32_t* __restrict__ counts) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= p.n1) return;
  float inv1, inv2, cos_alpha; uint32_t bkt_base;
  if (!join_ctx(p, k, 0, inv1, inv2, cos_alpha, bkt_base)) { bucket_of[k] = 0xffffffffu; return; }
  const int2 pr = p.A[k];
  const float4 a = p.Qn[pr.x], b = p.Qn[pr.y];
  float dx = __fsub_rn(b.x, a.x), dy = __fsub_rn(b.y, a.y), dz = __fsub_rn(b.z, a.z);
  const float ex = __fadd_rn(a.x, __fmul_rn(inv1, dx)), ey = __fadd_rn(a.y, __fmul_rn(inv1, dy)), ez = __fadd_rn(a.z, __fmul_rn(inv1, dz));
  normalize3(dx, dy, dz);
  const int pc = pos_cell(p, ex, ey, ez), dc = dir_cell(dx, dy, dz);
  const bool ok = pc >= 0 && dc >= 0 && dc < NG * NG * NG && ex >= 0.f && ey >= 0.f && ez >= 0.f && ex < 1.f && ey < 1.f && ez < 1.f;
  const uint32_t bkt = ok ? bkt_base + ((uint32_t)pc & (p.n_buckets - 1)) : 0xffffffffu;
  bucket_of[k] = bkt;
  key_of[k] = ((uint32_t)pc << 9) | (uint32_t)(dc & 511);     // eg <= 128 -> pc < 2^21
  if (ok) atomicAdd(counts + bkt, 1u);
}
__global__ void k2_join_scatter(long long n1, const uint32_t* __restrict__ bucket_of, uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n1 || bucket_of[k] == 0xffffffffu) return;
  sorted[atomicAdd(cursor + bucket_of[k], 1u)] = (uint32_t)k;
}

// The scatter above is atomic-ordered.  Every bucket of up to SORT_MAX entries is put into the order of its pairs' point ids (first,
// second) once, so that every query that walks it emits its quads in that order: deterministic output without a sort per query.
// Larger buckets (rare, skewed inputs) keep the atomic order and are flagged: a query that walks one orders its own quads.
constexpr uint32_t SORT_MAX = 32;
__global__ void k2_join_sort_buckets(const int2* __restrict__ A, const uint32_t* __restrict__ bucket_start, long long n_buckets, uint32_t* __restrict__ sorted,
                                     unsigned char* __restrict__ in_order) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_buckets) return;
  const uint32_t s = bucket_start[b], e = bucket_start[b + 1];
  const bool small = e - s <= SORT_MAX;
  in_order[b] = small ? 1 : 0;
  if (!small) return;
  for (uint32_t i = s + 1; i < e; ++i) {
    const uint32_t k = sorted[i];
    const int2 v = A[k];
    uint32_t j = i;
    while (j > s) {
      const uint32_t kp = sorted[j - 1];
      const int2 w = A[kp];
      if (!(w.x > v.x || (w.x == v.x && (w.y > v.y || (w.y == v.y && kp > k))))) break;
      sorted[j] = kp; --j;
    }
    sorted[j] = k;
  }
}

// B side: one thread per pair of the second edge; rasterise the cone of directions at angle alpha
// around the pair's direction (normalset.hpp:160-214) and collect the A pairs in the same position
// cell whose direction cell is coloured.
// Which B-side pairs can produce a quad at all: the pair's intermediate point lies in the unit cube and its position cell holds at
// least one A-side pair.  Their indices are compacted (warp ballot + one atomic per warp) so that the expensive cone rasterisation of
// k2_join_query runs on dense warps; the order of the list is arbitrary, results are indexed by the pair itself.
__global__ void __launch_bounds__(256) k2_join_probe(JoinParams p, const uint32_t* __restrict__ bucket_start, const uint32_t* __restrict__ sorted,
                                                     const uint32_t* __restrict__ key_of, uint32_t* __restrict__ list, uint32_t* __restrict__ n_list) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool live = false;
  float inv1, inv2, cos_alpha; uint32_t bkt_base;
  if (i < p.n2 && join_ctx(p, i, 1, inv1, inv2, cos_alpha, bkt_base)) {
    const int2 pr = p.B[i];
    const float4 a = p.Qn[pr.x], b = p.Qn[pr.y];
    const float dx = __fsub_rn(b.x, a.x), dy = __fsub_rn(b.y, a.y), dz = __fsub_rn(b.z, a.z);
    const float fx = __fadd_rn(a.x, __fmul_rn(inv2, dx)), fy = __fadd_rn(a.y, __fmul_rn(inv2, dy)), fz = __fadd_rn(a.z, __fmul_rn(inv2, dz));
    if (fx >= 0.f && fy >= 0.f && fz >= 0.f && fx < 1.f && fy < 1.f && fz < 1.f) {
      const int pc = pos_cell(p, fx, fy, fz);
      const uint32_t bkt = bkt_base + ((uint32_t)pc & (p.n_buckets - 1));
      const uint32_t s = bucket_start[bkt], e = bucket_start[bkt + 1];
      for (uint32_t t = s; t < e && !live; ++t) live = (int)(key_of[sorted[t]] >> 9) == pc;
    }
  }
  const unsigned bb = __ballot_sync(0xffffffffu, live);
  if (bb) {
    uint32_t base = 0;
    if ((threadIdx.x & 31) == 0) base = atomicAdd(n_list, (uint32_t)__popc(bb));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (live) list[base + __popc(bb & ((1u << (threadIdx.x & 31)) - 1u))] = (uint32_t)i;
  }
}

// Direction cells coloured by the cone of half-angle alpha around the unit direction (dx, dy, dz): the rasterisation of
// IndexedNormalSet::getNeighbors (normalset.hpp:160-214), sample for sample; col = 343 bits.
// Direction cell of the UN-normalised vector r: what normalize3 + dir_cell give -- three IEEE divisions by |r|, three by
// _nepsilon and a square root per sample, which is where the cone rasterisation spent half of its instructions -- obtained from
// u = (r_k rsqrt(|r|^2)) (0.5 / _nepsilon) + 0.5 / _nepsilon per axis.  That u is within 5e-6 of the value the reference's rounding
// sequence produces (u <= 7; every step of either chain is good to a few 1e-7 relative), so wherever it is farther than 3e-5 from
// an integer, its truncation IS the reference's cell coordinate; the (rare) samples that are not take the exact sequence.
__device__ __forceinline__ int dir_cell_of(float rx, float ry, float rz) {
  const float c = 0.5f / (1.0f / 7.0f + 0.00001f);
  const float rl = rsqrtf(__fmaf_rn(rx, rx, __fmaf_rn(ry, ry, rz * rz)));
  const float ux = __fmaf_rn(rx * rl, c, c), uy = __fmaf_rn(ry * rl, c, c), uz = __fmaf_rn(rz * rl, c, c);
  const float fx = floorf(ux), fy = floorf(uy), fz = floorf(uz);
  const float g = 3e-5f;
  const bool sure = ux - fx > g && fx + 1.0f - ux > g && uy - fy > g && fy + 1.0f - uy > g && uz - fz > g && fz + 1.0f - uz > g;   // NaN: false
  if (sure) return (int)fx + ((int)fy + (int)fz * NG) * NG;
  normalize3(rx, ry, rz);
  return dir_cell(rx, ry, rz);
}
__device__ __forceinline__ unsigned cone_samples(float cos_alpha, float& step, float& sa) {
  const float alpha = acosf(cos_alpha);
  const float perimeter = 2.0f * 3.14159265358979323846f * atanf(alpha);
  const unsigned nb = 2u * (unsigned)ceilf(perimeter * (float)NG / 2.0f);
  step = 2.0f * 3.14159265358979323846f / (float)nb;
  sa = sinf(alpha);
  return nb;
}
// one thread per (base of the chunk, sample): tab[b * 64 + t] = {sa cos(theta_t), sa sin(theta_t)}, tab[b * 64 + 63].x = number of samples
__global__ void k2_cone_table(const BaseOut* __restrict__ bases, int nb_bases, float2* __restrict__ tab) {
  const int b = blockIdx.x, t = threadIdx.x;
  if (b >= nb_bases) return;
  float step, sa;
  const unsigned ns = cone_samples(bases[b].cos_alpha, step, sa);
  float2 v = make_float2(0.f, 0.f);
  if ((unsigned)t < ns && t < 63) { const float th = (float)t * step; v = make_float2(sa * cosf(th), sa * sinf(th)); }
  if (t == 63) v.x = __uint_as_float(ns);
  tab[b * 64 + t] = v;
}
__device__ __forceinline__ void cone_cells(float dx, float dy, float dz, float cos_alpha, uint32_t col[11], const float2* __restrict__ tab = nullptr) {
#pragma unroll
  for (int t = 0; t < 11; ++t) col[t] = 0;
  float step = 0.f, sa = 0.f;
  unsigned nb;
  if (tab && __float_as_uint(__ldg(&tab[63].x)) <= 63u) nb = __float_as_uint(__ldg(&tab[63].x));
  else { tab = nullptr; nb = cone_samples(cos_alpha, step, sa); }
  // q = FromTwoVectors((0,0,1), n):  c = n.z; axis = z x n = (-n.y, n.x, 0); s = sqrt(2(1+c)); vec = axis/s; w = s/2
  const float c = dz;
  float vx, vy, vz, qw;
  if (c < -1.0f + 1e-6f) { vx = 1.f; vy = 0.f; vz = 0.f; qw = 0.f; }   // antiparallel: rotation by pi about x (Eigen picks an SVD axis)
  else {
    const float sq = sqrtf((1.0f + c) * 2.0f), invs = 1.0f / sq;
    vx = -dy * invs; vy = dx * invs; vz = 0.f; qw = sq * 0.5f;
  }
  for (unsigned t = 0; t < nb; ++t) {
    float sx, sy;
    if (tab) { const float2 cs = __ldg(tab + t); sx = cs.x; sy = cs.y; }
    else { const float th = (float)t * step; sx = sa * cosf(th); sy = sa * sinf(th); }
    const float sz = cos_alpha;
    // q * v = v + w * uv + vec x uv, uv = 2 vec x v
    const float ux = 2.0f * (vy * sz - vz * sy), uy = 2.0f * (vz * sx - vx * sz), uz = 2.0f * (vx * sy - vy * sx);
    float rx = sx + qw * ux + (vy * uz - vz * uy);
    float ry = sy + qw * uy + (vz * ux - vx * uz);
    float rz = sz + qw * uz + (vx * uy - vy * ux);
    const int id = dir_cell_of(rx, ry, rz);
    if (id >= 0 && id < NG * NG * NG) col[id >> 5] |= 1u << (id & 31);
  }
}

// `list` (optional): indices of the pairs to process, `*n_list` of them (k2_join_probe, or the count pass's own list of pairs that
// found something); without it thread i handles pair i.
template <bool FILL>
__global__ void __launch_bounds__(128) k2_join_query(JoinParams p, const uint32_t* __restrict__ bucket_start, const uint32_t* __restrict__ sorted,
                                                     const uint32_t* __restrict__ key_of, uint32_t* __restrict__ cnt, int4* __restrict__ out, long long cap,
                                                     const unsigned char* __restrict__ in_order, const uint32_t* __restrict__ list = nullptr,
                                                     const uint32_t* __restrict__ n_list = nullptr, uint32_t* __restrict__ list_out = nullptr,
                                                     uint32_t* __restrict__ n_list_out = nullptr, uint32_t* __restrict__ cone_cache = nullptr) {
  const long long t_id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (list ? t_id >= (long long)*n_list : t_id >= p.n2) return;
  const long long i = list ? (long long)list[t_id] : t_id;
  float inv1, inv2, cos_alpha; uint32_t bkt_base;
  if (FILL && cnt[i + 1] == cnt[i]) return;                // the count pass found nothing for this pair: skip the cone rasterisation
  if (!join_ctx(p, i, 1, inv1, inv2, cos_alpha, bkt_base)) { if (!FILL) cnt[i] = 0; return; }
  const int2 pr = p.B[i];
  const float4 a = p.Qn[pr.x], b = p.Qn[pr.y];
  float dx = __fsub_rn(b.x, a.x), dy = __fsub_rn(b.y, a.y), dz = __fsub_rn(b.z, a.z);
  const float fx = __fadd_rn(a.x, __fmul_rn(inv2, dx)), fy = __fadd_rn(a.y, __fmul_rn(inv2, dy)), fz = __fadd_rn(a.z, __fmul_rn(inv2, dz));
  uint32_t n = 0;
  long long w = FILL ? (long long)cnt[i] : 0;
  bool ordered = true;
  uint32_t col_keep[11];
#pragma unroll
  for (int t = 0; t < 11; ++t) col_keep[t] = 0;
  if (fx >= 0.f && fy >= 0.f && fz >= 0.f && fx < 1.f && fy < 1.f && fz < 1.f) {
    const int pc = pos_cell(p, fx, fy, fz);
    const uint32_t bkt = bkt_base + ((uint32_t)pc & (p.n_buckets - 1));
    ordered = in_order[bkt] != 0;
    const uint32_t s = bucket_start[bkt], e = bucket_start[bkt + 1];
    if (e > s) {
      normalize3(dx, dy, dz);                      // queryn
      // world-space query point for the final check (super4pcs.cc:135-139,160-170)
      const float4 wa = p.Q[pr.x], wb = p.Q[pr.y];
      const float qx = __fadd_rn(wa.x, __fmul_rn(inv2, __fsub_rn(wb.x, wa.x)));
      const float qy = __fadd_rn(wa.y, __fmul_rn(inv2, __fsub_rn(wb.y, wa.y)));
      const float qz = __fadd_rn(wa.z, __fmul_rn(inv2, __fsub_rn(wb.z, wa.z)));
      // coloured direction cells: 343 bits
      uint32_t* col = col_keep;
      cone_cells(dx, dy, dz, cos_alpha, col, p.cone_tab ? p.cone_tab + (size_t)(bkt_base / p.n_buckets) * 64 : nullptr);
      for (uint32_t t = s; t < e; ++t) {
        const uint32_t k = sorted[t];
        const uint32_t key = key_of[k];
        if ((int)(key >> 9) != pc) continue;                       // bucket collision
        const uint32_t dc = key & 511u;
        if (!((col[dc >> 5] >> (dc & 31)) & 1u)) continue;
        const int2 ap = p.A[k];
        const float4 pa = p.Q[ap.x], pb = p.Q[ap.y];
        // invPoint = pp1 + (pp2 - pp1) * invariant1 ; squaredNorm <= distance_threshold2 (sic: un-squared threshold)
        const float ix = __fadd_rn(pa.x, __fmul_rn(__fsub_rn(pb.x, pa.x), inv1));
        const float iy = __fadd_rn(pa.y, __fmul_rn(__fsub_rn(pb.y, pa.y), inv1));
        const float iz = __fadd_rn(pa.z, __fmul_rn(__fsub_rn(pb.z, pa.z), inv1));
        const float ddx = __fsub_rn(qx, ix), ddy = __fsub_rn(qy, iy), ddz = __fsub_rn(qz, iz);
        const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)), __fmul_rn(ddz, ddz));
        if (!(d2 <= p.thr2)) continue;
        if (FILL) { if (w < cap) out[w] = make_int4(ap.x, ap.y, pr.x, pr.y); ++w; }
        ++n;
      }
    }
  }
  if (FILL && n > 1 && !ordered) {
    // an over-long bucket kept its atomic order: order this query's quads by their first pair (unique key)
    const long long s0 = (long long)cnt[i], e0 = min(cap, s0 + (long long)n);
    for (long long a2 = s0 + 1; a2 < e0; ++a2) {
      const int4 v = out[a2];
      long long b2 = a2;
      while (b2 > s0 && (out[b2 - 1].x > v.x || (out[b2 - 1].x == v.x && out[b2 - 1].y > v.y))) { out[b2] = out[b2 - 1]; --b2; }
      out[b2] = v;
    }
  }
  if (!FILL) {
    cnt[i] = n;
    if (list_out && n) {                                                      // the fill / select pass runs on these only
      const uint32_t slot = atomicAdd(n_list_out, 1u);
      list_out[slot] = (uint32_t)i;
      if (cone_cache) {                                                       // ... and re-uses this pair's coloured cells
#pragma unroll
        for (int t = 0; t < 11; ++t) cone_cache[(size_t)slot * 12 + t] = col_keep[t];
      }
    }
  }
}

// ------------------------------------------------------------------------------- rigid transforms
struct V3 { float x, y, z; };
__device__ __forceinline__ V3 sub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
__device__ __forceinline__ bool normalize(V3& a) {
  const float s = dot(a, a);
  if (s == 0.f) return false;
  const float l = sqrtf(s);
  a.x /= l; a.y /= l; a.z /= l;
  return true;
}
__device__ __forceinline__ bool frame(V3 p0, V3 p1, V3 p2, V3 f[3]) {
  f[0] = sub(p1, p0);
  if (!normalize(f[0])) return false;
  const V3 e = sub(p2, p0);
  const float d = dot(e, f[0]);
  f[1] = {e.x - d * f[0].x, e.y - d * f[0].y, e.z - d * f[0].z};
  if (!normalize(f[1])) return false;
  f[2] = cross(f[0], f[1]);
  return true;
}

// One thread per quad.  Degenerate bases / quads -- for which the reference returns `true` with an
// UNINITIALISED matrix (match4pcsBase.cc:1533-1544) -- are rejected (ok = 0), as are non-orthogonal
// results (:1563, written R*R as in the reference).
__device__ bool rigid_from_quad(const float4* __restrict__ P, const float4* __restrict__ Q, const int* b, int4 quad, float* T) {
  const float4 b0 = P[b[0]], b1 = P[b[1]], b2 = P[b[2]];
  const float4 q0 = Q[quad.x], q1 = Q[quad.y], q2 = Q[quad.z];
  const V3 c1 = {(b0.x + b1.x + b2.x) / 3.0f, (b0.y + b1.y + b2.y) / 3.0f, (b0.z + b1.z + b2.z) / 3.0f};   // :1428
  const V3 c2 = {(q0.x + q1.x + q2.x) / 3.0f, (q0.y + q1.y + q2.y) / 3.0f, (q0.z + q1.z + q2.z) / 3.0f};   // :1452-1454
  V3 fp[3], fq[3];
  if (!frame({b0.x, b0.y, b0.z}, {b1.x, b1.y, b1.z}, {b2.x, b2.y, b2.z}, fp)) return false;
  if (!frame({q0.x, q0.y, q0.z}, {q1.x, q1.y, q1.z}, {q2.x, q2.y, q2.z}, fq)) return false;
  float R[3][3];
  const float fpv[3][3] = {{fp[0].x, fp[0].y, fp[0].z}, {fp[1].x, fp[1].y, fp[1].z}, {fp[2].x, fp[2].y, fp[2].z}};
  const float fqv[3][3] = {{fq[0].x, fq[0].y, fq[0].z}, {fq[1].x, fq[1].y, fq[1].z}, {fq[2].x, fq[2].y, fq[2].z}};
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) R[i][j] = fpv[0][i] * fqv[0][j] + fpv[1][i] * fqv[1][j] + fpv[2][i] * fqv[2][j];   // rotate_p^T rotate_q :1560
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float s = R[i][0] * R[0][i] + R[i][1] * R[1][i] + R[i][2] * R[2][i];
    if (s - 1.0f > 1e-6f) return false;
    if (!isfinite(s)) return false;
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    T[4 * i + 0] = R[i][0]; T[4 * i + 1] = R[i][1]; T[4 * i + 2] = R[i][2];
    const float cc = i == 0 ? c1.x : i == 1 ? c1.y : c1.z;
    T[4 * i + 3] = cc + (R[i][0] * (-c2.x) + R[i][1] * (-c2.y) + R[i][2] * (-c2.z));   // Tr(c1) R Tr(-c2) :1601-1610
  }
  return true;
}


// ------------------------------------------------------------------------------- fused fill: select, then transform
// The reference enumerates ALL congruent quads of a base and then keeps a random max_sampled_csets = 100 of them
// (match4pcsBase.cc:1858-1869) -- at 2 000 model points that is ~230 000 quads enumerated for 100 kept.  Materialising them all
// (quad, transform, flag: 68 bytes each) only to drop 99.9 % is what this pass avoids: it walks the same buckets in the same
// as the plain fill pass, applies the SAME Bernoulli selection (quad_selected: a hash of the quad itself, so the order in which a
// bucket lists its pairs is irrelevant and the buckets need not be sorted), and only for the selected quads computes the rigid
// transform and stages {order key, T} in the base's staging area (atomic slot; at most stage_cap slots).  k2c_stage_append then
// orders each base's staged entries by the key (B pair, then the A pair's points: the order of the unfused path) and keeps the
// first max_quads: exactly the hypotheses, in exactly the order, of the unfused path.
__global__ void __launch_bounds__(128) k2_join_select(JoinParams p, const uint32_t* __restrict__ bucket_start, const uint32_t* __restrict__ sorted,
                                                      const uint32_t* __restrict__ key_of, const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ list,
                                                      const uint32_t* __restrict__ n_list, const uint32_t* __restrict__ cone_cache,
                                                      const float4* __restrict__ P_unsorted, const uint32_t* __restrict__ qoff, int base_global0,
                                                      int max_quads, uint64_t seed, int stage_cap, uint32_t* __restrict__ stage_n,
                                                      uint32_t* __restrict__ stage_r, float* __restrict__ stage_T) {
  const long long t_id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t_id >= (long long)*n_list) return;
  const long long i = (long long)list[t_id];
  float inv1, inv2, cos_alpha; uint32_t bkt_base;
  if (!join_ctx(p, i, 1, inv1, inv2, cos_alpha, bkt_base)) return;
  const int b = (int)(bkt_base / p.n_buckets);            // base within the chunk
  const long long nq_b = (long long)qoff[b + 1] - (long long)qoff[b];
  const bool subsample = nq_b > max_quads;
  const double frac = fmin(1.0, 1.25 * (double)max_quads / (double)max(nq_b, 1ll));
  const unsigned long long thr = (unsigned long long)(frac * 9007199254740992.0);   // 2^53
  const uint64_t sb = mix64(seed ^ (0xABCDull + (uint64_t)(base_global0 + b)));
  uint32_t col[11];
#pragma unroll
  for (int t = 0; t < 11; ++t) col[t] = cone_cache[(size_t)t_id * 12 + t];
  const int2 pr = p.B[i];
  const float4 a = p.Qn[pr.x], bb = p.Qn[pr.y];
  const float dx = __fsub_rn(bb.x, a.x), dy = __fsub_rn(bb.y, a.y), dz = __fsub_rn(bb.z, a.z);
  const float fx = __fadd_rn(a.x, __fmul_rn(inv2, dx)), fy = __fadd_rn(a.y, __fmul_rn(inv2, dy)), fz = __fadd_rn(a.z, __fmul_rn(inv2, dz));
  const int pc = pos_cell(p, fx, fy, fz);
  const uint32_t bkt = bkt_base + ((uint32_t)pc & (p.n_buckets - 1));
  const uint32_t s = bucket_start[bkt], e = bucket_start[bkt + 1];
  const float4 wa = p.Q[pr.x], wb = p.Q[pr.y];
  const float qx = __fadd_rn(wa.x, __fmul_rn(inv2, __fsub_rn(wb.x, wa.x)));
  const float qy = __fadd_rn(wa.y, __fmul_rn(inv2, __fsub_rn(wb.y, wa.y)));
  const float qz = __fadd_rn(wa.z, __fmul_rn(inv2, __fsub_rn(wb.z, wa.z)));
  for (uint32_t t = s; t < e; ++t) {
    const uint32_t k = sorted[t];
    const uint32_t key = key_of[k];
    if ((int)(key >> 9) != pc) continue;
    const uint32_t dc = key & 511u;
    if (!((col[dc >> 5] >> (dc & 31)) & 1u)) continue;
    const int2 ap = p.A[k];
    const float4 pa = p.Q[ap.x], pb = p.Q[ap.y];
    const float ix = __fadd_rn(pa.x, __fmul_rn(__fsub_rn(pb.x, pa.x), inv1));
    const float iy = __fadd_rn(pa.y, __fmul_rn(__fsub_rn(pb.y, pa.y), inv1));
    const float iz = __fadd_rn(pa.z, __fmul_rn(__fsub_rn(pb.z, pa.z), inv1));
    const float ddx = __fsub_rn(qx, ix), ddy = __fsub_rn(qy, iy), ddz = __fsub_rn(qz, iz);
    const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)), __fmul_rn(ddz, ddz));
    if (!(d2 <= p.thr2)) continue;
    if (subsample && !quad_selected(sb, ap.x, ap.y, pr.x, pr.y, thr)) continue;
    float tq[12];
    if (!rigid_from_quad(P_unsorted, p.Q, p.bases[b].id, make_int4(ap.x, ap.y, pr.x, pr.y), tq)) continue;
    const uint32_t slot = atomicAdd(stage_n + b, 1u);
    if (slot < (uint32_t)stage_cap) {
      const size_t o = (size_t)b * stage_cap + slot;
      // order key = the position the unfused path gives this quad: by B pair, then by the A pair's points
      stage_r[2 * o] = (uint32_t)i; stage_r[2 * o + 1] = ((uint32_t)ap.x << 16) | (uint32_t)ap.y;
#pragma unroll
      for (int c = 0; c < 12; ++c) stage_T[12 * o + c] = tq[c];
    }
  }
}

// One CTA of 1024 threads: outoff[b] = exclusive scan of count(b) (a base's output size, capped by the caller) over the nb bases
// of a chunk, outoff[nb] = the total.  Thread t owns the contiguous bases [t per, (t + 1) per).
template <class Count>
__device__ __forceinline__ void capped_base_scan(int nb, Count count, uint32_t* __restrict__ outoff) {
  __shared__ uint32_t s_warp[32];
  const int per = (nb + 1023) / 1024, b0 = threadIdx.x * per, b1 = min(nb, b0 + per);
  uint32_t mine = 0;
  for (int b = b0; b < b1; ++b) mine += count(b);
  uint32_t incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)(threadIdx.x & 31) >= o) incl += t; }
  if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = incl;
  __syncthreads();
  uint32_t run = incl - mine;
  for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) run += s_warp[w];
  for (int b = b0; b < b1; ++b) { outoff[b] = run; run += count(b); }
  if (threadIdx.x == 1023) outoff[nb] = run;
}

// per-base output sizes min(staged, max_quads) -> exclusive scan; flags a staging overflow
__global__ void __launch_bounds__(1024) k2c_stage_out(const uint32_t* __restrict__ stage_n, int nb, int max_quads, int stage_cap, uint32_t* __restrict__ outoff,
                                                      uint32_t* __restrict__ overflow) {
  for (int b = threadIdx.x; b < nb; b += 1024)
    if (stage_n[b] > (uint32_t)stage_cap) atomicOr(overflow, 1u);
  capped_base_scan(nb, [&](int b) { return min(stage_n[b], (uint32_t)max_quads); }, outoff);
}

// one warp per base: rank of every staged entry by its order key (unique within a base), the first max_quads go out in that order
__global__ void __launch_bounds__(256) k2c_stage_append(const uint32_t* __restrict__ stage_n, const uint32_t* __restrict__ stage_r, const float* __restrict__ stage_T,
                                                        int nb, int max_quads, int stage_cap, const uint32_t* __restrict__ outoff, float* __restrict__ dst,
                                                        long long room) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= nb) return;
  const uint32_t n = min(stage_n[b], (uint32_t)stage_cap);
  const uint2* r = reinterpret_cast<const uint2*>(stage_r) + (size_t)b * stage_cap;
  for (uint32_t e = lane; e < n; e += 32) {
    const uint2 mine = r[e];
    uint32_t rank = 0;
    for (uint32_t j = 0; j < n; ++j) { const uint2 v = r[j]; rank += (v.x < mine.x || (v.x == mine.x && v.y < mine.y)) ? 1u : 0u; }
    if (rank >= (uint32_t)max_quads) continue;
    const long long o = (long long)outoff[b] + rank;
    if (o >= room) continue;
    const float* src = stage_T + 12 * ((size_t)b * stage_cap + e);
#pragma unroll
    for (int c = 0; c < 12; ++c) dst[12 * o + c] = src[c];
  }
}

__global__ void k2_rigid(const float4* __restrict__ P_unsorted, const float4* __restrict__ Q, const int* __restrict__ base4, const int4* __restrict__ quads,
                         long long n, float* __restrict__ T, uint8_t* __restrict__ ok) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int b[4] = {base4[0], base4[1], base4[2], base4[3]};
  float t[12];
  const bool good = rigid_from_quad(P_unsorted, Q, b, quads[i], t);
#pragma unroll
  for (int c = 0; c < 12; ++c) T[12 * i + c] = good ? t[c] : 0.f;
  ok[i] = good ? 1 : 0;
}

// ------------------------------------------------------------------------------- base selection
// One CTA per base.  Same procedure as SelectQuadrilateral in operMode 0, with a counter-based RNG
// instead of rand(): a random first point, the widest of `trials` random triangles whose two edges
// stay below max_base_diameter, the most coplanar fourth point that is not too close to the three,
// then the pairing with the smallest segment-to-segment distance and its two invariants (in double,
// as distSegmentToSegment is instantiated with Scalar = double, :428-435).

// distSegmentToSegment<Vector3f, double> (match4pcsBase.cc:81-148): the difference vectors and their dot products are fp32
// (Eigen's a0 b0 + (a1 b1 + a2 b2)), the case analysis runs in double (Scalar is deduced from the double invariants, :428-435),
// and the closing distance |w + inv1 u - inv2 v| is fp32 again with the invariants narrowed to float.  The symmetric pairings
// (i,j,k,l) / (k,l,i,j) tie in exact arithmetic, so which one TryQuadrilateral keeps depends on exactly this rounding.
__device__ float seg_seg(const float* p1, const float* p2, const float* q1, const float* q2, double& inv1, double& inv2) {
  const double kSmall = 0.0001;
  float u[3], v[3], w[3];
  for (int k = 0; k < 3; ++k) { u[k] = __fsub_rn(p2[k], p1[k]); v[k] = __fsub_rn(q2[k], q1[k]); w[k] = __fsub_rn(p1[k], q1[k]); }
  const double a = (double)dot3_tree(u[0], u[1], u[2], u[0], u[1], u[2]), b = (double)dot3_tree(u[0], u[1], u[2], v[0], v[1], v[2]),
               c = (double)dot3_tree(v[0], v[1], v[2], v[0], v[1], v[2]), d = (double)dot3_tree(u[0], u[1], u[2], w[0], w[1], w[2]),
               e = (double)dot3_tree(v[0], v[1], v[2], w[0], w[1], w[2]);
  const double f = a * c - b * b;
  double s1 = 0.0, s2 = f, t1 = 0.0, t2 = f;
  if (f < kSmall) { s1 = 0.0; s2 = 1.0; t1 = e; t2 = c; }
  else {
    s1 = (b * e - c * d); t1 = (a * e - b * d);
    if (s1 < 0.0) { s1 = 0.0; t1 = e; t2 = c; }
    else if (s1 > s2) { s1 = s2; t1 = e + b; t2 = c; }
  }
  if (t1 < 0.0) {
    t1 = 0.0;
    if (-d < 0.0) s1 = 0.0; else if (-d > a) s1 = s2; else { s1 = -d; s2 = a; }
  } else if (t1 > t2) {
    t1 = t2;
    if ((-d + b) < 0.0) s1 = 0; else if ((-d + b) > a) s1 = s2; else { s1 = (-d + b); s2 = a; }
  }
  inv1 = (fabs(s1) < kSmall ? 0.0 : s1 / s2);
  inv2 = (fabs(t1) < kSmall ? 0.0 : t1 / t2);
  const float i1 = (float)inv1, i2 = (float)inv2;
  float r[3];
  for (int k = 0; k < 3; ++k) r[k] = __fsub_rn(__fadd_rn(w[k], __fmul_rn(i1, u[k])), __fmul_rn(i2, v[k]));
  return __fsqrt_rn(dot3_tree(r[0], r[1], r[2], r[0], r[1], r[2]));
}

// TryQuadrilateral (match4pcsBase.cc:415-464): all ordered (i,j) with the remaining two in ascending order; the pairing with the
// smallest segment-to-segment distance wins (first minimum), its invariants are kept and the ids are re-ordered accordingly.
__device__ void try_quadrilateral(const float4* __restrict__ P, const int ids[4], BaseOut& o) {
  float pt[4][3];
  for (int k = 0; k < 4; ++k) { const float4 q = P[ids[k]]; pt[k][0] = q.x; pt[k][1] = q.y; pt[k][2] = q.z; }
  float min_d = 3.4028234663852886e38f; int bb[4] = {-1, -1, -1, -1}; float inv1 = 0.f, inv2 = 0.f;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      if (i == j) continue;
      int k = 0; while (k == i || k == j) k++;
      int l = 0; while (l == i || l == j || l == k) l++;
      double li1, li2;
      const float sd = seg_seg(pt[i], pt[j], pt[k], pt[l], li1, li2);
      if (sd < min_d) { min_d = sd; bb[0] = i; bb[1] = j; bb[2] = k; bb[3] = l; inv1 = (float)li1; inv2 = (float)li2; }
    }
  if (bb[0] >= 0) {
    for (int k = 0; k < 4; ++k) o.id[k] = ids[bb[k]];
    o.inv1 = inv1; o.inv2 = inv2; o.ok = 1;
    const float4 a0 = P[o.id[0]], a1 = P[o.id[1]], a2 = P[o.id[2]], a3 = P[o.id[3]];
    V3 e1 = {a1.x - a0.x, a1.y - a0.y, a1.z - a0.z}, e2 = {a3.x - a2.x, a3.y - a2.y, a3.z - a2.z};
    o.d1 = sqrtf(dot(e1, e1)); o.d2 = sqrtf(dot(e2, e2));     // distance1 / distance6 (:1951-1952)
    normalize(e1); normalize(e2);
    o.cos_alpha = dot(e1, e2);                                // super4pcs.cc:109-111
  }
}

__global__ void __launch_bounds__(256) k2_select_bases(const float4* __restrict__ P, int n, float max_diam, int trials, uint64_t seed, int base_lo, BaseOut* __restrict__ out) {
  __shared__ float s_val[256];
  __shared__ int s_idx[256];
  __shared__ int s_tri[3];
  const int base = base_lo + blockIdx.x, tid = threadIdx.x;      // the draws depend on the GLOBAL base index only (bases shard across GPUs)
  BaseOut o{};
  for (int attempt = 0; attempt < 16; ++attempt) {
    const uint64_t s0 = mix64(seed ^ mix64(((uint64_t)base << 8) | (uint64_t)attempt));
    const int first = (int)(mix64(s0) % (uint64_t)n);
    const float4 p0 = P[first];
    const float sqmax = max_diam * max_diam;
    // widest admissible triangle (first maximum in trial order wins, like the serial loop's strict '>')
    float best = 0.f; int best_t = 0x7fffffff;
    for (int t = tid; t < trials; t += 256) {
      const uint64_t r = mix64(s0 + 2 * (uint64_t)t + 1), r2 = mix64(s0 + 2 * (uint64_t)t + 2);
      const float4 a = P[(int)(r % (uint64_t)n)], b = P[(int)(r2 % (uint64_t)n)];
      const V3 u = {a.x - p0.x, a.y - p0.y, a.z - p0.z}, w = {b.x - p0.x, b.y - p0.y, b.z - p0.z};
      const V3 cr = cross(u, w);
      const float wide = sqrtf(dot(cr, cr));
      if (wide > best && dot(u, u) < sqmax && dot(w, w) < sqmax) { best = wide; best_t = t; }
    }
    s_val[tid] = best; s_idx[tid] = best_t;
    __syncthreads();
    for (int o2 = 128; o2 > 0; o2 >>= 1) {
      if (tid < o2) {
        const float v = s_val[tid + o2]; const int ix = s_idx[tid + o2];
        if (v > s_val[tid] || (v == s_val[tid] && ix < s_idx[tid])) { s_val[tid] = v; s_idx[tid] = ix; }
      }
      __syncthreads();
    }
    const int bt = s_idx[0];
    const bool have_tri = s_val[0] > 0.f && bt != 0x7fffffff;
    __syncthreads();
    if (!have_tri) continue;
    const int i1 = first, i2 = (int)(mix64(s0 + 2 * (uint64_t)bt + 1) % (uint64_t)n), i3 = (int)(mix64(s0 + 2 * (uint64_t)bt + 2) % (uint64_t)n);
    const float4 p1 = P[i1], p2 = P[i2], p3 = P[i3];
    // plane through the three points: A x + B y + C z = 1 (:527-546, evaluated in double, stored in float)
    const double x1 = p1.x, y1 = p1.y, z1 = p1.z, x2 = p2.x, y2 = p2.y, z2 = p2.z, x3 = p3.x, y3 = p3.y, z3 = p3.z;
    const float denom = (float)(-x3 * y2 * z1 + x2 * y3 * z1 + x3 * y1 * z2 - x1 * y3 * z2 - x2 * y1 * z3 + x1 * y2 * z3);
    if (denom == 0.f) continue;
    const float A = (float)((-y2 * z1 + y3 * z1 + y1 * z2 - y3 * z2 - y1 * z3 + y2 * z3) / denom);
    const float B = (float)((x2 * z1 - x3 * z1 - x1 * z2 + x3 * z2 + x1 * z3 - x2 * z3) / denom);
    const float C = (float)((-x2 * y1 + x3 * y1 + x1 * y2 - x3 * y2 - x1 * y3 + x2 * y3) / denom);
    const float too_small = (max_diam * 0.1f) * (max_diam * 0.1f);
    float bd = 3.4e38f; int bi = 0x7fffffff;
    for (int i = tid; i < n; i += 256) {
      const float4 q = P[i];
      const V3 qv = {q.x, q.y, q.z};
      const V3 d1 = sub(qv, {p1.x, p1.y, p1.z}), d2 = sub(qv, {p2.x, p2.y, p2.z}), d3 = sub(qv, {p3.x, p3.y, p3.z});
      if (dot(d1, d1) >= too_small && dot(d2, d2) >= too_small && dot(d3, d3) >= too_small) {
        const float dist = fabsf((float)((double)(A * q.x + B * q.y + C * q.z) - 1.0));
        if (dist < bd) { bd = dist; bi = i; }
      }
    }
    s_val[tid] = bd; s_idx[tid] = bi;
    __syncthreads();
    for (int o2 = 128; o2 > 0; o2 >>= 1) {
      if (tid < o2) {
        const float v = s_val[tid + o2]; const int ix = s_idx[tid + o2];
        if (v < s_val[tid] || (v == s_val[tid] && ix < s_idx[tid])) { s_val[tid] = v; s_idx[tid] = ix; }
      }
      __syncthreads();
    }
    const int i4 = s_idx[0];
    __syncthreads();
    if (i4 == 0x7fffffff) continue;
    if (tid == 0) {
      const int ids[4] = {i1, i2, i3, i4};
      try_quadrilateral(P, ids, o);
      s_tri[0] = o.ok;
    }
    __syncthreads();
    if (s_tri[0]) break;
  }
  if (tid == 0) out[blockIdx.x] = o;
}

// ------------------------------------------------------------------------------- StoCS (operMode 1, the shipped generator)
// Point-pair feature of Match4PCSBase::computePPF (match4pcsBase.cc:582-598) with approximate_bin (:150-160):
//   { |u| in mm -> nearest multiple of 5,  angle(n1,u), angle(n2,u), angle(n1,n2) in degrees -> nearest multiple of 10 },  u = p1 - p2.
// fp32 in Eigen's evaluation order (3-element reductions are a0 + (a1 + a2)); atan2f is emulated by rounding the double result.
// Packed key: d/5 << 15 | a1/10 << 10 | a2/10 << 5 | a3/10 (d < 10.24 m, angles in [0, 180]); PPF_NOKEY for anything else.
constexpr uint32_t PPF_NOKEY = 0xffffffffu;
constexpr int PPF_D5_MAX = 2048;
__host__ __device__ inline int approximate_bin(int val, int disc) {
  const int lower = val - (val % disc), upper = lower + disc;
  return (val - lower < upper - val) ? lower : upper;
}
// The angle features enter the key only through approximate_bin(int(deg), 10) = 10 floor((deg + 5) / 10) (deg >= 0: atan2 of a
// norm): the key changes at deg = 5, 15, ... 175 only.  The fast path evaluates the angle with the fp32 atan2f (a few ulp, i.e.
// < 1e-4 deg off the reference's correctly rounded value) and returns the bin unless deg lies within 2e-3 deg of such a boundary;
// there, and for non-finite inputs, the reference's own arithmetic decides (correctly rounded atan2 via double, float x 180,
// double / pi, truncation).  Bit-equal keys at a fraction of the double-precision work.
__device__ __forceinline__ int ppf_angle_exact(float y, float x) {
  const float a = (float)atan2((double)y, (double)x);           // atan2f
  return (int)((double)__fmul_rn(a, 180.0f) / 3.14159265358979323846);
}
__device__ __forceinline__ int ppf_angle_bin(float y, float x) {      // = approximate_bin(ppf_angle_exact(y, x), 10)
  const float t = __fmaf_rn(atan2f(y, x), 5.729578f, 0.5f);            // (deg + 5) / 10
  const float r = rintf(t);
  if (fabsf(t - r) > 2e-4f && t > 0.25f && t < 18.75f) return 10 * (int)t;
  return approximate_bin(ppf_angle_exact(y, x), 10);
}
__device__ __forceinline__ void ppf_raw(const float4 p1, const float4 n1, const float4 p2, const float4 n2, int k[4]) {
  const float ux = __fsub_rn(p1.x, p2.x), uy = __fsub_rn(p1.y, p2.y), uz = __fsub_rn(p1.z, p2.z);
  const float un = __fsqrt_rn(dot3_tree(ux, uy, uz, ux, uy, uz));
  auto crossn = [](float ax, float ay, float az, float bx, float by, float bz) {
    const float cx = __fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by)), cy = __fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz)),
                cz = __fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx));
    return __fsqrt_rn(dot3_tree(cx, cy, cz, cx, cy, cz));
  };
  k[0] = approximate_bin((int)__fmul_rn(un, 1000.0f), 5);
  k[1] = ppf_angle_bin(crossn(n1.x, n1.y, n1.z, ux, uy, uz), dot3_tree(n1.x, n1.y, n1.z, ux, uy, uz));
  k[2] = ppf_angle_bin(crossn(n2.x, n2.y, n2.z, ux, uy, uz), dot3_tree(n2.x, n2.y, n2.z, ux, uy, uz));
  k[3] = ppf_angle_bin(crossn(n1.x, n1.y, n1.z, n2.x, n2.y, n2.z), dot3_tree(n1.x, n1.y, n1.z, n2.x, n2.y, n2.z));
}
__host__ __device__ inline uint32_t ppf_pack(const int k[4]) {
  if (k[0] < 0 || k[0] % 5 || k[0] / 5 >= PPF_D5_MAX) return PPF_NOKEY;
  for (int t = 1; t < 4; ++t) if (k[t] < 0 || k[t] > 180 || k[t] % 10) return PPF_NOKEY;
  return ((uint32_t)(k[0] / 5) << 15) | ((uint32_t)(k[1] / 10) << 10) | ((uint32_t)(k[2] / 10) << 5) | (uint32_t)(k[3] / 10);
}
__device__ __forceinline__ uint32_t ppf_key(const float4 p1, const float4 n1, const float4 p2, const float4 n2) {
  int k[4];
  ppf_raw(p1, n1, p2, n2, k);
  return ppf_pack(k);
}
__device__ __forceinline__ bool ppf_present(const uint32_t* __restrict__ bits, uint32_t key) {
  return key != PPF_NOKEY && ((__ldg(bits + (key >> 5)) >> (key & 31)) & 1u);
}

// keys of arbitrary index pairs of one cloud (test hook + the map builder): pairs == nullptr -> all ordered (i, j), i != j, row-major
__global__ void k2s_keys(const float4* __restrict__ pts, const float4* __restrict__ nrm, int n, const int2* __restrict__ pairs, long long np,
                         int32_t* __restrict__ keys4, uint32_t* __restrict__ packed) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= np) return;
  int i, j;
  if (pairs) { i = pairs[t].x; j = pairs[t].y; } else { i = (int)(t / n); j = (int)(t % n); }
  int k[4] = {-1, -1, -1, -1};
  if (i != j || pairs) ppf_raw(pts[i], nrm[i], pts[j], nrm[j], k);
  if (keys4) { keys4[4 * t] = k[0]; keys4[4 * t + 1] = k[1]; keys4[4 * t + 2] = k[2]; keys4[4 * t + 3] = k[3]; }
  if (packed) packed[t] = (i != j || pairs) ? ppf_pack(k) : PPF_NOKEY;
}

// std::discrete_distribution<int>(w, w + n)(std::default_random_engine) exactly as libstdc++ evaluates it: probabilities
// p_i = w_i / sum (double, sequential std::accumulate), cumulative sums (sequential std::partial_sum, last forced to 1.0),
// u = generate_canonical<double, 53>(minstd_rand0) = two draws, index = lower_bound(cp, u).  One thread; sequential on purpose.
struct MinStd {
  uint32_t x;
  __device__ explicit MinStd(uint32_t seed) { x = seed % 2147483647u; if (x == 0) x = 1; }
  __device__ uint32_t next() { x = (uint32_t)(((uint64_t)x * 16807ull) % 2147483647ull); return x; }
  __device__ double canonical() {
    const double r = 2147483646.0;                 // max - min + 1
    double sum = (double)(next() - 1u);
    sum += (double)(next() - 1u) * r;
    double ret = sum / (r * r);
    if (ret >= 1.0) ret = 0.99999999999999988897769753748;   // nextafter(1, 0)
    return ret;
  }
};
__device__ int discrete_draw(const float* __restrict__ w, int n, MinStd& g) {
  if (n < 2) return 0;                             // _M_prob.size() < 2: no cumulative table, operator() returns 0 without drawing
  double sum = 0.0;
  for (int i = 0; i < n; ++i) sum += (double)w[i];
  const double u = g.canonical();
  double acc = 0.0;
  for (int i = 0; i < n - 1; ++i) {
    acc += (double)w[i] / sum;
    if (!(acc < u)) return i;                      // lower_bound: first cp_i >= u
  }
  return n - 1;                                    // cp.back() = 1.0 >= u always
}

struct StocsParams {
  const float4* P;        // centred scene points, original order
  const float4* aux;      // unit normal + prior, original order
  int n;
  const uint32_t* bits;   // presence bitset of the model's PPF map
  float* curr;            // n_bases x n scratch (curr_probabilities_)
  uint64_t seed;
  int base0;
};
__host__ __device__ inline uint32_t stocs_base_seed(uint64_t seed, int base, int attempt) {
  return (uint32_t)(mix64(seed ^ mix64(0x570C5ull + ((uint64_t)base << 8) + (uint64_t)attempt)) >> 32);
}

// Block-cooperative std::discrete_distribution draw over the weights w[0..n) (shared memory), bit-identical to discrete_draw above:
// the steps whose result depends on the evaluation order stay sequential on thread 0 unless they are provably exact, everything
// else is spread over the CTA.
//   normalise (the reference divides the float weights by their sequential float sum first, match4pcsBase.cc:652-657 etc.):
//     the sum is a chain of float adds on thread 0 -- or, when every non-zero weight is the same value c (binary priors) and k c is
//     exactly representable, the exact product k c (= what the chain gives, no rounding ever happens);
//   p_i = (double) w_i / sum_d with sum_d = sequential double sum: a double sum of <= 2^12 floats whose exponents span <= 17 binades
//     never rounds, so any summation order gives the sequential result and the CTA reduces it as a tree; otherwise thread 0 chains;
//   cumulative probabilities: the sequential rounding chain of std::partial_sum, thread 0, up to the drawn index.
// acc = c; then (m - 1) times acc = fl(acc + c): the float chain std::accumulate runs over m copies of the same value c > 0
// (zeros in between change nothing), in O(binades) steps instead of m.  Inside one binade [2^e, 2^(e+1)) every partial sum is a
// multiple of U = ulp and, while the exact acc + c stays below 2^(e+1), fl(acc + c) - acc is the same multiple d of U for every
// acc of the same parity -- and after one explicit step the parity no longer changes (a tie c = qU + U/2 rounds to the even
// neighbour, which makes d even).  So: one real add, read d off it, jump over all the following steps that stay regular, repeat.
#ifdef __CUDA_ARCH__
#define PGP_FADD_RN(a, b) __fadd_rn(a, b)
#define PGP_FSUB_RN(a, b) __fsub_rn(a, b)
#else
#define PGP_FADD_RN(a, b) ((a) + (b))      // host: the library is compiled with -ffp-contract=off, float stays float on x86-64 (SSE)
#define PGP_FSUB_RN(a, b) ((a) - (b))
#endif
__host__ __device__ inline float chain_sum_equal(float c, long long m) {
  if (m <= 0) return 0.f;
  float acc = c;
  long long rem = m - 1;
  while (rem > 0) {
    const float next = PGP_FADD_RN(acc, c);
    --rem;
    if (!(next > acc)) return acc;                                    // c is below half an ulp of acc: the chain has stalled
    int e0, e1;
    frexpf(acc, &e0); frexpf(next, &e1);
    const float d = PGP_FSUB_RN(next, acc);                              // exact (next <= 2 acc)
    acc = next;
    if (e0 != e1 || rem == 0) continue;                                // crossed into the next binade: its step is read off the next add
    // one more explicit step so that the parity of acc / U has settled (ties-to-even), then the regular run
    const float next2 = PGP_FADD_RN(acc, c);
    --rem;
    int e2; frexpf(next2, &e2);
    const float d2 = PGP_FSUB_RN(next2, acc);
    if (!(next2 > acc)) return acc;
    acc = next2;
    if (e2 != e1 || rem == 0) continue;
    (void)d;
    const double top = ldexp(1.0, e1);                                 // frexp: acc in [2^(e1-1), 2^e1)
    const double R = top - (double)c - (double)acc;                    // exact
    long long j = R > 0 ? (long long)ceil(R / (double)d2) : 0;         // steps k = 0 .. j-1 start from acc + k d2 with acc + k d2 + c < top
    if (j > rem) j = rem;
    acc = (float)((double)acc + (double)j * (double)d2);               // exact: a multiple of U below 2^(e1) (or equal to it)
    rem -= j;
  }
  return acc;
}

constexpr int K2S_T = 128;   // threads per base: the order-sensitive chains run on one thread, so what counts is how many bases an SM holds
__device__ int block_discrete_draw(float* w, double* wd, int n, MinStd& gen, bool normalise, int tid, float* s_f, double* s_dd, int* s_i) {
  // ---- statistics of the non-zero weights: count, min / max biased exponent, all-equal flag
  int cnt = 0, emin = 255, emax = 0;
  float first = 0.f; bool same = true;
  for (int i = tid; i < n; i += K2S_T) {
    const float v = w[i];
    if (v != 0.f) {
      const int e = (__float_as_int(v) >> 23) & 255;
      emin = min(emin, e); emax = max(emax, e); ++cnt;
      if (first == 0.f) first = v; else same &= v == first;
    }
  }
  // block reduce (warp shuffles, then 8 warps through shared memory)
  const int lane = tid & 31, wp = tid >> 5;
  for (int o = 16; o; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o); emin = min(emin, __shfl_xor_sync(0xffffffffu, emin, o)); emax = max(emax, __shfl_xor_sync(0xffffffffu, emax, o));
    const float of = __shfl_xor_sync(0xffffffffu, first, o); const int os = __shfl_xor_sync(0xffffffffu, (int)same, o);
    same = same && os && (of == 0.f || first == 0.f || of == first);
    if (first == 0.f) first = of;
  }
  if (lane == 0) { s_i[wp * 4] = cnt; s_i[wp * 4 + 1] = emin; s_i[wp * 4 + 2] = emax; s_i[wp * 4 + 3] = same; s_f[wp] = first; }
  __syncthreads();
  cnt = 0; emin = 255; emax = 0; same = true; first = 0.f;
  for (int k = 0; k < K2S_T / 32; ++k) {
    cnt += s_i[k * 4]; emin = min(emin, s_i[k * 4 + 1]); emax = max(emax, s_i[k * 4 + 2]);
    const float of = s_f[k];
    same = same && s_i[k * 4 + 3] && (of == 0.f || first == 0.f || of == first);
    if (first == 0.f) first = of;
  }
  __syncthreads();
  if (normalise) {
    // exact shortcut: k copies of c, with k * mantissa(c) < 2^24
    float fsum;
    bool exact = false;
    if (same && cnt > 0) {
      const uint32_t mant = ((uint32_t)__float_as_int(first) & 0x7fffffu) | 0x800000u;
      const uint32_t odd = mant >> (__ffs((int)mant) - 1);                 // significant bits of c
      exact = emin > 0 && (unsigned long long)odd * (unsigned long long)cnt < (1ull << 24);
    }
    if (exact) fsum = __fmul_rn((float)cnt, first);
    else if (same && cnt > 0 && emin > 0 && first > 0.f) fsum = chain_sum_equal(first, cnt);      // (every thread, redundantly: ~25 short rounds)
    else {
      if (tid == 0) { float acc = 0.f; for (int i = 0; i < n; ++i) acc = __fadd_rn(acc, w[i]); s_f[8] = acc; }
      __syncthreads();
      fsum = s_f[8];
      __syncthreads();
    }
    for (int i = tid; i < n; i += K2S_T) w[i] = __fdiv_rn(w[i], fsum);
    __syncthreads();
    if (cnt > 0) {                                                         // exponents after the division: recompute (cheap) for the double-sum test
      emin = 255; emax = 0;
      for (int i = tid; i < n; i += K2S_T) { const float v = w[i]; if (v != 0.f) { const int e = (__float_as_int(v) >> 23) & 255; emin = min(emin, e); emax = max(emax, e); } }
      for (int o = 16; o; o >>= 1) { emin = min(emin, __shfl_xor_sync(0xffffffffu, emin, o)); emax = max(emax, __shfl_xor_sync(0xffffffffu, emax, o)); }
      if (lane == 0) { s_i[wp * 4 + 1] = emin; s_i[wp * 4 + 2] = emax; }
      __syncthreads();
      emin = 255; emax = 0;
      for (int k = 0; k < K2S_T / 32; ++k) { emin = min(emin, s_i[k * 4 + 1]); emax = max(emax, s_i[k * 4 + 2]); }
      __syncthreads();
    }
  }
  if (n < 2) return 0;                                                     // (as discrete_draw: no table, no draw)
  // ---- sum_d
  for (int i = tid; i < n; i += K2S_T) wd[i] = (double)w[i];
  __syncthreads();
  int lg = 0; while ((1 << lg) < n) ++lg;
  const bool dexact = cnt > 0 && emin > 0 && (emax - emin) + lg <= 29;     // 24-bit terms, sum below 2^(emax + 1 + lg): fits 53 bits
  double dsum;
  if (dexact) {
    double part = 0.0;
    for (int i = tid; i < n; i += K2S_T) part += wd[i];
    for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) s_dd[wp] = part;
    __syncthreads();
    dsum = 0.0;
    for (int k = 0; k < K2S_T / 32; ++k) dsum += s_dd[k];
    __syncthreads();
  } else {
    if (tid == 0) { double acc = 0.0; for (int i = 0; i < n; ++i) acc += wd[i]; s_dd[8] = acc; }
    __syncthreads();
    dsum = s_dd[8];
    __syncthreads();
  }
  for (int i = tid; i < n; i += K2S_T) wd[i] = wd[i] / dsum;
  __syncthreads();
  // ---- the draw: the first i < n - 1 whose sequential partial sum reaches u.  The chain of n double adds is replaced by a block
  // scan: any association of the same non-negative terms (total ~ 1) lands within n 2^-52 of the sequential partial sum, so unless
  // some partial sum comes that close to u the two orders cross u at the same index; if one does (probability ~ 1e-9 per draw)
  // thread 0 walks the reference's chain.
  if (tid == 0) { s_dd[9] = gen.canonical(); s_i[0] = n - 1; s_i[1] = 0; }
  __syncthreads();
  const double u = s_dd[9];
  {
    const double band = (double)n * 4.5e-16;
    const int m = n - 1, chunk = (m + K2S_T - 1) / K2S_T, lo = min(tid * chunk, m), hi = min(lo + chunk, m);
    double part = 0.0;
    for (int i = lo; i < hi; ++i) part += wd[i];
    double incl = part;
    for (int o = 1; o < 32; o <<= 1) { const double t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) s_dd[wp] = incl;
    __syncthreads();
    double acc = incl - part;
    for (int k = 0; k < wp; ++k) acc += s_dd[k];
    int found = 0x7fffffff;
    bool amb = false;
    for (int i = lo; i < hi; ++i) {
      acc += wd[i];
      amb |= fabs(acc - u) <= band;
      if (found == 0x7fffffff && !(acc < u)) found = i;
    }
    if (found != 0x7fffffff) atomicMin(&s_i[0], found);
    if (amb) s_i[1] = 1;
    __syncthreads();
    if (s_i[1]) {                                                          // (uniform: shared flag)
      if (tid == 0) {
        double a2 = 0.0;
        int pick = n - 1;
        for (int i = 0; i < n - 1; ++i) {
          a2 += wd[i];
          if (!(a2 < u)) { pick = i; break; }
        }
        s_i[0] = pick;
      }
      __syncthreads();
    }
  }
  const int pick = s_i[0];
  __syncthreads();
  return pick;
}

// The draw of k2s_select_bases<SHARED> from the weights w[0..n), normalised first when `normalise` is set; every thread returns
// the index.  SHARED: w and its double copy wd in shared memory, the block-cooperative block_discrete_draw.  Otherwise w is in
// global memory and thread 0 does it all in the reference's order (sequential float sum, division, discrete_draw), broadcast
// through s_i[0].
template <bool SHARED>
__device__ __forceinline__ int stocs_draw(float* w, double* wd, int n, MinStd& gen, bool normalise, int tid, float* s_f, double* s_dd, int* s_i) {
  if (SHARED) return block_discrete_draw(w, wd, n, gen, normalise, tid, s_f, s_dd, s_i);
  if (tid == 0) {
    if (normalise) {
      float sum = 0.f;
      for (int i = 0; i < n; ++i) sum = __fadd_rn(sum, w[i]);
      for (int i = 0; i < n; ++i) w[i] = __fdiv_rn(w[i], sum);
    }
    s_i[0] = discrete_draw(w, n, gen);
  }
  __syncthreads();
  return s_i[0];
}

// One CTA per base: Match4PCSBase::SelectQuadrilateralStoCS (match4pcsBase.cc:600-792).  Each of the four points is drawn from
// prior x "the PPF of the edge to the previous point exists in the model's map" (x the coplanarity / spread filters for the
// 4th / 3rd point); the weights are evaluated by all threads, and the float normalisation and the draw reproduce the reference's
// sequential arithmetic bit for bit (stocs_draw), so that a given engine seed reproduces the reference's draw.
//   SHARED = true:  the weights (n floats + n doubles) in dynamic shared memory, K2S_T threads, block-cooperative draw;
//   SHARED = false: for scenes whose weights do not fit shared memory, one slice of sp.curr per base, 256 threads, the draw on
//                   thread 0.
template <bool SHARED>
__global__ void __launch_bounds__(SHARED ? K2S_T : 256, SHARED ? 8 : 0) k2s_select_bases(StocsParams sp, BaseOut* __restrict__ out) {
  constexpr int NT = SHARED ? K2S_T : 256;
  extern __shared__ __align__(16) unsigned char k2s_smem[];
  __shared__ int s_any;
  __shared__ int s_i[SHARED ? 32 : 2];
  __shared__ float s_f[SHARED ? 12 : 1];
  __shared__ double s_dd[SHARED ? 12 : 1];
  const int base = blockIdx.x, tid = threadIdx.x, n = sp.n;
  double* wd = reinterpret_cast<double*>(k2s_smem);
  float* curr = SHARED ? reinterpret_cast<float*>(wd + n) : sp.curr + (size_t)base * n;
  const float4* P = sp.P;
  BaseOut o{};
  for (int attempt = 0; attempt < 16; ++attempt) {      // Perform_N_steps re-draws until a base is accepted (:1831-1852)
    MinStd gen(stocs_base_seed(sp.seed, sp.base0 + base, attempt));
    // ---- point 1 ~ priors
    for (int i = tid; i < n; i += NT) curr[i] = sp.aux[i].w;
    __syncthreads();
    const int b1 = stocs_draw<SHARED>(curr, wd, n, gen, false, tid, s_f, s_dd, s_i);
    const float4 p1 = P[b1], a1 = sp.aux[b1];
    // ---- point 2: prior_i * prior_b1 * edge(b1, i)
    if (tid == 0) s_any = 0;
    __syncthreads();
    for (int i = tid; i < n; i += NT) {
      float w = 0.f;
      const float c = curr[i];
      if (i != b1 && c != 0.f) {
        const float4 ai = sp.aux[i];
        const float e = ppf_present(sp.bits, ppf_key(p1, a1, P[i], ai)) ? 1.f : 0.f;
        w = __fmul_rn(__fmul_rn(ai.w, a1.w), e);
      }
      curr[i] = w;
      if (w != 0.f) s_any = 1;
    }
    __syncthreads();
    if (!s_any) { __syncthreads(); continue; }
    const int b2 = stocs_draw<SHARED>(curr, wd, n, gen, true, tid, s_f, s_dd, s_i);
    const float4 p2 = P[b2], a2 = sp.aux[b2];
    // ---- point 3: curr_i * prior_b2 * edge(b2, i), minus the points whose (un-normalised!) angle test fails (:670-676)
    if (tid == 0) s_any = 0;
    __syncthreads();
    const float v1x = __fsub_rn(p2.x, p1.x), v1y = __fsub_rn(p2.y, p1.y), v1z = __fsub_rn(p2.z, p1.z);
    for (int i = tid; i < n; i += NT) {
      float w = 0.f;
      const float c = curr[i];
      const float4 pi = P[i];
      const float d = dot3_tree(v1x, v1y, v1z, __fsub_rn(pi.x, p1.x), __fsub_rn(pi.y, p1.y), __fsub_rn(pi.z, p1.z));
      // |d| < 0.8: acos(d) lies in (36.8, 143.2) degrees, min(a, 180 - a) > 30 whatever the rounding -- the case for metre-scale
      // vectors, whose un-normalised dot product is tiny; anything else takes the reference's arithmetic
      bool far30 = fabsf(d) < 0.8f;
      if (!far30) {
        float ang = (float)((double)__fmul_rn((float)acos((double)d), 180.0f) / 3.14159265358979323846);
        const float other = __fsub_rn(180.0f, ang);
        ang = other < ang ? other : ang;               // std::min(a, b) = (b < a) ? b : a   (NaN stays NaN -> not rejected)
        far30 = !(ang < 30.0f);
      }
      if (i != b1 && i != b2 && c != 0.f && far30) {
        const float4 ai = sp.aux[i];
        const float e = ppf_present(sp.bits, ppf_key(p2, a2, pi, ai)) ? 1.f : 0.f;
        w = __fmul_rn(__fmul_rn(c, a2.w), e);
      }
      curr[i] = w;
      if (w != 0.f) s_any = 1;
    }
    __syncthreads();
    if (!s_any) { __syncthreads(); continue; }
    const int b3 = stocs_draw<SHARED>(curr, wd, n, gen, true, tid, s_f, s_dd, s_i);
    const float4 p3 = P[b3], a3 = sp.aux[b3];
    // ---- point 4: near the plane of the three (<= 1 cm), >= 1 cm away from each of them, edge(b3, i)  (:717-763)
    if (tid == 0) s_any = 0;
    __syncthreads();
    const double x1 = p1.x, y1 = p1.y, z1 = p1.z, x2 = p2.x, y2 = p2.y, z2 = p2.z, x3 = p3.x, y3 = p3.y, z3 = p3.z;
    const float denom = (float)(-x3 * y2 * z1 + x2 * y3 * z1 + x3 * y1 * z2 - x1 * y3 * z2 - x2 * y1 * z3 + x1 * y2 * z3);
    float A = 0.f, B = 0.f, C = 0.f;
    if (denom != 0.f) {
      A = (float)((-y2 * z1 + y3 * z1 + y1 * z2 - y3 * z2 - y1 * z3 + y2 * z3) / (double)denom);
      B = (float)((x2 * z1 - x3 * z1 - x1 * z2 + x3 * z2 + x1 * z3 - x2 * z3) / (double)denom);
      C = (float)((-x2 * y1 + x3 * y1 + x1 * y2 - x3 * y2 - x1 * y3 + x2 * y3) / (double)denom);
    }
    for (int i = tid; i < n; i += NT) {
      float w = 0.f;
      const float c = curr[i];
      if (i != b1 && i != b2 && i != b3 && c != 0.f) {
        const float4 pi = P[i];
        bool keep = true;
        if (denom != 0.f) {
          const float lin = __fadd_rn(__fadd_rn(__fmul_rn(A, pi.x), __fmul_rn(B, pi.y)), __fmul_rn(C, pi.z));
          const float pd = fabsf(__fsub_rn(lin, 1.0f));        // (float) fabs((double) lin - 1.0): the double difference is exact, its rounding is this
          auto nrm = [&](const float4 q) {
            const float dx = __fsub_rn(pi.x, q.x), dy = __fsub_rn(pi.y, q.y), dz = __fsub_rn(pi.z, q.z);
            return __fsqrt_rn(dot3_tree(dx, dy, dz, dx, dy, dz));
          };
          // float against the double 0.01 (fl32(0.01) = 0.0099999998 < 0.01): x > 0.01 <=> x > 0.01f,  x < 0.01 <=> x <= 0.01f
          if (pd > 0.01f || nrm(p1) <= 0.01f || nrm(p2) <= 0.01f || nrm(p3) <= 0.01f) keep = false;
        }
        if (keep) {
          const float4 ai = sp.aux[i];
          const float e = ppf_present(sp.bits, ppf_key(p3, a3, pi, ai)) ? 1.f : 0.f;
          w = __fmul_rn(__fmul_rn(c, a3.w), e);
        }
      }
      curr[i] = w;
      if (w != 0.f) s_any = 1;
    }
    __syncthreads();
    if (!s_any) { __syncthreads(); continue; }
    const int b4 = stocs_draw<SHARED>(curr, wd, n, gen, true, tid, s_f, s_dd, s_i);
    if (tid == 0) {
      const int ids[4] = {b1, b2, b3, b4};
      try_quadrilateral(P, ids, o);
      s_i[1] = o.ok;
    }
    __syncthreads();
    const int okk = s_i[1];
    __syncthreads();
    if (okk) break;
  }
  if (tid == 0) out[base] = o;
}

// pair lists of the chunk's combos straight from the PPF map (ExtractCongruentSet in operMode 1, :1970-1981):
// combo 2b = map[ppf(b0, b1)], combo 2b+1 = map[ppf(b2, b3)]
struct PpfMapDev { const uint32_t* keys; const uint32_t* offsets; const int2* pairs; int n_keys; };
__device__ __forceinline__ int ppf_find(const PpfMapDev& m, uint32_t key) {
  if (key == PPF_NOKEY) return -1;
  int lo = 0, hi = m.n_keys;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(m.keys + mid) < key) lo = mid + 1; else hi = mid; }
  return (lo < m.n_keys && m.keys[lo] == key) ? lo : -1;
}
__global__ void k2s_combo_counts(PpfMapDev m, const float4* __restrict__ P, const float4* __restrict__ aux, const BaseOut* __restrict__ bases, int ncombo,
                                 uint32_t* __restrict__ cnt, int* __restrict__ slot) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncombo) return;
  const BaseOut& bo = bases[c >> 1];
  int k = -1;
  if (bo.ok) {
    const int i = bo.id[(c & 1) * 2], j = bo.id[(c & 1) * 2 + 1];
    k = ppf_find(m, ppf_key(P[i], aux[i], P[j], aux[j]));
  }
  slot[c] = k;
  cnt[c] = k >= 0 ? m.offsets[k + 1] - m.offsets[k] : 0u;
}
// a base needs both of its lists (pairs1.size() == 0 || pairs6.size() == 0 -> no quads, :1984-1986): the join finds nothing otherwise
__global__ void k2s_combo_copy(PpfMapDev m, const int* __restrict__ slot, const uint32_t* __restrict__ coff, int2* __restrict__ out) {
  const int c = blockIdx.y;
  const int k = slot[c];
  if (k < 0) return;
  const uint32_t n = m.offsets[k + 1] - m.offsets[k];
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) out[coff[c] + t] = m.pairs[m.offsets[k] + t];
}

struct Scratch {
  DevBuf adj, dist6, in_order, list1, list2, cnt, cnt2, off, flag, curr, pairs1, pairs2, quads, bucket_of, key_of, bucket_start, sorted, T, ok, base, qn;
  DevBuf cone_tab;                              // per base of the chunk: the cone's sample directions (k2_cone_table)
  DevBuf cone, stage_n, stage_r, stage_T;       // fused fill: cone masks of the pairs that found quads; per-base staging of the selected quads
  const Model* bases_owner = nullptr;   // the model whose last k2_generate call left its bases in `base` (k2_get_bases)
};
// the generator's device scratch belongs to the context (two contexts on one device must not share it); created on first use,
// released by k2_release (pgp_destroy)
Scratch& scratch_of(pgp_ctx* ctx) {
  if (!ctx->k2_scratch) ctx->k2_scratch = new Scratch();
  return *static_cast<Scratch*>(ctx->k2_scratch);
}

int scan_u32(pgp_ctx* ctx, uint32_t* data, int64_t n, uint64_t* total) {
  PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((n + 1) / 2048 + 4096) * 4));
  int rc = pgp_scan_exclusive_u32(ctx, data, n + 1, ctx->scene.scratch.as<uint32_t>());
  if (rc) return rc;
  uint32_t t = 0;
  PGP_CUDA(ctx, cudaMemcpyAsync(&t, data + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *total = t;
  return PGP_OK;
}

// all ordered pairs into `out` (device, grown as needed); returns the number of ORDERED pairs
int extract_pairs_dev(pgp_ctx* ctx, const Model& m, float dist, float eps, DevBuf& out, int64_t* n_pairs) {
  Scratch& sc = scratch_of(ctx);
  const int nq = m.nq, B = (nq + 255) / 256;
  PGP_CUDA(ctx, sc.cnt.reserve((size_t)(nq + 1) * 4));
  uint32_t* cnt = sc.cnt.as<uint32_t>();
  PGP_CUDA(ctx, cudaMemsetAsync(cnt, 0, (size_t)(nq + 1) * 4, ctx->stream));
  k2_pairs<false><<<B, 256, 0, ctx->stream>>>(m.search.as<float4>(), nq, dist, eps, cnt, nullptr, 0);
  ctx->launches++;
  uint64_t total = 0;
  int rc = scan_u32(ctx, cnt, nq, &total);
  if (rc) return rc;
  *n_pairs = (int64_t)total * 2;
  PGP_CUDA(ctx, out.reserve((size_t)std::max<int64_t>(*n_pairs, 1) * 8));
  if (total) {
    k2_pairs<true><<<B, 256, 0, ctx->stream>>>(m.search.as<float4>(), nq, dist, eps, cnt, out.as<int2>(), *n_pairs);
    ctx->launches++;
  }
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

int find_quads_dev(pgp_ctx* ctx, const Model& m, float cos_alpha, float inv1, float inv2, float eps, const int2* A, int64_t n1, const int2* B,
                   int64_t n2, DevBuf& out, int64_t* n_quads) {
  Scratch& sc = scratch_of(ctx);
  *n_quads = 0;
  if (n1 <= 0 || n2 <= 0) return PGP_OK;
  JoinParams p{};
  p.Qn = m.search_unit.as<float4>(); p.Q = m.search.as<float4>();
  p.A = A; p.n1 = n1; p.B = B; p.n2 = n2;
  p.inv1 = inv1; p.inv2 = inv2; p.cos_alpha = cos_alpha; p.thr2 = eps;
  // IndexedNormalSet(eps_n): gridDepth = int(-log2(eps_n)); egSize = 2^gridDepth; _epsilon = 1/egSize  (normalset.h:117-123)
  const float eps_n = eps / m.unit_ratio;
  int depth = (int)(-std::log2(eps_n));
  if (depth < 0) depth = 0;
  if (depth > 7) return pgp_fail(ctx, PGP_E_TOO_LARGE, "quad join: model diameter / delta too large (grid depth %d > 7)", depth);
  p.eg = 1 << depth;
  p.cell = 1.0f / (float)p.eg;
  p.n_buckets = 1u << std::min(3 * depth, 20);
  PGP_CUDA(ctx, sc.bucket_of.reserve((size_t)n1 * 4));
  PGP_CUDA(ctx, sc.key_of.reserve((size_t)n1 * 4));
  PGP_CUDA(ctx, sc.sorted.reserve((size_t)n1 * 4));
  PGP_CUDA(ctx, sc.bucket_start.reserve(((size_t)p.n_buckets + 1) * 8));
  uint32_t* bs = sc.bucket_start.as<uint32_t>();
  uint32_t* cursor = bs + p.n_buckets + 1;
  PGP_CUDA(ctx, cudaMemsetAsync(bs, 0, ((size_t)p.n_buckets + 1) * 4, ctx->stream));
  k2_join_keys<<<(unsigned)((n1 + 255) / 256), 256, 0, ctx->stream>>>(p, sc.bucket_of.as<uint32_t>(), sc.key_of.as<uint32_t>(), bs);
  ctx->launches++;
  uint64_t tot = 0;
  int rc = scan_u32(ctx, bs, p.n_buckets, &tot);
  if (rc) return rc;
  PGP_CUDA(ctx, cudaMemcpyAsync(cursor, bs, (size_t)p.n_buckets * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  k2_join_scatter<<<(unsigned)((n1 + 255) / 256), 256, 0, ctx->stream>>>(n1, sc.bucket_of.as<uint32_t>(), cursor, sc.sorted.as<uint32_t>());
  PGP_CUDA(ctx, sc.in_order.reserve((size_t)p.n_buckets + 16));
  k2_join_sort_buckets<<<(unsigned)((p.n_buckets + 255) / 256), 256, 0, ctx->stream>>>(p.A, bs, (long long)p.n_buckets, sc.sorted.as<uint32_t>(), sc.in_order.as<unsigned char>());
  ctx->launches += 2;
  PGP_CUDA(ctx, sc.cnt.reserve((size_t)(n2 + 1) * 4));
  uint32_t* cnt = sc.cnt.as<uint32_t>();
  PGP_CUDA(ctx, cudaMemsetAsync(cnt, 0, (size_t)(n2 + 1) * 4, ctx->stream));
  k2_join_query<false><<<(unsigned)((n2 + 127) / 128), 128, 0, ctx->stream>>>(p, bs, sc.sorted.as<uint32_t>(), sc.key_of.as<uint32_t>(), cnt, nullptr, 0, sc.in_order.as<unsigned char>());
  ctx->launches++;
  uint64_t nquads = 0;
  rc = scan_u32(ctx, cnt, n2, &nquads);
  if (rc) return rc;
  *n_quads = (int64_t)nquads;
  PGP_CUDA(ctx, out.reserve((size_t)std::max<uint64_t>(nquads, 1) * 16));
  if (nquads) {
    k2_join_query<true><<<(unsigned)((n2 + 127) / 128), 128, 0, ctx->stream>>>(p, bs, sc.sorted.as<uint32_t>(), sc.key_of.as<uint32_t>(), cnt, out.as<int4>(),
                                                                              (long long)nquads, sc.in_order.as<unsigned char>());
    ctx->launches++;
  }
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

}  // namespace

// host-callable copy of chain_sum_equal for the CPU test-suite (tests/test_host_arithmetic.py): the closed form must equal the
// brute-force float chain for every (c, m)
extern "C" PGP_API float pgp_host_chain_sum_equal(float c, long long m) { return chain_sum_equal(c, m); }


int k2_extract_pairs(pgp_ctx* ctx, const Model& m, float dist, float eps, int32_t* pairs_host, int64_t cap, int64_t* n_pairs) {
  Scratch& sc = scratch_of(ctx);
  int rc = extract_pairs_dev(ctx, m, dist, eps, sc.pairs1, n_pairs);
  if (rc) return rc;
  const int64_t n = std::min(cap, *n_pairs);
  if (pairs_host && n > 0) {
    PGP_CUDA(ctx, cudaMemcpyAsync(pairs_host, sc.pairs1.p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return PGP_OK;
}

int k2_find_quads(pgp_ctx* ctx, const Model& m, const int32_t* base4, float inv1, float inv2, float eps, const int32_t* p1, int64_t n1,
                  const int32_t* p2, int64_t n2, int32_t* quads_host, int64_t cap, int64_t* n_quads) {
  Scratch& sc = scratch_of(ctx);
  const Scene& s = ctx->scene;
  for (int k = 0; k < 4; ++k)
    if (base4[k] < 0 || base4[k] >= s.n) return pgp_fail(ctx, PGP_E_INVALID, "base id out of range");
  // angle between the base's two edges (super4pcs.cc:109-111) from the centred scene points
  float4 bp[4];
  for (int k = 0; k < 4; ++k) PGP_CUDA(ctx, cudaMemcpyAsync(&bp[k], s.unsorted.as<float4>() + base4[k], 16, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  auto unit = [](float4 a, float4 b, float o[3]) {
    o[0] = b.x - a.x; o[1] = b.y - a.y; o[2] = b.z - a.z;
    volatile float s2 = o[0] * o[0]; s2 = s2 + o[1] * o[1]; s2 = s2 + o[2] * o[2];
    float l = sqrtf(s2);
    o[0] /= l; o[1] /= l; o[2] /= l;
  };
  float u[3], v[3];
  unit(bp[0], bp[1], u); unit(bp[2], bp[3], v);
  volatile float ca = u[0] * v[0]; ca = ca + u[1] * v[1]; ca = ca + u[2] * v[2];
  *n_quads = 0;
  if (n1 <= 0 || n2 <= 0) return PGP_OK;
  PGP_CUDA(ctx, sc.pairs1.reserve((size_t)n1 * 8));
  PGP_CUDA(ctx, sc.pairs2.reserve((size_t)n2 * 8));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.pairs1.p, p1, (size_t)n1 * 8, cudaMemcpyHostToDevice, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.pairs2.p, p2, (size_t)n2 * 8, cudaMemcpyHostToDevice, ctx->stream));
  int rc = find_quads_dev(ctx, m, ca, inv1, inv2, eps, sc.pairs1.as<int2>(), n1, sc.pairs2.as<int2>(), n2, sc.quads, n_quads);
  if (rc) return rc;
  const int64_t n = std::min(cap, *n_quads);
  if (quads_host && n > 0) {
    PGP_CUDA(ctx, cudaMemcpyAsync(quads_host, sc.quads.p, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return PGP_OK;
}

int k2_rigid_from_quads(pgp_ctx* ctx, const Model& m, const int32_t* base4, const int32_t* quads_host, int64_t n, float* T_host, uint8_t* ok_host) {
  Scratch& sc = scratch_of(ctx);
  if (n == 0) return PGP_OK;
  for (int k = 0; k < 4; ++k)
    if (base4[k] < 0 || base4[k] >= ctx->scene.n) return pgp_fail(ctx, PGP_E_INVALID, "base id out of range");
  PGP_CUDA(ctx, sc.quads.reserve((size_t)n * 16));
  PGP_CUDA(ctx, sc.T.reserve((size_t)n * 48));
  PGP_CUDA(ctx, sc.ok.reserve((size_t)n));
  PGP_CUDA(ctx, sc.base.reserve(64));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.quads.p, quads_host, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.base.p, base4, 16, cudaMemcpyHostToDevice, ctx->stream));
  k2_rigid<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->scene.unsorted.as<float4>(), m.search.as<float4>(), sc.base.as<int>(), sc.quads.as<int4>(),
                                                                n, sc.T.as<float>(), sc.ok.as<uint8_t>());
  ctx->launches++;
  PGP_CUDA(ctx, cudaMemcpyAsync(T_host, sc.T.p, (size_t)n * 48, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(ok_host, sc.ok.p, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

// ------------------------------------------------------------------------------- batched driver
// All bases of a chunk go through every stage in ONE launch (pairs, join, transforms, subset,
// compaction); the host only reads three totals per chunk to size the next buffer.
namespace {

// quads of base b = [qoff[b], qoff[b+1]): the quads found by the B-side pairs of combo 2b+1
__global__ void k2b_quad_offsets(const uint32_t* __restrict__ qscan, const uint32_t* __restrict__ coff, int nb, uint32_t* __restrict__ qoff) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nb) qoff[b] = qscan[coff[2 * b + 1]];
  if (b == nb) qoff[nb] = qscan[coff[2 * nb]];
}

// transform of every quad + the keep flag of the per-base random subset (Perform_N_steps draws max_sampled_csets
// distinct quads per base, match4pcsBase.cc:1858-1869: here the ones with the smallest counter-based hash, oversampled
// by 25 % and cut at exactly max_quads by the scan positions below)
__global__ void k2b_rigid(const float4* __restrict__ P_unsorted, const float4* __restrict__ Q, const BaseOut* __restrict__ bases, int base0,
                          const uint32_t* __restrict__ qoff, int nb, const int4* __restrict__ quads, long long n, int max_quads, uint64_t seed,
                          float* __restrict__ T, uint32_t* __restrict__ flag) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int b = segment_of(qoff, nb, (uint32_t)i);
  float t[12];
  bool good = rigid_from_quad(P_unsorted, Q, bases[b].id, quads[i], t);
#pragma unroll
  for (int c = 0; c < 12; ++c) T[12 * i + c] = good ? t[c] : 0.f;
  const long long nq_b = (long long)qoff[b + 1] - (long long)qoff[b];
  if (good && max_quads > 0 && nq_b > max_quads) {
    const double frac = fmin(1.0, 1.25 * (double)max_quads / (double)nq_b);
    const unsigned long long thr = (unsigned long long)(frac * 9007199254740992.0);   // 2^53
    const uint64_t sb = mix64(seed ^ (0xABCDull + (uint64_t)(base0 + b)));
    const int4 qd = quads[i];
    good = quad_selected(sb, qd.x, qd.y, qd.z, qd.w, thr);
  }
  flag[i] = good ? 1u : 0u;
}

// ------------------------------------------------------------------------------- operMode 2: V4PCS (tetrahedron base, six-distance join)
// ExtractCongruentSet in operMode 2 (match4pcsBase.cc:1929-2039) runs ExtractPairs for the six edge lengths d1 = |b1 b2|,
// d2 = |b1 b3|, d3 = |b1 b4|, d4 = |b2 b3|, d5 = |b2 b4|, d6 = |b3 b4| of the base and FindCongruentQuadrilateralsV4PCS
// (:978-1044) joins them through (vertex, distance) connectivity maps: the result is every ordered 4-tuple (v1, v2, v3, v4) of
// model points with (v1,v2) in pairs1, (v1,v3) in pairs2, (v3,v2) in pairs4, (v1,v4) in pairs3, (v4,v2) in pairs5, (v4,v3) in
// pairs6.  On the device the six pair sets are bit matrices (row i, bit j: the pair filter of pairCreationFunctor.h:167-253 --
// float norm, |norm - d| <= eps compared in double, no self pairs; the filter is symmetric, so column v of a matrix is its row v),
// and the join is row ANDs + popcounts, one warp per (base, v1).  Quads come out sorted by (v1, v2, v3, v4); the reference's own
// order is an unordered_set iteration, so parity is on the set.

// widest random triangle as operMode 0 (SelectRandomTriangle :377-410), then the most voluminous of 100 random fourth points
// (SelectTetrahedronBase :466-503).  Counter-based RNG like k2_select_bases (the reference draws from rand()).
__global__ void __launch_bounds__(256) k2v_select_bases(const float4* __restrict__ P, int n, float max_diam, int trials, uint64_t seed, int base_lo, BaseOut* __restrict__ out) {
  __shared__ float s_val[256];
  __shared__ int s_idx[256];
  const int base = base_lo + blockIdx.x, tid = threadIdx.x;
  BaseOut o{};
  for (int attempt = 0; attempt < 16 && !o.ok; ++attempt) {
    const uint64_t s0 = mix64(seed ^ mix64(0x7E7A00000000ull | ((uint64_t)base << 8) | (uint64_t)attempt));
    const int first = (int)(mix64(s0) % (uint64_t)n);
    const float4 p0 = P[first];
    const float sqmax = max_diam * max_diam;
    float best = 0.f; int best_t = 0x7fffffff;
    for (int t = tid; t < trials; t += 256) {
      const uint64_t r = mix64(s0 + 2 * (uint64_t)t + 1), r2 = mix64(s0 + 2 * (uint64_t)t + 2);
      const float4 a = P[(int)(r % (uint64_t)n)], b = P[(int)(r2 % (uint64_t)n)];
      const V3 u = {a.x - p0.x, a.y - p0.y, a.z - p0.z}, w = {b.x - p0.x, b.y - p0.y, b.z - p0.z};
      const V3 cr = cross(u, w);
      const float wide = sqrtf(dot(cr, cr));
      if (wide > best && dot(u, u) < sqmax && dot(w, w) < sqmax) { best = wide; best_t = t; }
    }
    s_val[tid] = best; s_idx[tid] = best_t;
    __syncthreads();
    for (int o2 = 128; o2 > 0; o2 >>= 1) {
      if (tid < o2) {
        const float v = s_val[tid + o2]; const int ix = s_idx[tid + o2];
        if (v > s_val[tid] || (v == s_val[tid] && ix < s_idx[tid])) { s_val[tid] = v; s_idx[tid] = ix; }
      }
      __syncthreads();
    }
    const int bt = s_idx[0];
    const bool have_tri = s_val[0] > 0.f && bt != 0x7fffffff;
    __syncthreads();
    if (!have_tri) continue;
    const int i1 = first, i2 = (int)(mix64(s0 + 2 * (uint64_t)bt + 1) % (uint64_t)n), i3 = (int)(mix64(s0 + 2 * (uint64_t)bt + 2) % (uint64_t)n);
    const float4 p1 = P[i1], p2 = P[i2], p3 = P[i3];
    const V3 v1 = {p2.x - p1.x, p2.y - p1.y, p2.z - p1.z}, v2 = {p3.x - p1.x, p3.y - p1.y, p3.z - p1.z};
    const V3 nrm = cross(v1, v2);
    float vol = 0.f; int vt = 0x7fffffff, vi = -1;
    if (tid < 100) {                                    // 100 random fourth points, first maximum in trial order wins (strict '>')
      vi = (int)(mix64(s0 ^ (0x4444000000000000ull + (uint64_t)tid)) % (uint64_t)n);
      const float4 q = P[vi];
      const V3 v3 = {q.x - p1.x, q.y - p1.y, q.z - p1.z};
      vol = fabsf(dot(nrm, v3)) / 6.0f;
      vt = tid;
    }
    s_val[tid] = vol; s_idx[tid] = vt;
    __syncthreads();
    for (int o2 = 128; o2 > 0; o2 >>= 1) {
      if (tid < o2) {
        const float v = s_val[tid + o2]; const int ix = s_idx[tid + o2];
        if (v > s_val[tid] || (v == s_val[tid] && ix < s_idx[tid])) { s_val[tid] = v; s_idx[tid] = ix; }
      }
      __syncthreads();
    }
    const int wt = s_idx[0];
    const bool have4 = s_val[0] > 0.f && wt < 100;
    __syncthreads();
    if (!have4) continue;
    const int i4 = (int)(mix64(s0 ^ (0x4444000000000000ull + (uint64_t)wt)) % (uint64_t)n);
    o.id[0] = i1; o.id[1] = i2; o.id[2] = i3; o.id[3] = i4; o.ok = 1;
  }
  if (tid == 0) out[blockIdx.x] = o;
}

// the six edge lengths of every base: (a - b).norm() as Eigen evaluates it for a Vector3f, sqrt((x^2 + y^2) + z^2)
__global__ void k2v_base_dists(const float4* __restrict__ P, const BaseOut* __restrict__ bases, int nb, float* __restrict__ dist6) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nb * 6) return;
  const int b = t / 6, k = t % 6;
  const int ia = k < 3 ? 0 : k < 5 ? 1 : 2, ib = k == 0 ? 1 : k == 1 ? 2 : k == 2 ? 3 : k == 3 ? 2 : 3;    // (0,1) (0,2) (0,3) (1,2) (1,3) (2,3)
  const float4 a = P[bases[b].id[ia]], c = P[bases[b].id[ib]];
  const float x = __fsub_rn(a.x, c.x), y = __fsub_rn(a.y, c.y), z = __fsub_rn(a.z, c.z);
  dist6[t] = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)));
}

// bit matrices A[((b * 6 + k) * nq + i) * W + w]: bit (j & 31) of word j >> 5 = pair (i, j) passes the filter for distance k of base b
__global__ void __launch_bounds__(256) k2v_adjacency(const float4* __restrict__ Q, int nq, int W, const BaseOut* __restrict__ bases,
                                                     const float* __restrict__ dist6, float eps, uint32_t* __restrict__ A) {
  const int b = blockIdx.y;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)nq * W) return;
  const int i = (int)(idx % nq), w = (int)(idx / nq);           // consecutive lanes: consecutive i, the same 32 columns
  uint32_t bits[6] = {0, 0, 0, 0, 0, 0};
  if (bases[b].ok) {
    double d[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) d[k] = (double)dist6[b * 6 + k];
    const double e = (double)eps;
    const float4 qi = Q[i];
    const int j0 = w * 32, j1 = min(nq, j0 + 32);
    for (int j = j0; j < j1; ++j) {
      if (j == i) continue;
      const float4 p = Q[j];
      const float dx = __fsub_rn(qi.x, p.x), dy = __fsub_rn(qi.y, p.y), dz = __fsub_rn(qi.z, p.z);
      const double dd = (double)__fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz))));
#pragma unroll
      for (int k = 0; k < 6; ++k) if (!(fabs(dd - d[k]) > e)) bits[k] |= 1u << (j - j0);
    }
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) A[(((size_t)b * 6 + k) * nq + i) * W + w] = bits[k];
}

// one warp per (base, v1): count (FILL = false) or write (FILL = true, at the scanned offset) the quads that start with v1
template <bool FILL>
__global__ void __launch_bounds__(256) k2v_join(int nq, int W, int nb, const BaseOut* __restrict__ bases, const uint32_t* __restrict__ A,
                                                uint32_t* __restrict__ cnt, int4* __restrict__ out, long long cap) {
  const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= (long long)nb * nq) return;
  const int b = (int)(gw / nq), v1 = (int)(gw % nq);
  if (!bases[b].ok) { if (!FILL && lane == 0) cnt[gw] = 0; return; }
  if (FILL && cnt[gw + 1] == cnt[gw]) return;
  const size_t mat = (size_t)nq * W;
  const uint32_t* A1 = A + ((size_t)b * 6 + 0) * mat + (size_t)v1 * W;
  const uint32_t* A2 = A + ((size_t)b * 6 + 1) * mat + (size_t)v1 * W;
  const uint32_t* A3 = A + ((size_t)b * 6 + 2) * mat + (size_t)v1 * W;
  const uint32_t* M4 = A + ((size_t)b * 6 + 3) * mat;
  const uint32_t* M5 = A + ((size_t)b * 6 + 4) * mat;
  const uint32_t* M6 = A + ((size_t)b * 6 + 5) * mat;
  uint32_t n = 0;
  long long wpos = FILL ? (long long)cnt[gw] : 0;
  for (int w1 = 0; w1 < W; ++w1) {
    uint32_t word1 = A1[w1];                                   // uniform
    while (word1) {
      const int v2 = 32 * w1 + __ffs(word1) - 1;
      word1 &= word1 - 1;
      const uint32_t* A4 = M4 + (size_t)v2 * W;                // (v3, v2) in pairs4  <=>  bit v3 of row v2 (symmetric filter)
      const uint32_t* A5 = M5 + (size_t)v2 * W;
      for (int c3 = 0; c3 < W; c3 += 32) {
        const int l3 = c3 + lane;
        const uint32_t m3 = l3 < W ? (A2[l3] & A4[l3]) : 0u;
        unsigned nz = __ballot_sync(0xffffffffu, m3 != 0u);
        while (nz) {
          const int src = __ffs(nz) - 1;
          nz &= nz - 1;
          uint32_t bits3 = __shfl_sync(0xffffffffu, m3, src);
          while (bits3) {
            const int v3 = 32 * (c3 + src) + __ffs(bits3) - 1;
            bits3 &= bits3 - 1;
            const uint32_t* A6 = M6 + (size_t)v3 * W;          // (v4, v3) in pairs6
            for (int c4 = 0; c4 < W; c4 += 32) {
              const int l4 = c4 + lane;
              const uint32_t m4 = l4 < W ? (A3[l4] & A5[l4] & A6[l4]) : 0u;
              const uint32_t c = (uint32_t)__popc(m4);
              if (!FILL) {
                n += c;
              } else {
                uint32_t incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
                long long w = wpos + (long long)(incl - c);
                uint32_t mm = m4;
                while (mm) {
                  const int v4 = 32 * l4 + __ffs(mm) - 1;
                  mm &= mm - 1;
                  if (w < cap) out[w] = make_int4(v1, v2, v3, v4);
                  ++w;
                }
                wpos += (long long)__shfl_sync(0xffffffffu, incl, 31);
              }
            }
          }
        }
      }
    }
  }
  if (!FILL) {
    n = __reduce_add_sync(0xffffffffu, n);
    if (lane == 0) cnt[gw] = n;
  }
}

__global__ void k2v_quad_offsets(const uint32_t* __restrict__ scan, int nq, int nb, uint32_t* __restrict__ qoff) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b <= nb) qoff[b] = scan[(size_t)b * nq];
}

// per-base kept counts (capped when max_quads > 0) -> exclusive scan
__global__ void __launch_bounds__(1024) k2b_base_out(const uint32_t* __restrict__ fscan, const uint32_t* __restrict__ qoff, int nb, int max_quads, uint32_t* __restrict__ outoff) {
  capped_base_scan(nb, [&](int b) {
    const uint32_t k = fscan[qoff[b + 1]] - fscan[qoff[b]];
    return max_quads > 0 && k > (uint32_t)max_quads ? (uint32_t)max_quads : k;
  }, outoff);
}

__global__ void k2b_append(const float* __restrict__ T, const uint32_t* __restrict__ fscan, const uint32_t* __restrict__ qoff, int nb, int max_quads,
                           const uint32_t* __restrict__ outoff, long long n, float* __restrict__ dst, long long room) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || fscan[i + 1] == fscan[i]) return;
  const int b = segment_of(qoff, nb, (uint32_t)i);
  const uint32_t pos = fscan[i] - fscan[qoff[b]];
  if (max_quads > 0 && pos >= (uint32_t)max_quads) return;
  const long long o = (long long)outoff[b] + pos;
  if (o >= room) return;
#pragma unroll
  for (int c = 0; c < 12; ++c) dst[12 * o + c] = T[12 * i + c];
}

}  // namespace

namespace {

// operMode 2, one chunk of bases (device array, `ok` set): six bit matrices per base, count, scan, fill.  Leaves the quads in
// sc.quads (sorted by base, v1, v2, v3, v4), qoff[0..nb] (device) = first quad of each base, *nquads = their number.
int v4pcs_chunk(pgp_ctx* ctx, const Model& m, const BaseOut* d_bases, int nb, float eps, uint32_t* qoff, uint64_t* nquads) {
  Scratch& sc = scratch_of(ctx);
  const Scene& s = ctx->scene;
  cudaStream_t st = ctx->stream;
  const int nq = m.nq, W = (nq + 31) / 32;
  const size_t rows = (size_t)nb * nq;
  PGP_CUDA(ctx, sc.adj.reserve(rows * 6 * W * 4 + 64));
  PGP_CUDA(ctx, sc.dist6.reserve((size_t)nb * 6 * 4 + 64));
  PGP_CUDA(ctx, sc.cnt.reserve((rows + 1) * 4));
  uint32_t* cnt = sc.cnt.as<uint32_t>();
  k2v_base_dists<<<(nb * 6 + 127) / 128, 128, 0, st>>>(s.unsorted.as<float4>(), d_bases, nb, sc.dist6.as<float>());
  k2v_adjacency<<<dim3((unsigned)(((size_t)nq * W + 255) / 256), (unsigned)nb), 256, 0, st>>>(m.search.as<float4>(), nq, W, d_bases, sc.dist6.as<float>(), eps,
                                                                                              sc.adj.as<uint32_t>());
  PGP_CUDA(ctx, cudaMemsetAsync(cnt + rows, 0, 4, st));
  const unsigned gj = (unsigned)((rows * 32 + 255) / 256);
  k2v_join<false><<<gj, 256, 0, st>>>(nq, W, nb, d_bases, sc.adj.as<uint32_t>(), cnt, nullptr, 0);
  ctx->launches += 3;
  PGP_CUDA(ctx, cudaGetLastError());
  int rc = scan_u32(ctx, cnt, (int64_t)rows, nquads);
  if (rc) return rc;
  if (*nquads == 0 || *nquads >= (1ull << 31)) return PGP_OK;
  PGP_CUDA(ctx, sc.quads.reserve((size_t)*nquads * 16));
  k2v_join<true><<<gj, 256, 0, st>>>(nq, W, nb, d_bases, sc.adj.as<uint32_t>(), cnt, sc.quads.as<int4>(), (long long)*nquads);
  k2v_quad_offsets<<<(nb + 256) / 256, 256, 0, st>>>(cnt, nq, nb, qoff);
  ctx->launches += 2;
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

// Unfused tail of a chunk of nb bases: the rigid transform of each of the nquads quads in sc.quads (base b's at
// [qoff[b], qoff[b+1])), the per-base subset, and the kept transforms appended at dst, at most `room` of them.  *added = how many.
int append_unfused(pgp_ctx* ctx, const Model& m, const pgp_pcs_opts* o, uint64_t seed, const BaseOut* d_bases, int base_global0, int nb,
                   const uint32_t* qoff, uint64_t nquads, uint32_t* outoff, float* dst, int64_t room, int64_t* added) {
  Scratch& sc = scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  PGP_CUDA(ctx, sc.T.reserve((size_t)nquads * 48));
  PGP_CUDA(ctx, sc.flag.reserve((size_t)(nquads + 1) * 4));
  uint32_t* flag = sc.flag.as<uint32_t>();
  PGP_CUDA(ctx, cudaMemsetAsync(flag + nquads, 0, 4, st));
  const unsigned gr = (unsigned)((nquads + 127) / 128);
  k2b_rigid<<<gr, 128, 0, st>>>(ctx->scene.unsorted.as<float4>(), m.search.as<float4>(), d_bases, base_global0, qoff, nb, sc.quads.as<int4>(),
                                (long long)nquads, o->max_quads_per_base, seed, sc.T.as<float>(), flag);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((nquads + 1) / 2048 + 4096) * 4));
  int rc = pgp_scan_exclusive_u32(ctx, flag, (int64_t)nquads + 1, ctx->scene.scratch.as<uint32_t>());
  if (rc) return rc;
  k2b_base_out<<<1, 1024, 0, st>>>(flag, qoff, nb, o->max_quads_per_base, outoff);
  k2b_append<<<gr, 128, 0, st>>>(sc.T.as<float>(), flag, qoff, nb, o->max_quads_per_base, outoff, (long long)nquads, dst, room);
  ctx->launches += 2;
  PGP_CUDA(ctx, cudaGetLastError());
  uint32_t n = 0;
  PGP_CUDA(ctx, cudaMemcpyAsync(&n, outoff + nb, 4, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  *added = std::min<int64_t>(room, (int64_t)n);
  return PGP_OK;
}

}  // namespace

// Congruent quads of ONE base in operMode 2 (parity hook): base4 = scene ids, quads_host: cap x 4, sorted by (v1, v2, v3, v4)
int k2_find_quads_v4pcs(pgp_ctx* ctx, const Model& m, const int32_t* base4, float eps, int32_t* quads_host, int64_t cap, int64_t* n_quads) {
  Scratch& sc = scratch_of(ctx);
  const Scene& s = ctx->scene;
  for (int k = 0; k < 4; ++k)
    if (base4[k] < 0 || base4[k] >= s.n) return pgp_fail(ctx, PGP_E_INVALID, "base id out of range");
  PGP_CUDA(ctx, sc.base.reserve(sizeof(BaseOut) + 64));
  PGP_CUDA(ctx, sc.off.reserve(64 * 4));
  BaseOut h{};
  for (int k = 0; k < 4; ++k) h.id[k] = base4[k];
  h.ok = 1;
  BaseOut* d_base = reinterpret_cast<BaseOut*>(sc.base.as<char>() + 64);
  PGP_CUDA(ctx, cudaMemcpyAsync(d_base, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));      // h is a local
  uint64_t nquads = 0;
  int rc = v4pcs_chunk(ctx, m, d_base, 1, eps, sc.off.as<uint32_t>(), &nquads);
  if (rc) return rc;
  if (nquads >= (1ull << 31)) return pgp_fail(ctx, PGP_E_TOO_LARGE, "congruent quads of one base exceed 2^31");
  *n_quads = (int64_t)nquads;
  const int64_t k = std::min<int64_t>((int64_t)nquads, cap);
  if (k > 0 && quads_host) PGP_CUDA(ctx, cudaMemcpyAsync(quads_host, sc.quads.p, (size_t)k * 16, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PGP_OK;
}

// Bases [base_lo, base_hi) of the o->n_bases the request draws: every draw (base selection, per-base subset) is keyed by the GLOBAL
// base index, so a base yields the same hypotheses whichever GPU generates it and however the bases are chunked (SURVEY 8e: bases
// shard across GPUs, per-base independence of match4pcsBase.cc:1855-1877).
int k2_generate(pgp_ctx* ctx, Model& m, const pgp_pcs_opts* o, uint64_t seed, int base_lo, int base_hi, int64_t max_hyp, int64_t* n_hyp) {
  Scratch& sc = scratch_of(ctx);
  const Scene& s = ctx->scene;
  cudaStream_t st = ctx->stream;
  *n_hyp = 0;
  m.n_gen = 0;
  m.gen_scored = false;
  m.n_gen_bases = 0;
  if (base_hi <= base_lo) return PGP_OK;
  const int nb_total = base_hi - base_lo;
  sc.bases_owner = &m;
  const int nq = m.nq;
  float max_diam = o->max_base_diameter;
  if (!(max_diam > 0.f)) max_diam = m.search_diameter;   // P_diameter_ estimate of init() (:274-283)
  const float eps = s.delta;          // distance_factor * options_.delta, distance_factor = 1 (match4pcsBase.h:99)
  int depth = 0, chunk;
  uint32_t nbk = 0;
  if (o->mode == 2) {
    // bases per chunk: six nq x nq bit matrices each, about 1 GB in all
    chunk = (int)std::max<double>(1.0, std::min<double>(64.0, 1.0e9 / (24.0 * (double)nq * (double)((nq + 31) / 32))));
  } else {
    // join grid (IndexedNormalSet, normalset.h:117-123); buckets per base capped at 2^15 (collisions are filtered by the key)
    const float eps_n = eps / m.unit_ratio;
    depth = (int)(-std::log2(eps_n));
    if (depth < 0) depth = 0;
    if (depth > 7) return pgp_fail(ctx, PGP_E_TOO_LARGE, "quad join: model diameter / delta too large (grid depth %d > 7)", depth);
    nbk = 1u << std::min(3 * depth, 15);
    // bases per chunk.  Every chunk costs ~25 launches and three host-read totals whatever its size, so chunks are made as large as
    // the join's buffers allow (32 bytes per pair + 8 bytes per hash bucket; budget ~2 GB each of the B200's 180 GB): operMode 0 has
    // ~10 % of nq^2 ordered pairs per (base, edge), operMode 1 the PPF map's mean row length.  A chunk that turns out too large is
    // halved below (`shrink`); the hypotheses do not depend on the chunking.
    const double pairs_per_base = o->mode == 1 ? 3.0 * (double)m.n_ppf_pairs / (double)std::max(1, m.n_ppf_keys) : 0.2 * (double)nq * (double)nq;
    chunk = (int)std::max(1.0, std::min({o->mode == 1 ? 4096.0 : 256.0, 6.0e7 / std::max(1.0, pairs_per_base), 2.5e8 / (double)nbk}));
  }
  PGP_CUDA(ctx, sc.base.reserve((size_t)nb_total * sizeof(BaseOut) + 64));
  PGP_CUDA(ctx, m.gen_T.reserve((size_t)std::max<int64_t>(max_hyp, 1) * 48));
  BaseOut* d_bases_all = reinterpret_cast<BaseOut*>(sc.base.as<char>() + 64);
  const bool stocs = o->mode == 1;
  PpfMapDev pm{};
  if (stocs) {
    if (m.n_ppf_keys <= 0) return pgp_fail(ctx, PGP_E_INVALID, "PCS mode 1 (StoCS) needs the model's PPF map: pgp_set_ppf_map / pgp_build_ppf_map");
    if (!s.has_nrm) return pgp_fail(ctx, PGP_E_INVALID, "PCS mode 1 (StoCS) needs scene normals");
    pm.keys = m.ppf_keys.as<uint32_t>(); pm.offsets = m.ppf_offsets.as<uint32_t>(); pm.pairs = m.ppf_pairs.as<int2>(); pm.n_keys = m.n_ppf_keys;
    StocsParams sp{};
    sp.P = s.unsorted.as<float4>(); sp.aux = s.aux_orig.as<float4>(); sp.n = s.n; sp.bits = m.ppf_bits.as<uint32_t>();
    sp.seed = seed;
    const size_t smem_sel = (size_t)s.n * 12 + 16;                    // the weights of one base: n floats + n doubles in shared memory
    if (smem_sel <= 200 * 1024) {
      PGP_CUDA(ctx, cudaFuncSetAttribute(k2s_select_bases<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sel));
      sp.curr = nullptr; sp.base0 = base_lo;
      k2s_select_bases<true><<<nb_total, K2S_T, smem_sel, st>>>(sp, d_bases_all);
    } else {
      // larger scenes: one weight vector of |P| floats per base in global memory, the bases selected in batches of at most ~1 GB of them
      const int bsel = (int)std::max<int64_t>(1, std::min<int64_t>(nb_total, ((int64_t)1 << 28) / std::max(1, s.n)));
      PGP_CUDA(ctx, sc.curr.reserve((size_t)bsel * s.n * 4));
      sp.curr = sc.curr.as<float>();
      for (int b0 = 0; b0 < nb_total; b0 += bsel) {
        sp.base0 = base_lo + b0;
        k2s_select_bases<false><<<std::min(bsel, nb_total - b0), 256, 0, st>>>(sp, d_bases_all + b0);
        if (b0) ctx->launches++;
      }
    }
  } else if (o->mode == 2) {
    k2v_select_bases<<<nb_total, 256, 0, st>>>(s.unsorted.as<float4>(), s.n, max_diam, std::max(1, o->base_trials), seed, base_lo, d_bases_all);
  } else {
    k2_select_bases<<<nb_total, 256, 0, st>>>(s.unsorted.as<float4>(), s.n, max_diam, std::max(1, o->base_trials), seed, base_lo, d_bases_all);
  }
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  int64_t cur = 0;
  // A chunk whose pair lists or congruent quads outgrow the 32-bit offsets / the free device memory (highly symmetric models: very
  // many pairs at one distance) is retried with half as many bases; one base alone that does not fit is an error.
  size_t mem_free = 0, mem_total = 0;
  PGP_CUDA(ctx, cudaMemGetInfo(&mem_free, &mem_total));
  int nb = 0;
  for (int base0 = 0; base0 < nb_total && cur < max_hyp; base0 += nb) {
    nb = std::min(chunk, nb_total - base0);
    const int ncombo = 2 * nb;
    auto shrink = [&]() { if (nb <= 1) return false; chunk = std::max(1, nb / 2); nb = 0; return true; };   // nb = 0: the loop repeats base0
    const BaseOut* d_bases = d_bases_all + base0;
    PGP_CUDA(ctx, sc.off.reserve((size_t)(4 * nb + 16) * 4 + 64));
    uint32_t* coff = sc.off.as<uint32_t>();            // ncombo + 1
    uint32_t* qoff = coff + ncombo + 2;                // nb + 1
    uint32_t* outoff = qoff + nb + 2;                  // nb + 1
    const int64_t room = max_hyp - cur;
    int64_t added = 0;
    int rc;
    if (o->mode == 2) {
      // ---- V4PCS quads of the chunk, then the unfused tail
      uint64_t nquads = 0;
      rc = v4pcs_chunk(ctx, m, d_bases, nb, eps, qoff, &nquads);
      if (rc) return rc;
      if (nquads == 0) continue;
      if (nquads >= (1ull << 31)) {
        if (shrink()) continue;
        return pgp_fail(ctx, PGP_E_TOO_LARGE, "congruent quads of one base exceed 2^31");
      }
      rc = append_unfused(ctx, m, o, seed, d_bases, base_lo + base0, nb, qoff, nquads, outoff, m.gen_T.as<float>() + 12 * cur, room, &added);
      if (rc) return rc;
      cur += added;
      continue;
    }
    // ---- pairs of all 2 nb (base, edge) combos
    const size_t ncnt = (size_t)ncombo * nq;
    PGP_CUDA(ctx, sc.cnt.reserve((ncnt + 1) * 4));
    uint32_t* cnt = sc.cnt.as<uint32_t>();
    int64_t ntot = 0;
    if (stocs) {
      // pair lists come out of the PPF map: count per combo, scan, copy
      int* slot = reinterpret_cast<int*>(cnt);
      PGP_CUDA(ctx, cudaMemsetAsync(coff, 0, (size_t)(ncombo + 1) * 4, st));
      k2s_combo_counts<<<(ncombo + 63) / 64, 64, 0, st>>>(pm, s.unsorted.as<float4>(), s.aux_orig.as<float4>(), d_bases, ncombo, coff, slot);
      ctx->launches++;
      PGP_CUDA(ctx, cudaGetLastError());
      uint64_t tot = 0;
      rc = scan_u32(ctx, coff, ncombo, &tot);                               // sync 1
      if (rc) return rc;
      ntot = (int64_t)tot;
      if (ntot == 0) continue;
      if (ntot >= (1ll << 31) || (size_t)ntot * 24 > mem_free / 2) {
        if (shrink()) continue;
        return pgp_fail(ctx, PGP_E_TOO_LARGE, "pair lists of one base exceed 2^31 entries / the device memory");
      }
      PGP_CUDA(ctx, sc.pairs1.reserve((size_t)ntot * 8));
      k2s_combo_copy<<<dim3(64, (unsigned)ncombo), 256, 0, st>>>(pm, slot, coff, sc.pairs1.as<int2>());
      ctx->launches++;
      PGP_CUDA(ctx, cudaGetLastError());
    } else {
      PGP_CUDA(ctx, cudaMemsetAsync(cnt, 0, (ncnt + 1) * 4, st));
      const dim3 pgrid((unsigned)((nq + 255) / 256), (unsigned)ncombo);
      k2b_pairs<false><<<pgrid, 256, 0, st>>>(m.search.as<float4>(), nq, d_bases, eps, cnt, nullptr);
      ctx->launches++;
      PGP_CUDA(ctx, cudaGetLastError());
      uint64_t unordered = 0;
      rc = scan_u32(ctx, cnt, (int64_t)ncnt, &unordered);                   // sync 1
      if (rc) return rc;
      ntot = (int64_t)unordered * 2;
      if (ntot == 0) continue;
      if (ntot >= (1ll << 31) || (size_t)ntot * 24 > mem_free / 2) {
        if (shrink()) continue;
        return pgp_fail(ctx, PGP_E_TOO_LARGE, "pair lists of one base exceed 2^31 entries / the device memory");
      }
      PGP_CUDA(ctx, sc.pairs1.reserve((size_t)ntot * 8));
      k2b_pairs<true><<<pgrid, 256, 0, st>>>(m.search.as<float4>(), nq, d_bases, eps, cnt, sc.pairs1.as<int2>());
      k2b_combo_offsets<<<(ncombo + 256) / 256, 256, 0, st>>>(cnt, nq, ncombo, coff);
      ctx->launches += 2;
      PGP_CUDA(ctx, cudaGetLastError());
    }
    // ---- join
    JoinParams p{};
    p.Qn = m.search_unit.as<float4>(); p.Q = m.search.as<float4>();
    p.A = sc.pairs1.as<int2>(); p.n1 = ntot; p.B = p.A; p.n2 = ntot;
    p.thr2 = eps;
    p.eg = 1 << depth; p.cell = 1.0f / (float)p.eg; p.n_buckets = nbk;
    p.bases = d_bases; p.coff = coff; p.ncombo = ncombo;
    PGP_CUDA(ctx, sc.cone_tab.reserve((size_t)nb * 64 * sizeof(float2)));
    k2_cone_table<<<nb, 64, 0, st>>>(d_bases, nb, sc.cone_tab.as<float2>());
    ctx->launches++;
    p.cone_tab = sc.cone_tab.as<float2>();
    const size_t nbuckets = (size_t)nb * nbk;
    PGP_CUDA(ctx, sc.bucket_of.reserve((size_t)ntot * 4));
    PGP_CUDA(ctx, sc.key_of.reserve((size_t)ntot * 4));
    PGP_CUDA(ctx, sc.sorted.reserve((size_t)ntot * 4));
    PGP_CUDA(ctx, sc.bucket_start.reserve((nbuckets + 1) * 8));
    uint32_t* bs = sc.bucket_start.as<uint32_t>();
    uint32_t* cursor = bs + nbuckets + 1;
    PGP_CUDA(ctx, cudaMemsetAsync(bs, 0, (nbuckets + 1) * 4, st));
    const unsigned gk = (unsigned)((ntot + 255) / 256);
    k2_join_keys<<<gk, 256, 0, st>>>(p, sc.bucket_of.as<uint32_t>(), sc.key_of.as<uint32_t>(), bs);
    ctx->launches++;
    PGP_CUDA(ctx, cudaGetLastError());
    PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((nbuckets + 1) / 2048 + 4096) * 4));
    rc = pgp_scan_exclusive_u32(ctx, bs, (int64_t)nbuckets + 1, ctx->scene.scratch.as<uint32_t>());
    if (rc) return rc;
    PGP_CUDA(ctx, cudaMemcpyAsync(cursor, bs, nbuckets * 4, cudaMemcpyDeviceToDevice, st));
    k2_join_scatter<<<gk, 256, 0, st>>>(ntot, sc.bucket_of.as<uint32_t>(), cursor, sc.sorted.as<uint32_t>());
    // with a per-base cap the selected quads are transformed inside the join (k2_join_select) and neither the order of the pairs
    // inside a bucket nor the quads themselves are ever needed; the cone masks of the pairs that find quads are kept (48 bytes each)
    const bool fused = o->max_quads_per_base > 0 && nq < 65536 && (size_t)ntot * 48 < mem_free / 4;
    PGP_CUDA(ctx, sc.in_order.reserve(nbuckets + 16));
    if (fused) PGP_CUDA(ctx, cudaMemsetAsync(sc.in_order.p, 1, nbuckets, st));
    else k2_join_sort_buckets<<<(unsigned)((nbuckets + 255) / 256), 256, 0, st>>>(p.A, bs, (long long)nbuckets, sc.sorted.as<uint32_t>(), sc.in_order.as<unsigned char>());
    ctx->launches += 2;
    PGP_CUDA(ctx, cudaGetLastError());
    PGP_CUDA(ctx, sc.cnt2.reserve((size_t)(ntot + 1) * 4));
    uint32_t* cnt2 = sc.cnt2.as<uint32_t>();
    PGP_CUDA(ctx, cudaMemsetAsync(cnt2, 0, (size_t)(ntot + 1) * 4, st));
    // probe -> list of the B pairs with an A pair in their position cell -> count pass on those (dense warps) -> list of the pairs
    // that found quads -> fill pass on those
    PGP_CUDA(ctx, sc.list1.reserve((size_t)ntot * 4 + 16));
    PGP_CUDA(ctx, sc.list2.reserve((size_t)ntot * 4 + 16));
    uint32_t* n_lists = reinterpret_cast<uint32_t*>(ctx->work.as<char>() + 384);      // [0] = |list1|, [1] = |list2|, [2] = staging overflow
    PGP_CUDA(ctx, cudaMemsetAsync(n_lists, 0, 12, st));
    k2_join_probe<<<gk, 256, 0, st>>>(p, bs, sc.sorted.as<uint32_t>(), sc.key_of.as<uint32_t>(), sc.list1.as<uint32_t>(), n_lists);
    const unsigned gq = (unsigned)((ntot + 127) / 128);
    if (fused) PGP_CUDA(ctx, sc.cone.reserve((size_t)ntot * 48 + 64));
    k2_join_query<false><<<gq, 128, 0, st>>>(p, bs, sc.sorted.as<uint32_t>(), sc.key_of.as<uint32_t>(), cnt2, nullptr, 0, sc.in_order.as<unsigned char>(), sc.list1.as<uint32_t>(), n_lists,
                                             sc.list2.as<uint32_t>(), n_lists + 1, fused ? sc.cone.as<uint32_t>() : nullptr);
    ctx->launches += 2;
    PGP_CUDA(ctx, cudaGetLastError());
    uint64_t nquads = 0;
    rc = scan_u32(ctx, cnt2, ntot, &nquads);                                // sync 2
    if (rc) return rc;
    if (nquads == 0) continue;
    if (nquads >= (1ull << 31)) {
      if (shrink()) continue;
      return pgp_fail(ctx, PGP_E_TOO_LARGE, "congruent quads of one base exceed 2^31");
    }
    k2b_quad_offsets<<<(nb + 256) / 256, 256, 0, st>>>(cnt2, coff, nb, qoff);
    ctx->launches++;
    if (fused) {
      // ---- fused: select (the reference's random subset of max_sampled_csets quads per base) BEFORE transforming; see k2_join_select
      const int stage_cap = o->max_quads_per_base * 5 / 2 + 64;            // mean 1.25 max_quads selected per base, sigma ~ sqrt of that
      PGP_CUDA(ctx, sc.stage_n.reserve((size_t)nb * 4 + 16));
      PGP_CUDA(ctx, sc.stage_r.reserve((size_t)nb * stage_cap * 8));
      PGP_CUDA(ctx, sc.stage_T.reserve((size_t)nb * stage_cap * 48));
      PGP_CUDA(ctx, cudaMemsetAsync(sc.stage_n.p, 0, (size_t)nb * 4, st));
      k2_join_select<<<gq, 128, 0, st>>>(p, bs, sc.sorted.as<uint32_t>(), sc.key_of.as<uint32_t>(), cnt2, sc.list2.as<uint32_t>(), n_lists + 1, sc.cone.as<uint32_t>(),
                                         s.unsorted.as<float4>(), qoff, base_lo + base0, o->max_quads_per_base, seed, stage_cap, sc.stage_n.as<uint32_t>(),
                                         sc.stage_r.as<uint32_t>(), sc.stage_T.as<float>());
      k2c_stage_out<<<1, 1024, 0, st>>>(sc.stage_n.as<uint32_t>(), nb, o->max_quads_per_base, stage_cap, outoff, n_lists + 2);
      k2c_stage_append<<<(unsigned)((nb * 32 + 255) / 256), 256, 0, st>>>(sc.stage_n.as<uint32_t>(), sc.stage_r.as<uint32_t>(), sc.stage_T.as<float>(), nb,
                                                                          o->max_quads_per_base, stage_cap, outoff, m.gen_T.as<float>() + 12 * cur, room);
      ctx->launches += 3;
      PGP_CUDA(ctx, cudaGetLastError());
      uint32_t overflow = 0;
      PGP_CUDA(ctx, cudaMemcpyAsync(&overflow, n_lists + 2, 4, cudaMemcpyDeviceToHost, st));
      uint32_t added_f = 0;
      PGP_CUDA(ctx, cudaMemcpyAsync(&added_f, outoff + nb, 4, cudaMemcpyDeviceToHost, st));
      PGP_CUDA(ctx, cudaStreamSynchronize(st));                             // sync 3
      if (overflow) return pgp_fail(ctx, PGP_E_CAPACITY, "more than %d quads of one base passed the random selection (expected ~%d): try another seed", stage_cap, o->max_quads_per_base * 5 / 4);
      cur += std::min<int64_t>(room, (int64_t)added_f);
      continue;
    }
    // ---- unfused (no per-base cap): every quad is materialised, transformed and flagged
    if ((size_t)nquads * 68 > mem_free / 2) {
      if (shrink()) continue;
      return pgp_fail(ctx, PGP_E_TOO_LARGE, "congruent quads of one base exceed the device memory");
    }
    PGP_CUDA(ctx, sc.quads.reserve((size_t)nquads * 16));
    k2_join_query<true><<<gq, 128, 0, st>>>(p, bs, sc.sorted.as<uint32_t>(), sc.key_of.as<uint32_t>(), cnt2, sc.quads.as<int4>(), (long long)nquads,
                                            sc.in_order.as<unsigned char>(), sc.list2.as<uint32_t>(), n_lists + 1);
    ctx->launches++;
    // ---- transforms, subset, compaction behind the hypotheses already generated (sync 3)
    rc = append_unfused(ctx, m, o, seed, d_bases, base_lo + base0, nb, qoff, nquads, outoff, m.gen_T.as<float>() + 12 * cur, room, &added);
    if (rc) return rc;
    cur += added;
  }
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  PGP_CUDA(ctx, cudaGetLastError());
  m.n_gen = std::min<int64_t>(cur, max_hyp);
  m.n_gen_bases = nb_total;
  *n_hyp = m.n_gen;
  return PGP_OK;
}

// bases of the last k2_generate call on this device (they stay in the scratch buffer): ids (n x 4 scene indices,
// in the pairing TryQuadrilateral chose), inv (n x 2), ok flags
int k2_get_bases(pgp_ctx* ctx, const Model& m, int n_bases, int32_t* ids_host, float* inv_host, uint8_t* ok_host) {
  Scratch& sc = scratch_of(ctx);
  if (sc.bases_owner != &m) return pgp_fail(ctx, PGP_E_INVALID, "the bases on the device belong to another object's pgp_generate_pcs call");
  if (n_bases <= 0 || sc.base.cap < (size_t)n_bases * sizeof(BaseOut) + 64) return pgp_fail(ctx, PGP_E_INVALID, "no bases generated");
  std::vector<BaseOut> b(n_bases);
  PGP_CUDA(ctx, cudaMemcpyAsync(b.data(), sc.base.as<char>() + 64, (size_t)n_bases * sizeof(BaseOut), cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < n_bases; ++i) {
    for (int k = 0; k < 4; ++k) ids_host[4 * i + k] = b[i].id[k];
    inv_host[2 * i] = b[i].inv1; inv_host[2 * i + 1] = b[i].inv2;
    ok_host[i] = b[i].ok ? 1 : 0;
  }
  return PGP_OK;
}

// ------------------------------------------------------------------------------- PPF map (host side)
// Installs a map given as {4-int key -> list of (i, j)} rows (what Objects::readPPFMap loads from PPFMap.txt,
// PPE/src/data_layer/Objects.cpp:31-49).  Keys outside the packable range can never be produced by the scene side either.
int k2_set_ppf_map(pgp_ctx* ctx, Model& m, const int32_t* keys4, const int64_t* offsets, const int32_t* pairs, int64_t n_keys) {
  std::vector<std::pair<uint32_t, int64_t>> order;
  order.reserve((size_t)n_keys);
  for (int64_t k = 0; k < n_keys; ++k) {
    const int kk[4] = {keys4[4 * k], keys4[4 * k + 1], keys4[4 * k + 2], keys4[4 * k + 3]};
    const uint32_t pk = ppf_pack(kk);
    if (pk != PPF_NOKEY && offsets[k + 1] > offsets[k]) order.push_back({pk, k});
  }
  std::stable_sort(order.begin(), order.end(), [](const std::pair<uint32_t, int64_t>& a, const std::pair<uint32_t, int64_t>& b) { return a.first < b.first; });
  m.h_ppf_keys.clear(); m.h_ppf_offsets.clear(); m.h_ppf_pairs.clear();
  m.h_ppf_offsets.push_back(0);
  for (size_t t = 0; t < order.size(); ++t) {
    const int64_t k = order[t].second;
    if (t > 0 && order[t].first == order[t - 1].first) {       // duplicate key rows: concatenate
      m.h_ppf_offsets.pop_back();
    } else {
      m.h_ppf_keys.push_back(order[t].first);
    }
    for (int64_t e = offsets[k]; e < offsets[k + 1]; ++e) {
      const int32_t i = pairs[2 * e], j = pairs[2 * e + 1];
      if (i < 0 || j < 0 || i >= m.nq || j >= m.nq) return pgp_fail(ctx, PGP_E_INVALID, "PPF map pair (%d, %d) out of range for a %d-point search cloud", i, j, m.nq);
      m.h_ppf_pairs.push_back(i); m.h_ppf_pairs.push_back(j);
    }
    if (m.h_ppf_pairs.size() / 2 >= (1ull << 31)) return pgp_fail(ctx, PGP_E_TOO_LARGE, "PPF map too large");
    m.h_ppf_offsets.push_back((uint32_t)(m.h_ppf_pairs.size() / 2));
  }
  m.n_ppf_keys = (int)m.h_ppf_keys.size();
  m.n_ppf_pairs = (int64_t)m.h_ppf_pairs.size() / 2;
  const size_t bit_words = ((size_t)PPF_D5_MAX << 15) / 32;
  std::vector<uint32_t> bits(bit_words, 0u);
  for (uint32_t pk : m.h_ppf_keys) bits[pk >> 5] |= 1u << (pk & 31);
  cudaStream_t st = ctx->stream;
  PGP_CUDA(ctx, m.ppf_keys.reserve(std::max<size_t>(m.h_ppf_keys.size(), 1) * 4));
  PGP_CUDA(ctx, m.ppf_offsets.reserve(m.h_ppf_offsets.size() * 4));
  PGP_CUDA(ctx, m.ppf_pairs.reserve(std::max<size_t>(m.h_ppf_pairs.size(), 2) * 4));
  PGP_CUDA(ctx, m.ppf_bits.reserve(bit_words * 4));
  if (m.n_ppf_keys) PGP_CUDA(ctx, cudaMemcpyAsync(m.ppf_keys.p, m.h_ppf_keys.data(), m.h_ppf_keys.size() * 4, cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaMemcpyAsync(m.ppf_offsets.p, m.h_ppf_offsets.data(), m.h_ppf_offsets.size() * 4, cudaMemcpyHostToDevice, st));
  if (m.n_ppf_pairs) PGP_CUDA(ctx, cudaMemcpyAsync(m.ppf_pairs.p, m.h_ppf_pairs.data(), m.h_ppf_pairs.size() * 4, cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaMemcpyAsync(m.ppf_bits.p, bits.data(), bit_words * 4, cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  return PGP_OK;
}

// The offline builder the reference does not ship (its PPFMap.txt files are a download): every ordered pair (i, j), i != j,
// of the SEARCH cloud under the key computePPF gives it -- keys on the device (the same function that keys the scene side),
// grouping on the host (stable: rows in (i, j) order inside a key).
int k2_build_ppf_map(pgp_ctx* ctx, Model& m) {
  Scratch& sc = scratch_of(ctx);
  const int n = m.nq;
  if (n > 16384) return pgp_fail(ctx, PGP_E_TOO_LARGE, "PPF map builder: search cloud of %d points (limit 16384)", n);
  const long long np = (long long)n * n;
  PGP_CUDA(ctx, sc.cnt2.reserve((size_t)np * 4));
  k2s_keys<<<(unsigned)((np + 255) / 256), 256, 0, ctx->stream>>>(m.search.as<float4>(), m.search_nrm.as<float4>(), n, nullptr, np, nullptr, sc.cnt2.as<uint32_t>());
  ctx->launches++;
  std::vector<uint32_t> packed((size_t)np);
  PGP_CUDA(ctx, cudaMemcpyAsync(packed.data(), sc.cnt2.p, (size_t)np * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  PGP_CUDA(ctx, cudaGetLastError());
  std::vector<uint32_t> idx;
  idx.reserve((size_t)np);
  for (long long t = 0; t < np; ++t) if (packed[t] != PPF_NOKEY) idx.push_back((uint32_t)t);
  std::stable_sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b) { return packed[a] < packed[b]; });
  std::vector<int32_t> keys4, pairs;
  std::vector<int64_t> offsets;
  pairs.reserve(idx.size() * 2);
  for (size_t t = 0; t < idx.size(); ++t) {
    const uint32_t pk = packed[idx[t]];
    if (t == 0 || pk != packed[idx[t - 1]]) {
      offsets.push_back((int64_t)t);
      keys4.push_back((int32_t)(pk >> 15) * 5); keys4.push_back((int32_t)((pk >> 10) & 31) * 10);
      keys4.push_back((int32_t)((pk >> 5) & 31) * 10); keys4.push_back((int32_t)(pk & 31) * 10);
    }
    pairs.push_back((int32_t)(idx[t] / (uint32_t)n)); pairs.push_back((int32_t)(idx[t] % (uint32_t)n));
  }
  offsets.push_back((int64_t)idx.size());
  return k2_set_ppf_map(ctx, m, keys4.data(), offsets.data(), pairs.data(), (int64_t)keys4.size() / 4);
}

// computePPF of arbitrary scene index pairs (parity hook): keys4_host n x 4
int k2_scene_ppf_keys(pgp_ctx* ctx, const int32_t* pairs_host, int64_t n, int32_t* keys4_host) {
  Scratch& sc = scratch_of(ctx);
  const Scene& s = ctx->scene;
  if (n <= 0) return PGP_OK;
  for (int64_t t = 0; t < 2 * n; ++t)
    if (pairs_host[t] < 0 || pairs_host[t] >= s.n) return pgp_fail(ctx, PGP_E_INVALID, "scene index out of range");
  PGP_CUDA(ctx, sc.pairs2.reserve((size_t)n * 8));
  PGP_CUDA(ctx, sc.cnt2.reserve((size_t)n * 16));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.pairs2.p, pairs_host, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  k2s_keys<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(s.unsorted.as<float4>(), s.aux_orig.as<float4>(), s.n, sc.pairs2.as<int2>(), n,
                                                                 sc.cnt2.as<int32_t>(), nullptr);
  ctx->launches++;
  PGP_CUDA(ctx, cudaMemcpyAsync(keys4_host, sc.cnt2.p, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

uint32_t k2_stocs_engine_seed(uint64_t seed, int base, int attempt) { return stocs_base_seed(seed, base, attempt); }

void k2_release(pgp_ctx* ctx) {
  if (!ctx->k2_scratch) return;
  Scratch* sc = static_cast<Scratch*>(ctx->k2_scratch);
  for (DevBuf* b : {&sc->adj, &sc->dist6, &sc->in_order, &sc->list1, &sc->list2, &sc->cnt, &sc->cnt2, &sc->off, &sc->flag, &sc->curr, &sc->pairs1, &sc->pairs2, &sc->quads,
                    &sc->bucket_of, &sc->key_of, &sc->bucket_start, &sc->sorted, &sc->T, &sc->ok, &sc->base, &sc->qn, &sc->cone_tab, &sc->cone, &sc->stage_n, &sc->stage_r, &sc->stage_T})
    b->release();
  delete sc;
  ctx->k2_scratch = nullptr;
}
