// K1b -- fine tri-state classification of the scene grid.
//
// The reference decides "is some scene point within delta of T q" with a kd-tree descent per
// query (S4/accelerators/kdtree.h:394-459, called from Verify, S4/algorithms/match4pcsBase.cc:
// 1713-1718).  Here the decision is tabulated once per scene for (almost) all of space: every cell
// whose 27-neighbourhood holds scene points is cut into 8x8x8 sub-voxels and each sub-voxel is
// labelled
//     OUT    no scene point can pass d2 <= delta^2 for ANY query that lands in the voxel,
//     IN     one scene point passes it for EVERY query that lands in the voxel,
//     AMBIG  neither could be proven (the voxel straddles the surface of the union of delta-balls).
// Only AMBIG queries (a few %) still run the exact fp32 test in K3, so the labels must be
// conservative under every rounding the scoring kernel can commit; see DESIGN.md "Exactness of the
// tri-state labels" for the bounds behind `inflate`, dlo2 and dhi2.
#include <math.h>

#include "pgp_internal.cuh"

namespace {

constexpr int F = 8;
constexpr int CLS_THREADS = 128;
constexpr int CLS_CHUNK = 512;

// Domination pruning of candidate lists.  For a voxel with centre c and half-size hs (inflated), a scene point p is DOMINATED by a
// scene point b when b is strictly closer than p to every query q = c + e, |e_i| <= hs, that can land in the voxel:
//     |q-p|^2 - |q-b|^2 = (|c-p|^2 - |c-b|^2) + 2 e.(b-p) >= (c2p - c2b) - 2 hs |b-p|_1 > margin.
// Then p can never be the nearest in-range point of such a query, nor tie with it, and whenever p passes d2 <= delta^2 so does b:
// p is dropped from the voxel's list (b stays, or is itself dominated by a point that stays).  `margin` = 1e-5 delta^2 is > 10x the
// rounding of the two fp32 squared distances K3 compares (relative 3e-7 of <= 2 delta^2 each); the 1e-5 (c2p + c2b) term covers
// the rounding of this test itself.  With 1.25 mm voxels and a few mm between scene points this leaves the 2-3 points whose
// bisector planes cross the voxel instead of every point within delta + voxel diagonal.
__device__ __forceinline__ bool dominated(const float4 p, float bx, float by, float bz, float hs, float c2p, float c2b, float margin) {
  const float spread = 2.0f * hs * (fabsf(bx - p.x) + fabsf(by - p.y) + fabsf(bz - p.z));
  return (c2p - c2b) - spread > margin + 1e-5f * (c2p + c2b);
}

__global__ void k1f_popc(const uint32_t* __restrict__ bitmap, int64_t n_words, uint32_t* __restrict__ out) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < n_words) out[w] = __popc(bitmap[w]);
}
__global__ void k1f_bmrank(const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ prefix, int64_t n_words, int64_t n_cells,
                           uint2* __restrict__ bmrank, uint32_t* __restrict__ block_cell) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_words * 32) return;
  const int64_t w = c >> 5;
  const uint32_t bits = bitmap[w], pre = prefix[w];
  if ((c & 31) == 0) bmrank[w] = make_uint2(bits, pre);
  if (c < n_cells && ((bits >> (c & 31)) & 1u)) block_cell[pre + __popc(bits & ((1u << (c & 31)) - 1u))] = (uint32_t)c;
}

// one CTA per block (= per cell with an occupied 27-neighbourhood): 4 sub-voxels per thread.
// Pass A: labels + per-voxel number of "near" points (candidates of the exact test) + block header.  The block's record region is
// sized for the OVERFLOW records only (beyond the two every AMBIG voxel keeps in its slot, see k1f_fill_lists).
__global__ void __launch_bounds__(CLS_THREADS) k1f_classify(const uint32_t* __restrict__ block_cell, const uint32_t* __restrict__ cell_start,
                                                            const float4* __restrict__ pts, GridParams g, uint32_t* __restrict__ codes,
                                                            uint16_t* __restrict__ near_cnt, uint32_t* __restrict__ hdr,
                                                            uint32_t* __restrict__ region_recs, uint32_t* __restrict__ region_amb,
                                                            unsigned long long* __restrict__ total_recs, int* __restrict__ overflow) {
  __shared__ float4 s_p[CLS_CHUNK];
  __shared__ unsigned char s_code[F * F * F];
  __shared__ uint32_t s_tot;
  const int b = blockIdx.x;
  const uint32_t c = block_cell[b];
  const int cx = (int)(c % g.dim[0]), cy = (int)((c / g.dim[0]) % g.dim[1]), cz = (int)(c / ((uint32_t)g.dim[0] * g.dim[1]));
  const float hs = 0.5f * g.hf + g.inflate;
  float vx[4], vy[4], vz[4];
  bool in[4] = {false, false, false, false};
  int near[4] = {0, 0, 0, 0};
  float bx[4], by[4], bz[4], bc2[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
  const float dom_margin = 1e-5f * g.dhi2;
  if (threadIdx.x == 0) s_tot = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int v = threadIdx.x + CLS_THREADS * j;
    vx[j] = __fmaf_rn((float)(cx * F + (v & 7)) + 0.5f, g.hf, g.lo[0]);
    vy[j] = __fmaf_rn((float)(cy * F + ((v >> 3) & 7)) + 0.5f, g.hf, g.lo[1]);
    vz[j] = __fmaf_rn((float)(cz * F + (v >> 6)) + 0.5f, g.hf, g.lo[2]);
  }
  for (int row = 0; row < 9; ++row) {
    const int oy = row % 3 - 1, oz = row / 3 - 1;
    const int r = ((cz + oz) * g.dim[1] + (cy + oy)) * g.dim[0] + cx;
    const uint32_t s = cell_start[r - 1], e = cell_start[r + 2];
    for (uint32_t base = s; base < e; base += CLS_CHUNK) {
      const int m = (int)min((uint32_t)CLS_CHUNK, e - base);
      __syncthreads();
      for (int t = threadIdx.x; t < m; t += CLS_THREADS) s_p[t] = pts[base + t];
      __syncthreads();
      for (int t = 0; t < m; ++t) {
        const float4 p = s_p[t];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float ax = fabsf(p.x - vx[j]), ay = fabsf(p.y - vy[j]), az = fabsf(p.z - vz[j]);
          const float lx = fmaxf(ax - hs, 0.f), ly = fmaxf(ay - hs, 0.f), lz = fmaxf(az - hs, 0.f);
          const float hx = ax + hs, hy = ay + hs, hz = az + hs;
          const float mind2 = __fmaf_rn(lx, lx, __fmaf_rn(ly, ly, lz * lz));
          const float maxd2 = __fmaf_rn(hx, hx, __fmaf_rn(hy, hy, hz * hz));
          if (mind2 <= g.dhi2) {
            // candidate of the exact test unless the closest-to-centre candidate seen so far dominates it (k1f_fill_lists makes the
            // same decisions in the same sweep order)
            const float c2 = __fmaf_rn(p.x - vx[j], p.x - vx[j], __fmaf_rn(p.y - vy[j], p.y - vy[j], (p.z - vz[j]) * (p.z - vz[j])));
            if (!(bc2[j] < INFINITY && dominated(p, bx[j], by[j], bz[j], hs, c2, bc2[j], dom_margin))) near[j] += 1;
            if (c2 < bc2[j]) { bc2[j] = c2; bx[j] = p.x; by[j] = p.y; bz[j] = p.z; }
          }
          in[j] |= maxd2 <= g.dlo2;
        }
      }
    }
  }
  uint32_t my_list = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int v = threadIdx.x + CLS_THREADS * j;
    const int code = in[j] ? 1 : (near[j] > 0 ? 2 : 0);
    s_code[v] = (unsigned char)code;
    if (code == 2 && near[j] > 65535) atomicOr(overflow, 1);      // absurd density: the host drops the fine grid
    const int nn = code == 2 ? min(near[j], 65535) : 0;
    near_cnt[(size_t)b * 512 + v] = (uint16_t)nn;
    my_list += (uint32_t)max(nn - 2, 0);
  }
  my_list = __reduce_add_sync(0xffffffffu, my_list);
  if ((threadIdx.x & 31) == 0 && my_list) atomicAdd(&s_tot, my_list);
  __syncthreads();
  if (threadIdx.x < 32) {
    uint32_t w = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) w |= (uint32_t)s_code[threadIdx.x * 16 + k] << (2 * k);
    codes[(size_t)b * 32 + threadIdx.x] = w;
    // header: ambig-rank prefix per group of 64 voxels (4 words), number of ambig voxels, overflow records
    const uint32_t amb = __popc(w & 0xAAAAAAAAu);
    uint32_t incl = amb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += t; }
    const uint32_t excl = incl - amb;
    const uint32_t n_amb = __shfl_sync(0xffffffffu, incl, 31);
    // gp[k] = ambig voxels before group k = excl at word 4k
    const uint32_t g_lo = __shfl_sync(0xffffffffu, excl, (threadIdx.x & 3) * 8);       // groups 0,2,4,6
    const uint32_t g_hi = __shfl_sync(0xffffffffu, excl, (threadIdx.x & 3) * 8 + 4);   // groups 1,3,5,7
    if (threadIdx.x < 4) hdr[(size_t)b * 8 + threadIdx.x] = g_lo | (g_hi << 16);
    if (threadIdx.x == 0) {
      hdr[(size_t)b * 8 + 4] = 0;
      hdr[(size_t)b * 8 + 5] = n_amb;
      hdr[(size_t)b * 8 + 6] = s_tot;
      hdr[(size_t)b * 8 + 7] = 0;
      region_recs[b] = s_tot;
      region_amb[b] = n_amb;
      if (s_tot) atomicAdd(total_recs, (unsigned long long)s_tot);
    }
  }
}

// Pass B: candidate lists of the AMBIG voxels, laid out for K3's phase 2.  A voxel's candidates are every scene point whose distance
// to the (inflated) voxel is <= delta (1 + 1e-5), minus the dominated ones, with the candidate closest to the voxel centre FIRST (the
// most likely hit: K3's existence test stops at the first point within delta):
//   hdrw[b * 32 + w]  = global rank of the first AMBIG voxel of label word w of block b (ranks run over all blocks, voxel order),
//   aslot[rank]       = one 32-byte slot per AMBIG voxel, two float4 {x0, y0, z0, n} {x1, y1, z1, first overflow record}: the first
//                       two candidates (the second is a copy of the first when n = 1) and the number of candidates n >= 1,
//   aovf[...]         = float4 copies {x, y, z, original index} of candidates 3 .. n, in list order.
// A query that fell into an AMBIG voxel reads hdrw, then one sector; only when both inline candidates miss and n > 2 does it go on.
__global__ void __launch_bounds__(CLS_THREADS) k1f_fill_lists(const uint32_t* __restrict__ block_cell, const uint32_t* __restrict__ cell_start,
                                                              const float4* __restrict__ pts, GridParams g, const uint32_t* __restrict__ codes,
                                                              const uint16_t* __restrict__ near_cnt, const uint32_t* __restrict__ hdr,
                                                              const uint32_t* __restrict__ ovf_base, const uint32_t* __restrict__ amb_base,
                                                              uint32_t* __restrict__ hdrw, float4* __restrict__ aslot, float4* __restrict__ aovf) {
  __shared__ float4 s_p[CLS_CHUNK];
  __shared__ uint16_t s_av[F * F * F];       // AMBIG voxels in rank order
  __shared__ uint32_t s_off[F * F * F + 1];  // their overflow offsets within the block's region
  const int b = blockIdx.x;
  const uint32_t n_amb = hdr[(size_t)b * 8 + 5];
  const uint32_t abase = amb_base[b], obase = ovf_base[b];
  // rank order = voxel order; per-word rank prefixes + the compact voxel list from the code words
  if (threadIdx.x < 32) {
    const uint32_t w = codes[(size_t)b * 32 + threadIdx.x] & 0xAAAAAAAAu;
    uint32_t cnt = __popc(w), incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += t; }
    uint32_t r = incl - cnt, ww = w;
    hdrw[(size_t)b * 32 + threadIdx.x] = abase + r;
    while (ww) { int bit = __ffs(ww) - 1; ww &= ww - 1; s_av[r++] = (uint16_t)(threadIdx.x * 16 + (bit >> 1)); }
  }
  if (n_amb == 0) return;
  const uint32_t c = block_cell[b];
  const int cx = (int)(c % g.dim[0]), cy = (int)((c / g.dim[0]) % g.dim[1]), cz = (int)(c / ((uint32_t)g.dim[0] * g.dim[1]));
  const float hs = 0.5f * g.hf + g.inflate;
  __syncthreads();
  // offsets: serial scan by one warp over <= 512 entries (tiny)
  if (threadIdx.x < 32) {
    uint32_t run = 0;
    for (uint32_t r0 = 0; r0 < n_amb; r0 += 32) {
      const uint32_t r = r0 + threadIdx.x;
      uint32_t cnt = r < n_amb ? (uint32_t)max((int)near_cnt[(size_t)b * 512 + s_av[r]] - 2, 0) : 0u, incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += t; }
      if (r < n_amb) s_off[r] = run + incl - cnt;
      run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (threadIdx.x == 0) s_off[n_amb] = run;
  }
  __syncthreads();
  // fill: thread t owns AMBIG voxels t, t+128, ... (up to 4).  Candidate k of the sweep goes to slot half k (k < 2) or to overflow
  // record k - 2; afterwards the closest-to-centre candidate trades places with candidate 0.
  float vx[4], vy[4], vz[4], bd2[4], bx[4], by[4], bz[4];
  const float dom_margin = 1e-5f * g.dhi2;
  uint32_t n[4], ovf[4], bpos[4];
  bool live[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t r = threadIdx.x + CLS_THREADS * j;
    live[j] = r < n_amb;
    const int v = live[j] ? s_av[r] : 0;
    vx[j] = __fmaf_rn((float)(cx * F + (v & 7)) + 0.5f, g.hf, g.lo[0]);
    vy[j] = __fmaf_rn((float)(cy * F + ((v >> 3) & 7)) + 0.5f, g.hf, g.lo[1]);
    vz[j] = __fmaf_rn((float)(cz * F + (v >> 6)) + 0.5f, g.hf, g.lo[2]);
    ovf[j] = live[j] ? obase + s_off[r] : 0u;
    n[j] = 0; bpos[j] = 0; bd2[j] = INFINITY;
  }
  auto rec = [&](int j, uint32_t k) -> float4* {
    return k < 2 ? aslot + 2 * (size_t)(abase + threadIdx.x + CLS_THREADS * j) + k : aovf + ovf[j] + (k - 2);
  };
  const uint32_t active_j = (n_amb + CLS_THREADS - 1) / CLS_THREADS;
  for (int row = 0; row < 9; ++row) {
    const int oy = row % 3 - 1, oz = row / 3 - 1;
    const int rr = ((cz + oz) * g.dim[1] + (cy + oy)) * g.dim[0] + cx;
    const uint32_t s = cell_start[rr - 1], e = cell_start[rr + 2];
    for (uint32_t base = s; base < e; base += CLS_CHUNK) {
      const int m = (int)min((uint32_t)CLS_CHUNK, e - base);
      __syncthreads();
      for (int t = threadIdx.x; t < m; t += CLS_THREADS) s_p[t] = pts[base + t];
      __syncthreads();
      for (int t = 0; t < m; ++t) {
        const float4 p = s_p[t];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if ((uint32_t)j < active_j && live[j]) {
            const float dx = p.x - vx[j], dy = p.y - vy[j], dz = p.z - vz[j];
            const float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
            const float lx = fmaxf(ax - hs, 0.f), ly = fmaxf(ay - hs, 0.f), lz = fmaxf(az - hs, 0.f);
            const float mind2 = __fmaf_rn(lx, lx, __fmaf_rn(ly, ly, lz * lz));
            if (mind2 <= g.dhi2) {
              const float c2 = __fmaf_rn(dx, dx, __fmaf_rn(dy, dy, dz * dz));
              const bool keep = !(bd2[j] < INFINITY && dominated(p, bx[j], by[j], bz[j], hs, c2, bd2[j], dom_margin));   // as k1f_classify counted
              if (c2 < bd2[j]) { bd2[j] = c2; bx[j] = p.x; by[j] = p.y; bz[j] = p.z; if (keep) bpos[j] = n[j]; }    // strict <: first of equals
              if (keep) *rec(j, n[j]++) = p;
            }
          }
        }
      }
    }
  }
  // closest candidate first, then the slot's count and overflow offset (own writes, same thread: program order)
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if ((uint32_t)j < active_j && live[j]) {
      float4 r0 = *rec(j, 0);
      if (bpos[j] != 0) { float4* pb = rec(j, bpos[j]); const float4 t = *pb; *pb = r0; r0 = t; }
      const float4 r1 = n[j] > 1 ? *rec(j, 1) : r0;
      *rec(j, 0) = make_float4(r0.x, r0.y, r0.z, __uint_as_float(n[j]));
      *rec(j, 1) = make_float4(r1.x, r1.y, r1.z, __uint_as_float(ovf[j]));
    }
  }
}


// ---------------------------------------------------------------------------------------------
// K1c -- nearest-candidate lists of every non-OUT voxel, for WeightedVerify
// (S4/algorithms/match4pcsBase.cc:1733-1766), which needs the IDENTITY of the nearest in-range
// scene point (KdTree::doQueryRestrictedClosestIndex, S4/accelerators/kdtree.h:394-459), not just
// its existence.  For a voxel V (inflated box) and a scene point p let lo(p) / hi(p) be the
// smallest / largest distance from p to a point of V.  Whatever query q lands in V, its nearest
// scene point p* satisfies d(q,p*) <= d(q,p') <= hi(p') for every p', and d(q,p*) <= delta, hence
//     lo(p*)^2 <= min( min_p' hi(p')^2 , delta^2 )      (+ rounding margins, DESIGN.md 4)
// -- the list of all points passing that bound holds the nearest neighbour (and every point that
// can tie with it) of every query of the voxel.  At 1/8-cell voxels that is ~2 points (after the
// domination pruning) instead of the ~60 in the 27 cells.  Layout: wcnt[block * 512 + voxel] = list length (a byte),
// wword[block * 32 + w] = first entry of label word w's 16 voxels, wlists = the candidates' ORIGINAL indices (4 bytes each;
// the points are read from the cloud in original order, 16 bytes per scene point and L2-resident), vrec = the per-voxel cone
// record that lets scoring skip the search altogether when the candidates' normals agree (k1w_fill).
__device__ __forceinline__ void box_d2(const float4 p, float vx, float vy, float vz, float hs, float& mind2, float& maxd2) {
  const float ax = fabsf(p.x - vx), ay = fabsf(p.y - vy), az = fabsf(p.z - vz);
  const float lx = fmaxf(ax - hs, 0.f), ly = fmaxf(ay - hs, 0.f), lz = fmaxf(az - hs, 0.f);
  const float hx = ax + hs, hy = ay + hs, hz = az + hs;
  mind2 = __fmaf_rn(lx, lx, __fmaf_rn(ly, ly, lz * lz));
  maxd2 = __fmaf_rn(hx, hx, __fmaf_rn(hy, hy, hz * hz));
}

__device__ __forceinline__ float centre_d2(const float4 p, float vx, float vy, float vz) {
  const float dx = p.x - vx, dy = p.y - vy, dz = p.z - vz;
  return __fmaf_rn(dx, dx, __fmaf_rn(dy, dy, dz * dz));
}

// all scene points of the 27 cells around cell (cx,cy,cz), staged through shared memory; every
// thread of the CTA must call it (it synchronises).  fn(point, sorted position)
template <class Fn>
__device__ __forceinline__ void sweep27(const uint32_t* __restrict__ cell_start, const float4* __restrict__ pts, const GridParams& g, int cx, int cy,
                                        int cz, float4* s_p, Fn&& fn) {
  for (int row = 0; row < 9; ++row) {
    const int oy = row % 3 - 1, oz = row / 3 - 1;
    const int r = ((cz + oz) * g.dim[1] + (cy + oy)) * g.dim[0] + cx;
    const uint32_t s = cell_start[r - 1], e = cell_start[r + 2];
    for (uint32_t base = s; base < e; base += CLS_CHUNK) {
      const int m = (int)min((uint32_t)CLS_CHUNK, e - base);
      __syncthreads();
      for (int t = threadIdx.x; t < m; t += CLS_THREADS) s_p[t] = pts[base + t];
      __syncthreads();
      for (int t = 0; t < m; ++t) fn(s_p[t], base + (uint32_t)t);
    }
  }
}

__device__ __forceinline__ float wlist_threshold(float u2, float dhi2) { return fminf(u2 * (1.0f + 4e-5f), dhi2); }

constexpr uint32_t VREC_UNDECIDED = 255u;
constexpr uint32_t WV_CNT_BITS = 8, WV_CNT_MAX = (1u << WV_CNT_BITS) - 1u, WV_REL_MAX = (1u << (32 - WV_CNT_BITS)) - 1u;   // counts are stored as bytes

// Pass A: list length of every voxel of the block (0 for OUT voxels) -> wvox (count only), block total -> region.
// 4 voxels per thread (v = tid + 128 j).
__global__ void __launch_bounds__(CLS_THREADS) k1w_count(const uint32_t* __restrict__ block_cell, const uint32_t* __restrict__ cell_start,
                                                         const float4* __restrict__ pts, GridParams g, const uint32_t* __restrict__ codes,
                                                         uint32_t* __restrict__ wvox, uint32_t* __restrict__ region_entries,
                                                         unsigned long long* __restrict__ total_entries, int* __restrict__ overflow) {
  __shared__ float4 s_p[CLS_CHUNK];
  __shared__ uint32_t s_tot;
  const int b = blockIdx.x;
  const uint32_t c = block_cell[b];
  const int cx = (int)(c % g.dim[0]), cy = (int)((c / g.dim[0]) % g.dim[1]), cz = (int)(c / ((uint32_t)g.dim[0] * g.dim[1]));
  const float hs = 0.5f * g.hf + g.inflate;
  float vx[4], vy[4], vz[4], u2[4], thr[4];
  int cnt[4] = {0, 0, 0, 0};
  bool live[4];
  if (threadIdx.x == 0) s_tot = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int v = threadIdx.x + CLS_THREADS * j;
    vx[j] = __fmaf_rn((float)(cx * F + (v & 7)) + 0.5f, g.hf, g.lo[0]);
    vy[j] = __fmaf_rn((float)(cy * F + ((v >> 3) & 7)) + 0.5f, g.hf, g.lo[1]);
    vz[j] = __fmaf_rn((float)(cz * F + (v >> 6)) + 0.5f, g.hf, g.lo[2]);
    u2[j] = INFINITY;
    live[j] = ((codes[(size_t)b * 32 + (v >> 4)] >> ((v & 15) * 2)) & 3u) != 0u;
  }
  float bx[4], by[4], bz[4], bc2[4] = {INFINITY, INFINITY, INFINITY, INFINITY};     // the scene point closest to the voxel centre
  const float dom_margin = 1e-5f * g.dhi2;
  sweep27(cell_start, pts, g, cx, cy, cz, s_p, [&](const float4 p, uint32_t) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float lo2, hi2; box_d2(p, vx[j], vy[j], vz[j], hs, lo2, hi2); u2[j] = fminf(u2[j], hi2);
      const float c2 = centre_d2(p, vx[j], vy[j], vz[j]);
      if (c2 < bc2[j]) { bc2[j] = c2; bx[j] = p.x; by[j] = p.y; bz[j] = p.z; }
    }
  });
#pragma unroll
  for (int j = 0; j < 4; ++j) thr[j] = wlist_threshold(u2[j], g.dhi2);
  sweep27(cell_start, pts, g, cx, cy, cz, s_p, [&](const float4 p, uint32_t) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float lo2, hi2; box_d2(p, vx[j], vy[j], vz[j], hs, lo2, hi2);
      cnt[j] += (lo2 <= thr[j] && !dominated(p, bx[j], by[j], bz[j], hs, centre_d2(p, vx[j], vy[j], vz[j]), bc2[j], dom_margin)) ? 1 : 0;
    }
  });
  uint32_t mine = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int v = threadIdx.x + CLS_THREADS * j;
    const uint32_t nn = live[j] ? (uint32_t)cnt[j] : 0u;
    if (nn > WV_CNT_MAX) atomicOr(overflow, 1);
    wvox[(size_t)b * 512 + v] = min(nn, WV_CNT_MAX);
    mine += min(nn, WV_CNT_MAX);
  }
  mine = __reduce_add_sync(0xffffffffu, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&s_tot, mine);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_tot > WV_REL_MAX) atomicOr(overflow, 1);
    region_entries[b] = s_tot;
    if (s_tot) atomicAdd(total_entries, (unsigned long long)s_tot);
  }
}

// Pass B: per-block exclusive scan of the counts -> wvox = rel << 8 | count, then the fill: the ORIGINAL INDEX of every candidate
// (4 bytes; scoring fetches the point itself from the L2-resident cloud in original order, Scene::unsorted) and, per voxel, the
// cone record `vrec`:
//     vrec[block * 512 + voxel] = code << 24 | rep
// rep = position of the voxel's first candidate in the CELL-SORTED cloud (Scene::aux: the representatives of neighbouring voxels are
// neighbours in memory, so the 32 look-ups of a warp -- one compact patch of the model -- share sectors); code tells how far the other candidates' normals are from rep's:
//     0          every candidate has bit-identical (unit normal, prior): WeightedVerify's gate and weight do not depend on WHICH
//                candidate is the nearest, so scoring evaluates the exact gate once on rep and never searches,
//     1 .. 254   |n_i - n_rep| <= code * VREC_EPS_STEP for every candidate and all priors are equal: scoring decides the gate for
//                all candidates at once whenever the dot product with rep's normal clears the 30-degree threshold by that margin,
//     255        mixed priors, an empty list, more than 2^24 scene points: always the exact nearest search.
__global__ void __launch_bounds__(CLS_THREADS) k1w_fill(const uint32_t* __restrict__ block_cell, const uint32_t* __restrict__ cell_start,
                                                        const float4* __restrict__ pts, const float4* __restrict__ aux, GridParams g,
                                                        uint32_t* __restrict__ wvox, const uint32_t* __restrict__ region_base,
                                                        uint32_t* __restrict__ wlists, unsigned char* __restrict__ wcnt, uint32_t* __restrict__ wword,
                                                        uint32_t* __restrict__ vrec, int rep_ok) {
  __shared__ float4 s_p[CLS_CHUNK];
  __shared__ uint32_t s_warp[CLS_THREADS / 32];
  const int b = blockIdx.x;
  const uint32_t base = region_base[b];
  const uint32_t c = block_cell[b];
  const int cx = (int)(c % g.dim[0]), cy = (int)((c / g.dim[0]) % g.dim[1]), cz = (int)(c / ((uint32_t)g.dim[0] * g.dim[1]));
  const float hs = 0.5f * g.hf + g.inflate;
  // thread t owns voxels 4t .. 4t+3 here (contiguous, so the scan is one pass)
  uint32_t cnt[4], rel[4];
  uint32_t mine = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) { cnt[j] = wvox[(size_t)b * 512 + threadIdx.x * 4 + j] & WV_CNT_MAX; mine += cnt[j]; }
  uint32_t incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)(threadIdx.x & 31) >= o) incl += t; }
  if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = incl;
  __syncthreads();
  uint32_t run = incl - mine;
  for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) run += s_warp[w];
  const uint32_t total = s_warp[0] + s_warp[1] + s_warp[2] + s_warp[3];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    rel[j] = run; run += cnt[j];
    wvox[(size_t)b * 512 + threadIdx.x * 4 + j] = (rel[j] << WV_CNT_BITS) | cnt[j];
  }
  // what scoring reads (L2-resident: 512 + 128 bytes per block instead of 2 KB): the count of every voxel as a byte, and the first
  // record of every label word's 16 voxels; a voxel's first record = that + the counts of the voxels before it in the word
  *reinterpret_cast<uchar4*>(wcnt + (size_t)b * 512 + threadIdx.x * 4) = make_uchar4((unsigned char)cnt[0], (unsigned char)cnt[1], (unsigned char)cnt[2], (unsigned char)cnt[3]);
  if ((threadIdx.x & 3) == 0) wword[(size_t)b * 32 + (threadIdx.x >> 2)] = base + rel[0];
  uint4* vout = reinterpret_cast<uint4*>(vrec + (size_t)b * 512 + threadIdx.x * 4);
  if (total == 0) { *vout = make_uint4(VREC_UNDECIDED << 24, VREC_UNDECIDED << 24, VREC_UNDECIDED << 24, VREC_UNDECIDED << 24); return; }      // uniform over the CTA
  float vx[4], vy[4], vz[4], u2[4], thr[4];
  uint32_t wr[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int v = threadIdx.x * 4 + j;
    vx[j] = __fmaf_rn((float)(cx * F + (v & 7)) + 0.5f, g.hf, g.lo[0]);
    vy[j] = __fmaf_rn((float)(cy * F + ((v >> 3) & 7)) + 0.5f, g.hf, g.lo[1]);
    vz[j] = __fmaf_rn((float)(cz * F + (v >> 6)) + 0.5f, g.hf, g.lo[2]);
    u2[j] = INFINITY;
    wr[j] = cnt[j] ? base + rel[j] : 0xffffffffu;
  }
  float bx[4], by[4], bz[4], bc2[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
  const float dom_margin = 1e-5f * g.dhi2;
  sweep27(cell_start, pts, g, cx, cy, cz, s_p, [&](const float4 p, uint32_t) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float lo2, hi2; box_d2(p, vx[j], vy[j], vz[j], hs, lo2, hi2); u2[j] = fminf(u2[j], hi2);
      const float c2 = centre_d2(p, vx[j], vy[j], vz[j]);
      if (c2 < bc2[j]) { bc2[j] = c2; bx[j] = p.x; by[j] = p.y; bz[j] = p.z; }
    }
  });
#pragma unroll
  for (int j = 0; j < 4; ++j) thr[j] = wlist_threshold(u2[j], g.dhi2);
  // cone of the candidates' normals around the first candidate's (rep)
  uint32_t rep[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
  float n0x[4], n0y[4], n0z[4], pr0[4], maxd2[4] = {0.f, 0.f, 0.f, 0.f};
  bool mixed[4] = {false, false, false, false};
  sweep27(cell_start, pts, g, cx, cy, cz, s_p, [&](const float4 p, uint32_t pos) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (wr[j] != 0xffffffffu) {
        float lo2, hi2;
        box_d2(p, vx[j], vy[j], vz[j], hs, lo2, hi2);
        if (lo2 <= thr[j] && !dominated(p, bx[j], by[j], bz[j], hs, centre_d2(p, vx[j], vy[j], vz[j]), bc2[j], dom_margin)) {   // as k1w_count counted
          const uint32_t orig = (uint32_t)__float_as_int(p.w);
          wlists[wr[j]++] = orig;
          const float4 a = __ldg(aux + pos);
          if (rep[j] == 0xffffffffu) { rep[j] = pos; n0x[j] = a.x; n0y[j] = a.y; n0z[j] = a.z; pr0[j] = a.w; }
          else {
            const float dx = a.x - n0x[j], dy = a.y - n0y[j], dz = a.z - n0z[j];
            maxd2[j] = fmaxf(maxd2[j], __fmaf_rn(dx, dx, __fmaf_rn(dy, dy, dz * dz)));
            mixed[j] |= a.w != pr0[j];
          }
        }
      }
    }
  });
  uint32_t out[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t code = VREC_UNDECIDED;
    if (rep_ok && rep[j] != 0xffffffffu && !mixed[j]) {
      if (maxd2[j] == 0.f) code = 0u;
      else {
        const float eps = sqrtf(maxd2[j]) * (1.0f + 1e-6f) + 1e-7f;
        const float cf = ceilf(eps / VREC_EPS_STEP);
        code = cf > 254.f ? VREC_UNDECIDED : (uint32_t)fmaxf(cf, 1.f);
      }
    }
    out[j] = (code << 24) | (code == VREC_UNDECIDED ? 0u : rep[j]);
  }
  *vout = make_uint4(out[0], out[1], out[2], out[3]);
}


// statistics of the label structure (reports / tuning): out[0..5] = blocks all-OUT, all-IN, mixed; voxels OUT, IN, AMBIG
__global__ void k1f_stats(const uint32_t* __restrict__ codes, int n_blocks, unsigned long long* __restrict__ out) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= n_blocks) return;
  const uint32_t w = codes[(size_t)b * 32 + (threadIdx.x & 31)];
  const int n_in = __popc(w & 0x55555555u), n_amb = __popc(w & 0xAAAAAAAAu);
  const int tin = __reduce_add_sync(0xffffffffu, n_in), tam = __reduce_add_sync(0xffffffffu, n_amb);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(out + (tin == 512 ? 1 : (tin + tam == 0 ? 0 : 2)), 1ull);
    atomicAdd(out + 3, (unsigned long long)(512 - tin - tam));
    atomicAdd(out + 4, (unsigned long long)tin);
    atomicAdd(out + 5, (unsigned long long)tam);
  }
}


// ---- K1d: lower bound of the distance to the nearest scene point, on a lattice of R sub-cells per cell edge ----------------
// For a sub-cell C and an occupied sub-cell C' that differ by (kx, ky, kz) sub-cells, every point of C is at least
// (h/R) sqrt(gx^2 + gy^2 + gz^2) away from every point of C', g = max(|k| - 1, 0).  S(C) = min over the occupied sub-cells of
// gx^2 + gy^2 + gz^2 separates per axis (a min-plus pass along x, then y, then z, window +-W sub-cells; nothing occupied inside
// the window -> S = W^2, still a lower bound).  K3 uses it to drop whole groups of model points whose bounding sphere cannot
// reach the scene; R = 2 halves what the "|k| - 1" rule gives away (up to one sub-cell per axis).
__global__ void k1d_mark(const float4* __restrict__ pts, int n, GridParams g, int R, unsigned char* __restrict__ occ) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = pts[i];
  const float fr = (float)R;
  int sx = (int)(cell_coord(p.x, g.lo[0], g.inv_h) * fr), sy = (int)(cell_coord(p.y, g.lo[1], g.inv_h) * fr), sz = (int)(cell_coord(p.z, g.lo[2], g.inv_h) * fr);
  sx = min(max(sx, 0), g.dim[0] * R - 1); sy = min(max(sy, 0), g.dim[1] * R - 1); sz = min(max(sz, 0), g.dim[2] * R - 1);
  occ[((size_t)sz * (g.dim[1] * R) + sy) * (g.dim[0] * R) + sx] = 1;
}

template <int PASS>   // 0: occupancy -> S along x, 1: += y, 2: += z and conversion to metres
__global__ void k1d_pass(const unsigned char* __restrict__ occ, const uint16_t* __restrict__ in, uint16_t* __restrict__ out, float* __restrict__ dist,
                         int dx, int dy, int dz, int W, float sub_h) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= (int64_t)dx * dy * dz) return;
  const int cx = (int)(c % dx), cy = (int)((c / dx) % dy), cz = (int)(c / ((int64_t)dx * dy));
  const int pos = PASS == 0 ? cx : PASS == 1 ? cy : cz;
  const int dim = PASS == 0 ? dx : PASS == 1 ? dy : dz;
  const int64_t stride = PASS == 0 ? 1 : PASS == 1 ? dx : (int64_t)dx * dy;
  int best = W * W;
  const int t0 = max(-W, -pos), t1 = min(W, dim - 1 - pos);
  for (int t = t0; t <= t1; ++t) {
    const int64_t cc = c + t * stride;
    const int gap = max(abs(t) - 1, 0);
    const int v = PASS == 0 ? (occ[cc] ? 0 : W * W) : (int)in[cc];
    best = min(best, v + gap * gap);
  }
  if (PASS < 2) out[c] = (uint16_t)best;
  // 0.04 sub-cells: the sub-cell of a point is computed in fp32 (error < 2e-3 sub-cells per axis, DESIGN.md), (1 - 1e-4): sqrtf / product rounding
  else dist[c] = fmaxf(0.f, sub_h * sqrtf((float)best) * (1.0f - 1e-4f) - 0.04f * sub_h);
}

}  // namespace

int k1_build_fine(pgp_ctx* ctx) {
  Scene& s = ctx->scene;
  GridParams& g = s.g;
  cudaStream_t st = ctx->stream;
  const int64_t nw = s.bitmap_words;
  g.fine = 0; g.n_blocks = 0;
  s.wlists_ready = false; s.wlists_tried = false;
  // rank structure over the dilated-occupancy bitmap
  PGP_CUDA(ctx, s.bmrank.reserve((size_t)nw * 8 + 16));
  PGP_CUDA(ctx, s.cursor.reserve((size_t)(nw + 1) * 4));
  PGP_CUDA(ctx, s.scratch.reserve((size_t)((nw + 1) / 2048 + 4096) * 4));
  uint32_t* pre = s.cursor.as<uint32_t>();
  PGP_CUDA(ctx, cudaMemsetAsync(pre, 0, (size_t)(nw + 1) * 4, st));
  k1f_popc<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>(s.bitmap.as<uint32_t>(), nw, pre);
  ctx->launches++;
  int rc = pgp_scan_exclusive_u32(ctx, pre, nw + 1, s.scratch.as<uint32_t>());
  if (rc) return rc;
  uint32_t nb = 0;
  PGP_CUDA(ctx, cudaMemcpyAsync(&nb, pre + nw, 4, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  if ((size_t)nb * 128 > ((size_t)8 << 30)) return PGP_OK;      // absurdly large (and label offsets are 32-bit): stay on the 27-cell path
  PGP_CUDA(ctx, s.block_cell.reserve((size_t)nb * 4 + 16));
  PGP_CUDA(ctx, s.codes.reserve((size_t)nb * 128 + 256));
  PGP_CUDA(ctx, cudaMemsetAsync(s.codes.as<char>() + (size_t)nb * 128, 0, 128, st));   // zero dummy block behind the last one
  k1f_bmrank<<<(unsigned)((nw * 32 + 255) / 256), 256, 0, st>>>(s.bitmap.as<uint32_t>(), pre, nw, g.n_cells, s.bmrank.as<uint2>(),
                                                              s.block_cell.as<uint32_t>());
  ctx->launches++;

  // conservative margins (DESIGN.md): positions are uncertain by eps_pos (fast FMA transform vs the
  // reference's rounding sequence) plus the rounding of the voxel index itself.
  float maxabs = 0.f;
  int dmax = 0;
  for (int k = 0; k < 3; ++k) {
    maxabs = fmaxf(maxabs, fmaxf(fabsf(g.lo[k]), fabsf(g.lo[k] + g.h * (float)g.dim[k])));
    dmax = g.dim[k] > dmax ? g.dim[k] : dmax;
  }
  g.hf = g.h / (float)F;
  g.inv_hf = g.inv_h * (float)F;
  g.pos_bound = 3.0f * maxabs;
  const float eps_pos = 32.0f * 5.9604645e-8f * (g.pos_bound + maxabs);
  g.inflate = g.hf * (2e-3f + 16.0f * 5.9604645e-8f * (float)(dmax * F)) + eps_pos;
  const double d = (double)s.delta;
  g.dlo2 = (float)((d * (1.0 - 1e-5)) * (d * (1.0 - 1e-5)));
  g.dhi2 = (float)((d * (1.0 + 1e-5)) * (d * (1.0 + 1e-5)));
  // the OUT label also needs: everything within delta(1+1e-5) + inflate of a cell lies in its 27 cells
  if (!((double)g.h * (1.0 - 4e-4) >= d * (1.0 + 1e-5) + (double)g.inflate)) return PGP_OK;   // margins do not close: no fine grid
  s.n_ovf_records = 0;
  if ((size_t)nb * 32 >= ((size_t)1 << 28)) return PGP_OK;          // K3 packs (label word index, rank) into one 32-bit queue entry
  if (nb > 0) {
    PGP_CUDA(ctx, s.near_cnt.reserve((size_t)nb * 512 * 2));
    PGP_CUDA(ctx, s.hdr.reserve((size_t)nb * 32));
    PGP_CUDA(ctx, s.hdrw.reserve((size_t)nb * 128));
    PGP_CUDA(ctx, s.region.reserve((size_t)(nb + 1) * 8));
    PGP_CUDA(ctx, s.scratch.reserve((size_t)((nb + 1) / 2048 + 4096) * 4));
    uint32_t* region = s.region.as<uint32_t>();            // overflow records per block -> first overflow record of the block
    uint32_t* region_amb = region + (nb + 1);              // AMBIG voxels per block -> global rank of the block's first one
    unsigned long long* d_total = reinterpret_cast<unsigned long long*>(ctx->work.as<char>() + 192);
    PGP_CUDA(ctx, cudaMemsetAsync(region, 0, (size_t)(nb + 1) * 8, st));
    PGP_CUDA(ctx, cudaMemsetAsync(d_total, 0, 8, st));
    PGP_CUDA(ctx, cudaMemsetAsync(ctx->work.as<int>() + 40, 0, 4, st));
    k1f_classify<<<nb, CLS_THREADS, 0, st>>>(s.block_cell.as<uint32_t>(), s.cell_start.as<uint32_t>(), s.pts.as<float4>(), g, s.codes.as<uint32_t>(),
                                             s.near_cnt.as<uint16_t>(), s.hdr.as<uint32_t>(), region, region_amb, d_total, ctx->work.as<int>() + 40);
    ctx->launches++;
    rc = pgp_scan_exclusive_u32(ctx, region, (int64_t)nb + 1, s.scratch.as<uint32_t>());
    if (rc) return rc;
    rc = pgp_scan_exclusive_u32(ctx, region_amb, (int64_t)nb + 1, s.scratch.as<uint32_t>());
    if (rc) return rc;
    unsigned long long total = 0;
    uint32_t n_amb_total = 0;
    int overflow = 0;
    PGP_CUDA(ctx, cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaMemcpyAsync(&n_amb_total, region_amb + nb, 4, cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaMemcpyAsync(&overflow, ctx->work.as<int>() + 40, 4, cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaStreamSynchronize(st));
    if (overflow || total >= (1ull << 32) - 64) return PGP_OK;     // g.fine stays 0: scoring uses the 27-cell path
    size_t free_b = 0, total_b = 0;
    PGP_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
    if ((size_t)total * 16 + (size_t)n_amb_total * 32 + ((size_t)256 << 20) > free_b + s.aovf.cap + s.aslot.cap) return PGP_OK;
    PGP_CUDA(ctx, s.aovf.reserve((size_t)total * 16 + 16));
    PGP_CUDA(ctx, s.aslot.reserve((size_t)n_amb_total * 32 + 32));     // (cudaMalloc: 256-byte aligned, so every slot is one sector)
    k1f_fill_lists<<<nb, CLS_THREADS, 0, st>>>(s.block_cell.as<uint32_t>(), s.cell_start.as<uint32_t>(), s.pts.as<float4>(), g, s.codes.as<uint32_t>(),
                                               s.near_cnt.as<uint16_t>(), s.hdr.as<uint32_t>(), region, region_amb, s.hdrw.as<uint32_t>(),
                                               s.aslot.as<float4>(), s.aovf.as<float4>());
    ctx->launches++;
    s.n_ovf_records = (int64_t)total;
    s.n_ambig_voxels = (int64_t)n_amb_total;
  }
  // K1d distance field on the R-times refined lattice (R = 2 unless the grid is huge)
  {
    const int R = g.n_cells <= (16ll << 20) ? 2 : 1;
    const int dx = g.dim[0] * R, dy = g.dim[1] * R, dz = g.dim[2] * R;
    const int64_t ns = (int64_t)dx * dy * dz;
    const int W = 12 * R;                                   // 12 cells: beyond that a group is culled whatever its radius
    PGP_CUDA(ctx, s.dist.reserve((size_t)ns * 4));
    PGP_CUDA(ctx, s.dist_tmp.reserve((size_t)ns * 5 + 64));
    unsigned char* occ = s.dist_tmp.as<unsigned char>();
    uint16_t* pa = reinterpret_cast<uint16_t*>(occ + ((ns + 63) & ~63ll));
    uint16_t* pb = pa + ns;
    PGP_CUDA(ctx, cudaMemsetAsync(occ, 0, (size_t)ns, st));
    k1d_mark<<<(s.n + 255) / 256, 256, 0, st>>>(s.pts.as<float4>(), s.n, g, R, occ);
    const unsigned blocks = (unsigned)((ns + 255) / 256);
    const float sub_h = g.h / (float)R;
    k1d_pass<0><<<blocks, 256, 0, st>>>(occ, nullptr, pa, nullptr, dx, dy, dz, W, sub_h);
    k1d_pass<1><<<blocks, 256, 0, st>>>(nullptr, pa, pb, nullptr, dx, dy, dz, W, sub_h);
    k1d_pass<2><<<blocks, 256, 0, st>>>(nullptr, pb, nullptr, s.dist.as<float>(), dx, dy, dz, W, sub_h);
    ctx->launches += 4;
    s.dist_r = R;
  }
  PGP_CUDA(ctx, cudaGetLastError());
  g.n_blocks = (int)nb;
  g.fine = F;
  return PGP_OK;
}

// K1c driver: built lazily by the first WEIGHTED scoring call on a scene (k3_score).
// Leaves scene.wlists_ready false (scoring keeps the 27-cell search) when the lists would not fit.
int k1_build_wlists(pgp_ctx* ctx) {
  Scene& s = ctx->scene;
  const GridParams& g = s.g;
  s.wlists_ready = false;
  s.wlists_tried = true;
  if (g.fine != F || g.n_blocks <= 0) return PGP_OK;
  cudaStream_t st = ctx->stream;
  const uint32_t nb = (uint32_t)g.n_blocks;
  size_t free_b = 0, total_b = 0;
  PGP_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
  if ((size_t)nb * 2048 + (64u << 20) > free_b + s.wvox.cap) return PGP_OK;
  PGP_CUDA(ctx, s.wvox.reserve((size_t)nb * 512 * 4));
  PGP_CUDA(ctx, s.wbase.reserve((size_t)(nb + 1) * 4));
  PGP_CUDA(ctx, s.wcnt.reserve((size_t)nb * 512 + 64));
  PGP_CUDA(ctx, s.wword.reserve((size_t)nb * 128 + 64));
  PGP_CUDA(ctx, s.scratch.reserve((size_t)((nb + 1) / 2048 + 4096) * 4));
  uint32_t* region = s.wbase.as<uint32_t>();
  unsigned long long* d_total = reinterpret_cast<unsigned long long*>(ctx->work.as<char>() + 192);
  int* d_over = ctx->work.as<int>() + 40;
  PGP_CUDA(ctx, cudaMemsetAsync(region, 0, (size_t)(nb + 1) * 4, st));
  PGP_CUDA(ctx, cudaMemsetAsync(d_total, 0, 8, st));
  PGP_CUDA(ctx, cudaMemsetAsync(d_over, 0, 4, st));
  k1w_count<<<nb, CLS_THREADS, 0, st>>>(s.block_cell.as<uint32_t>(), s.cell_start.as<uint32_t>(), s.pts.as<float4>(), g, s.codes.as<uint32_t>(),
                                        s.wvox.as<uint32_t>(), region, d_total, d_over);
  ctx->launches++;
  unsigned long long total = 0;
  int overflow = 0;
  PGP_CUDA(ctx, cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaMemcpyAsync(&overflow, d_over, 4, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  if (overflow || total >= (1ull << 32) - 64) return PGP_OK;      // 32-bit entry offsets
  PGP_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
  if ((size_t)total * 4 + (size_t)nb * 2048 + (64u << 20) > free_b + s.wlists.cap + s.vrec.cap) return PGP_OK;
  int rc = pgp_scan_exclusive_u32(ctx, region, (int64_t)nb + 1, s.scratch.as<uint32_t>());
  if (rc) return rc;
  PGP_CUDA(ctx, s.wlists.reserve((size_t)total * 4 + 16));
  PGP_CUDA(ctx, s.vrec.reserve((size_t)nb * 2048 + 16));
  k1w_fill<<<nb, CLS_THREADS, 0, st>>>(s.block_cell.as<uint32_t>(), s.cell_start.as<uint32_t>(), s.pts.as<float4>(), s.aux.as<float4>(), g,
                                       s.wvox.as<uint32_t>(), region, s.wlists.as<uint32_t>(), s.wcnt.as<unsigned char>(), s.wword.as<uint32_t>(),
                                       s.vrec.as<uint32_t>(), s.n <= (1 << 24) ? 1 : 0);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  s.n_wlist_entries = (int64_t)total;
  s.wlists_ready = true;
  return PGP_OK;
}

int k1_fine_stats(pgp_ctx* ctx, int64_t* out8) {
  Scene& s = ctx->scene;
  for (int i = 0; i < 8; ++i) out8[i] = 0;
  if (s.g.fine != F || s.g.n_blocks <= 0) return PGP_OK;
  unsigned long long* d = reinterpret_cast<unsigned long long*>(ctx->work.as<char>() + 256);
  PGP_CUDA(ctx, cudaMemsetAsync(d, 0, 64, ctx->stream));
  k1f_stats<<<(s.g.n_blocks + 7) / 8, 256, 0, ctx->stream>>>(s.codes.as<uint32_t>(), s.g.n_blocks, d);
  ctx->launches++;
  unsigned long long h[8];
  PGP_CUDA(ctx, cudaMemcpyAsync(h, d, 64, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < 6; ++i) out8[i] = (int64_t)h[i];
  out8[6] = s.n_ovf_records;
  out8[7] = s.wlists_ready ? s.n_wlist_entries : 0;
  return PGP_OK;
}
