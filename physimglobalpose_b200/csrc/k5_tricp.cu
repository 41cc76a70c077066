// K5 -- trimmed ICP refinement of the top-k poses, one CTA per pose, the whole iteration loop on
// the device (no host round trip per iteration).
//
// Replaces pcl::recognition::TrimmedICP<pcl::PointXYZ,float>::align as called from
// UCTState::performTrICP (PPE/src/hypothesis_verification/mcts/UCTState.cpp:121-204) and
// utilities::performTrICP (PPE/src/misc/utilities.cpp:651-680): target = model cloud, source = scene
// segment, guess = inverse(pose), n_keep = |trim * N_src| truncated, loop while
// energy/old_energy < ratio.  PCL is not vendored in the reference tree: the algorithm follows the
// call sites and PCL's published TrimmedICP (the CPU checker restates the same algorithm; PARITY UNPINNED, see DESIGN.md).
//
// Per iteration and pose: exact 1-NN of every transformed source point in a model-space grid
// (ring search with a proven stop bound), radix-select of the n_keep-th smallest squared distance,
// 16 double sums (energy, two centroids, 3x3 cross products) block-reduced, Horn's closed-form
// rotation from the 4x4 symmetric eigenproblem (Jacobi) -- the same fit as SVD/Umeyama without scale.
#include <cooperative_groups.h>
#include <float.h>
#include <math.h>

#include <algorithm>
#include <vector>

#include "pgp_internal.cuh"

namespace {

constexpr int TT = 1024;

struct TGrid { float lo[3]; float g, inv_g; int dim[3]; };

struct TricpParams {
  const float4* src; int ns;
  const float4* tgt; const uint32_t* tstart; TGrid tg; int nt;   // target sorted by grid cell (w = original index)
  const float4* tgt_orig;                                          // target in original order
  float* d2; int* nn;            // k x ns scratch
  float* T;                      // k x 12, in/out (source -> target)
  int n_keep; float ratio; int max_iter;
  int* iters; float* energy;
};

__global__ void k5_tgrid_count(const float4* __restrict__ pts, int n, TGrid tg, uint32_t* __restrict__ cell_of, uint32_t* __restrict__ counts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = pts[i];
  int cx = min(max((int)((p.x - tg.lo[0]) * tg.inv_g), 0), tg.dim[0] - 1);
  int cy = min(max((int)((p.y - tg.lo[1]) * tg.inv_g), 0), tg.dim[1] - 1);
  int cz = min(max((int)((p.z - tg.lo[2]) * tg.inv_g), 0), tg.dim[2] - 1);
  const uint32_t c = (uint32_t)((cz * tg.dim[1] + cy) * tg.dim[0] + cx);
  cell_of[i] = c;
  atomicAdd(counts + c, 1u);
}
__global__ void k5_tgrid_scatter(const float4* __restrict__ pts, int n, const uint32_t* __restrict__ cell_of, uint32_t* __restrict__ cursor,
                                 float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = pts[i];
  p.w = __int_as_float(i);
  out[atomicAdd(cursor + cell_of[i], 1u)] = p;
}

// exact 1-NN: rings of cells around the (clamped) query cell; after ring r every unvisited point is at least r*g away, so the
// search stops once best <= (r g)^2 -- or, with a finite cap2, once (r g)^2 >= cap2: then every unvisited point is farther than
// sqrt(cap2) and the caller only needs to know THAT (the trimmed set keeps the n_keep smallest distances; a point beyond the
// current trim radius is dropped whatever its exact distance).  A result <= cap2 is always the exact nearest neighbour.
// In fp32 the cell coordinate fl(fl(x - lo) * inv_g) of a point or query is off by up to 3 * 2^-24 * u cells (u <= rmax inside the
// grid; a clamped query is farther out than its cell says), so a point just across a face can sit (r - 1 - 6 * 2^-24 * rmax) g
// from the query: the bound subtracts that (as 4 FLT_EPSILON * rmax cells), and the 1e-6 factor covers the rounding of d2.
// The returned id is always in [0, nt): a query whose squared distances are all NaN or overflow (none below FLT_MAX) gets id 0
// with d2 = FLT_MAX, as the capped branch reports a point beyond the cap.
__device__ __forceinline__ void nn_search(const TricpParams& p, float qx, float qy, float qz, float cap2, float& best, int& best_id) {
  const TGrid& tg = p.tg;
  const int cx = min(max((int)floorf((qx - tg.lo[0]) * tg.inv_g), 0), tg.dim[0] - 1);
  const int cy = min(max((int)floorf((qy - tg.lo[1]) * tg.inv_g), 0), tg.dim[1] - 1);
  const int cz = min(max((int)floorf((qz - tg.lo[2]) * tg.inv_g), 0), tg.dim[2] - 1);
  best = FLT_MAX; best_id = -1;
  const int rmax = max(tg.dim[0], max(tg.dim[1], tg.dim[2]));
  const float slack = 4.0f * FLT_EPSILON * (float)rmax * tg.g;
  for (int r = 0; r <= rmax; ++r) {
    if (r > 0) {
      const float bound = fmaxf((float)(r - 1) * tg.g - slack, 0.f);   // ring r-1 is complete: unvisited points are >= (r-1) g away
      const float b2 = bound * bound * 0.999999f;
      if (best_id >= 0 && best <= b2) break;
      if (b2 >= cap2) { if (!(best <= cap2)) { best = FLT_MAX; best_id = 0; } break; }
    }
    const int z0 = max(cz - r, 0), z1 = min(cz + r, tg.dim[2] - 1), y0 = max(cy - r, 0), y1 = min(cy + r, tg.dim[1] - 1);
    const int x0 = max(cx - r, 0), x1 = min(cx + r, tg.dim[0] - 1);
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) {
        const bool shell_row = (abs(z - cz) == r) || (abs(y - cy) == r);
        const int rowbase = (z * tg.dim[1] + y) * tg.dim[0];
        if (shell_row) {
          const uint32_t s = p.tstart[rowbase + x0], e = p.tstart[rowbase + x1 + 1];
          for (uint32_t i = s; i < e; ++i) {
            const float4 t = p.tgt[i];
            const float dx = qx - t.x, dy = qy - t.y, dz = qz - t.z;
            const float d2 = dx * dx + dy * dy + dz * dz;
            const int id = __float_as_int(t.w);
            if (d2 < best || (d2 == best && id < best_id)) { best = d2; best_id = id; }
          }
        } else {
          // only the two end cells of this row belong to ring r
#pragma unroll
          for (int side = 0; side < 2; ++side) {
            const int x = side == 0 ? cx - r : cx + r;
            if (x < 0 || x >= tg.dim[0]) continue;
            const uint32_t s = p.tstart[rowbase + x], e = p.tstart[rowbase + x + 1];
            for (uint32_t i = s; i < e; ++i) {
              const float4 t = p.tgt[i];
              const float dx = qx - t.x, dy = qy - t.y, dz = qz - t.z;
              const float d2 = dx * dx + dy * dy + dz * dz;
              const int id = __float_as_int(t.w);
              if (d2 < best || (d2 == best && id < best_id)) { best = d2; best_id = id; }
            }
          }
        }
      }
  }
  if (best_id < 0) best_id = 0;
}

__device__ void jacobi4(double A[4][4], double V[4][4]) {
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) V[i][j] = (i == j);
  double scale = 0;
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) scale += A[i][j] * A[i][j];
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0;
    for (int i = 0; i < 4; ++i) for (int j = i + 1; j < 4; ++j) off += A[i][j] * A[i][j];
    // converged to double precision: the off-diagonal mass is below eps^2 of the matrix (Jacobi converges quadratically, so the
    // sweep that gets here has already over-shot; running on to 1e-300 costs five more sweeps for nothing)
    if (off <= 1e-34 * scale || off < 1e-300) break;
    for (int p = 0; p < 4; ++p)
      for (int q = p + 1; q < 4; ++q) {
        if (fabs(A[p][q]) < 1e-300) continue;
        const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
        for (int k = 0; k < 4; ++k) { const double akp = A[k][p], akq = A[k][q]; A[k][p] = cs * akp - sn * akq; A[k][q] = sn * akp + cs * akq; }
        for (int k = 0; k < 4; ++k) { const double apk = A[p][k], aqk = A[q][k]; A[p][k] = cs * apk - sn * aqk; A[q][k] = sn * apk + cs * aqk; }
        for (int k = 0; k < 4; ++k) { const double vkp = V[k][p], vkq = V[k][q]; V[k][p] = cs * vkp - sn * vkq; V[k][q] = sn * vkp + cs * vkq; }
      }
  }
}

// Largest eigenpair of the symmetric, traceless 4x4 matrix of Horn's quaternion fit without an iterative diagonalisation: the
// characteristic polynomial x^4 + c2 x^2 + c1 x + c0 of N / |N|_F from traces of powers (Faddeev-LeVerrier), Newton from x = 1 >=
// lambda_max (monotone: every root is real and the polynomial is convex to the right of the largest), eigenvector = the column of
// adj(N - lambda I) with the largest diagonal cofactor (rank 3 => adj = c q q^T).  Returns false when the largest eigenvalue is
// (nearly) double -- the fit is then ill-posed and the caller diagonalises with Jacobi instead.
__host__ __device__ bool max_eigvec4(const double N[4][4], double q[4]) {
  double f2 = 0;
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) f2 += N[i][j] * N[i][j];
  if (!(f2 > 1e-280) || !(f2 < 1e280)) return false;
  const double inv = 1.0 / sqrt(f2);
  double A[4][4], M2[4][4];
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) A[i][j] = N[i][j] * inv;
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) { double s = 0; for (int k = 0; k < 4; ++k) s += A[i][k] * A[k][j]; M2[i][j] = s; }
  double t1 = 0, t2 = 0, t3 = 0, t4 = 0;
  for (int i = 0; i < 4; ++i) { t1 += A[i][i]; t2 += M2[i][i]; for (int j = 0; j < 4; ++j) { t3 += M2[i][j] * A[i][j]; t4 += M2[i][j] * M2[i][j]; } }
  // Faddeev-LeVerrier, general trace (t1 is rounding-sized here but costs nothing to carry)
  const double c3 = -t1, c2 = -0.5 * (t2 + c3 * t1), c1 = -(t3 + c3 * t2 + c2 * t1) / 3.0, c0 = -0.25 * (t4 + c3 * t3 + c2 * t2 + c1 * t1);
  double x = 1.0 + 1e-12;
  for (int it = 0; it < 100; ++it) {
    const double P = (((x + c3) * x + c2) * x + c1) * x + c0, dP = ((4.0 * x + 3.0 * c3) * x + 2.0 * c2) * x + c1;
    if (!(dP > 0)) return false;
    const double d = P / dP;
    x -= d;
    if (fabs(d) < 1e-15) break;
  }
  for (int i = 0; i < 4; ++i) A[i][i] -= x;
  auto minor3 = [&](int i, int j) {
    int r[3], c[3];
    for (int k = 0, n = 0; k < 4; ++k) if (k != i) r[n++] = k;
    for (int k = 0, n = 0; k < 4; ++k) if (k != j) c[n++] = k;
    return A[r[0]][c[0]] * (A[r[1]][c[1]] * A[r[2]][c[2]] - A[r[1]][c[2]] * A[r[2]][c[1]]) -
           A[r[0]][c[1]] * (A[r[1]][c[0]] * A[r[2]][c[2]] - A[r[1]][c[2]] * A[r[2]][c[0]]) +
           A[r[0]][c[2]] * (A[r[1]][c[0]] * A[r[2]][c[1]] - A[r[1]][c[1]] * A[r[2]][c[0]]);
  };
  int jb = 0;
  double cb = 0;
  for (int j = 0; j < 4; ++j) { const double c = fabs(minor3(j, j)); if (c > cb) { cb = c; jb = j; } }
  if (!(cb > 1e-7)) return false;
  for (int i = 0; i < 4; ++i) q[i] = (((i + jb) & 1) ? -1.0 : 1.0) * minor3(i, jb);
  return true;
}

// R, t minimising sum |R s + t - g|^2 from n, sum s, sum g, sum s g^T
__device__ void rigid_fit(double n, const double* S, float* T) {
  double cs[3] = {S[0] / n, S[1] / n, S[2] / n}, cg[3] = {S[3] / n, S[4] / n, S[5] / n};
  double H[3][3];
  for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) H[a][b] = S[6 + 3 * a + b] - n * cs[a] * cg[b];
  const double Sxx = H[0][0], Sxy = H[0][1], Sxz = H[0][2], Syx = H[1][0], Syy = H[1][1], Syz = H[1][2], Szx = H[2][0], Szy = H[2][1], Szz = H[2][2];
  double N[4][4] = {{Sxx + Syy + Szz, Syz - Szy, Szx - Sxz, Sxy - Syx},
                    {Syz - Szy, Sxx - Syy - Szz, Sxy + Syx, Szx + Sxz},
                    {Szx - Sxz, Sxy + Syx, -Sxx + Syy - Szz, Syz + Szy},
                    {Sxy - Syx, Szx + Sxz, Syz + Szy, -Sxx - Syy + Szz}};
  // (one thread runs this while the CTA waits: the Jacobi sweeps -- double divisions and square roots in a dependent chain -- were a
  // fifth of the kernel's time; the closed form needs ~15 divisions in all)
  double q4[4];
  if (!max_eigvec4(N, q4)) {
    double V[4][4];
    jacobi4(N, V);
    int best = 0;
    for (int k = 1; k < 4; ++k) if (N[k][k] > N[best][best]) best = k;
    for (int k = 0; k < 4; ++k) q4[k] = V[k][best];
  }
  double qw = q4[0], qx = q4[1], qy = q4[2], qz = q4[3];
  const double nrm = sqrt(qw * qw + qx * qx + qy * qy + qz * qz);
  qw /= nrm; qx /= nrm; qy /= nrm; qz /= nrm;
  const double R[3][3] = {{1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw)},
                          {2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw)},
                          {2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)}};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) T[4 * i + j] = (float)R[i][j];
    T[4 * i + 3] = (float)(cg[i] - (R[i][0] * cs[0] + R[i][1] * cs[1] + R[i][2] * cs[2]));
  }
}

// Two CTAs (one thread-block cluster) per pose: CTA r owns the source points [r * ceil(ns / 2), ...) -- their correspondences, their
// share of the radix-select histograms and of the 16 sums.  The halves meet through distributed shared memory: after a cluster
// barrier each CTA adds the partner's histogram (or partial sums) to its own IN THE SAME ORDER, so both take identical decisions
// and carry identical transforms -- nothing is broadcast, and the serial fit runs redundantly on both.  64 poses then fill 128 of
// the 148 SMs and the per-iteration critical path (the slowest pose decides the kernel's time) halves.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TT, 1) k5_tricp_kernel(const TricpParams p) {
  namespace cg = cooperative_groups;
  cg::cluster_group cl = cg::this_cluster();
  __shared__ float sT[12];
  __shared__ uint32_t s_hist[2][256];    // double-buffered by pass parity: the partner may still read pass p while pass p+1 fills
  __shared__ uint32_t s_sel[4];          // prefix, remaining rank, CTA 0's count of values equal to tau
  __shared__ uint32_t s_warp[TT / 32];
  __shared__ double s_red[TT / 32][16];
  __shared__ double s_part[16];
  __shared__ int s_cont;
  const unsigned cr = cl.block_rank();
  const uint32_t* r_hist = cl.map_shared_rank(&s_hist[0][0], cr ^ 1u);
  const double* r_part = cl.map_shared_rank(&s_part[0], cr ^ 1u);
  const int pose = blockIdx.x >> 1, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int half = (p.ns + 1) >> 1;
  const int i_lo = cr ? half : 0, i_hi = cr ? p.ns : half;
  float* d2 = p.d2 + (size_t)pose * p.ns;
  int* nn = p.nn + (size_t)pose * p.ns;
  if (tid < 12) sT[tid] = p.T[12 * pose + tid];
  __syncthreads();
  float energy = FLT_MAX, old_energy = FLT_MAX;
  int it = 0;
  // Search radius of the next iteration: 4 x the squared trim radius of the previous one.  Source points that are far from the
  // model (the half the trim drops; clutter) otherwise dominate the iteration -- their ring searches sweep hundreds of cells for a
  // distance that is thrown away.  If the n_keep-th smallest distance found under the cap is not below it, the cap cut into the
  // kept set: the correspondences are searched again without a cap, so the kept set and its sums are always the exact ones.
  float cap2 = FLT_MAX;
  for (;;) {
    // 1. correspondences of this CTA's half
    for (int i = i_lo + tid; i < i_hi; i += TT) {
      const float4 s = p.src[i];
      const float qx = sT[0] * s.x + sT[1] * s.y + sT[2] * s.z + sT[3];
      const float qy = sT[4] * s.x + sT[5] * s.y + sT[6] * s.z + sT[7];
      const float qz = sT[8] * s.x + sT[9] * s.y + sT[10] * s.z + sT[11];
      float best; int id;
      nn_search(p, qx, qy, qz, cap2, best, id);
      d2[i] = best; nn[i] = id;
    }
    // 2. n_keep-th smallest squared distance over BOTH halves: MSB-first radix select on the float bits (d2 >= 0)
    uint32_t prefix = 0, rank = (uint32_t)p.n_keep;     // 1-based rank inside the current bucket
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      uint32_t* hist = s_hist[pass & 1];
      if (tid < 256) hist[tid] = 0;
      __syncthreads();                                   // (also orders this thread block's d2 writes before its reads)
      for (int i = i_lo + tid; i < i_hi; i += TT) {
        const uint32_t b = __float_as_uint(d2[i]);
        if (pass == 0 || (b >> (shift + 8)) == prefix) atomicAdd(&hist[(b >> shift) & 255u], 1u);
      }
      cl.sync();
      if (warp == 0) {
        // first digit whose inclusive prefix count reaches the rank: 8 bins per lane, warp scan of the lane sums
        const uint32_t* rh = r_hist + (pass & 1) * 256;
        uint32_t h[8], h0[8], mine = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint32_t a = hist[lane * 8 + k], b = rh[lane * 8 + k];
          h[k] = a + b; h0[k] = cr ? b : a; mine += h[k];
        }
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        const unsigned hit = __ballot_sync(0xffffffffu, incl >= rank);
        const int l = hit ? __ffs(hit) - 1 : 31;
        if (lane == l) {
          uint32_t acc = incl - mine; int dgt = 0;
          for (; dgt < 7; ++dgt) { if (acc + h[dgt] >= rank) break; acc += h[dgt]; }
          s_sel[0] = (prefix << 8) | (uint32_t)(lane * 8 + dgt); s_sel[1] = rank - acc;
          uint32_t e0 = h0[0], et = h[0];
#pragma unroll
          for (int k = 1; k < 8; ++k) if (k == dgt) { e0 = h0[k]; et = h[k]; }
          s_sel[2] = e0;                                 // last pass: how many values equal to tau CTA 0 holds,
          s_sel[3] = et;                                 // and how many there are in all
        }
      }
      __syncthreads();
      prefix = s_sel[0]; rank = s_sel[1];
      __syncthreads();
    }
    const uint32_t tau = prefix;          // bits of the n_keep-th smallest d2; `rank` of the equal ones are kept, lowest source index first
    if (cap2 != FLT_MAX && !(__uint_as_float(tau) < cap2)) { cap2 = FLT_MAX; continue; }      // (uniform over the cluster: both CTAs formed the same tau)
    cap2 = fmaxf(4.0f * __uint_as_float(tau), 1e-12f);
    // 3. sums over the kept correspondences (equal-to-tau ones admitted in index order: CTA 0 holds the lower indices)
    double acc[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) acc[k] = 0.0;
    uint32_t eq_seen = cr ? s_sel[2] : 0u;
    const bool all_eq = s_sel[3] == rank;          // every value equal to tau is kept (the usual case: tau is unique): no ordering needed
    for (int i0 = i_lo; i0 < i_hi; i0 += TT) {
      const int i = i0 + tid;
      const uint32_t b = i < i_hi ? __float_as_uint(d2[i]) : 0xffffffffu;
      const bool eq = i < i_hi && b == tau;
      uint32_t before = 0, total = 0;
      if (!all_eq) {                                 // (uniform over the cluster)
        const unsigned bal = __ballot_sync(0xffffffffu, eq);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        before = eq_seen;
        for (int w = 0; w < TT / 32; ++w) { const uint32_t c = s_warp[w]; if (w < warp) before += c; total += c; }
        before += __popc(bal & ((1u << lane) - 1u));
      }
      const bool keep = i < i_hi && (b < tau || (eq && (all_eq || before < rank)));
      if (keep) {
        const float4 s = p.src[i];
        const float4 g = p.tgt_orig[nn[i]];
        acc[0] += (double)d2[i];
        acc[1] += s.x; acc[2] += s.y; acc[3] += s.z;
        acc[4] += g.x; acc[5] += g.y; acc[6] += g.z;
        acc[7] += (double)s.x * g.x; acc[8] += (double)s.x * g.y; acc[9] += (double)s.x * g.z;
        acc[10] += (double)s.y * g.x; acc[11] += (double)s.y * g.y; acc[12] += (double)s.y * g.z;
        acc[13] += (double)s.z * g.x; acc[14] += (double)s.z * g.y; acc[15] += (double)s.z * g.z;
      }
      eq_seen += total;
      if (!all_eq) __syncthreads();
    }
    // 16 sums over the warp with 16 shuffles instead of 80: at every butterfly step a lane hands HALF of its partial sums to its
    // partner and keeps the other half, so the values per lane halve while the lanes per value double; lane l ends with the
    // complete sum number (bits 4..1 of l)
#pragma unroll
    for (int half = 8, off = 16; half >= 1; half >>= 1, off >>= 1) {
      const bool upper = (lane & off) != 0;
#pragma unroll
      for (int j = 0; j < half; ++j) {
        const double send = upper ? acc[j] : acc[j + half];
        const double keep = upper ? acc[j + half] : acc[j];
        acc[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
    acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 1);
    if (!(lane & 1)) s_red[warp][((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1)] = acc[0];
    __syncthreads();
    if (tid < 16) { double v = 0; for (int w = 0; w < TT / 32; ++w) v += s_red[w][tid]; s_part[tid] = v; }
    cl.sync();
    if (tid == 0) {
      double S[16];
      for (int k = 0; k < 16; ++k) S[k] = cr ? r_part[k] + s_part[k] : s_part[k] + r_part[k];      // CTA 0's half + CTA 1's half, in both
      old_energy = energy;
      energy = (float)S[0];
      if (energy <= FLT_MAX) {                     // a kept squared distance overflowed: no fit, and the ratio test below stops
        float Tn[12];
        rigid_fit((double)p.n_keep, S + 1, Tn);
        for (int k = 0; k < 12; ++k) sT[k] = Tn[k];
      }
      ++it;
      s_cont = ((energy / old_energy) < p.ratio && it < p.max_iter) ? 1 : 0;
    }
    __syncthreads();
    if (!s_cont) break;
  }
  if (cr == 0) {
    if (tid < 12) p.T[12 * pose + tid] = sT[tid];
    if (tid == 0) { if (p.iters) p.iters[pose] = it; if (p.energy) p.energy[pose] = energy; }
  }
  cl.sync();                                             // the partner may still be reading this CTA's shared memory
}

// device scratch of the refinement: owned by the context (two contexts on one device must not share it), created on first
// use, released by k5_release (pgp_destroy)
struct TScratch { DevBuf seg, d2, nn, T, iters, energy, cell_of, cursor; };
TScratch& tscratch_of(pgp_ctx* ctx) {
  if (!ctx->k5_scratch) ctx->k5_scratch = new TScratch();
  return *static_cast<TScratch*>(ctx->k5_scratch);
}

// model-space grid over the raw validation cloud (the TrICP target)
int build_target_grid(pgp_ctx* ctx, Model& m) {
  if (m.tgrid_ready) return PGP_OK;
  TScratch& ts = tscratch_of(ctx);
  const int n = m.nv;
  TGrid tg;
  float ext = 0.f;
  for (int k = 0; k < 3; ++k) ext = std::max(ext, m.val_raw_hi[k] - m.val_raw_lo[k]);
  // cell edge: the model is a SURFACE, so ~n of the cells^3 cells are occupied when cells ~ 2 cbrt(n) (about one point per occupied
  // cell: the 27-cell ring of a query near the surface then holds ~8 points instead of ~32 at cells = cbrt(n))
  const int cells = std::max(1, std::min(96, (int)std::ceil(2.0 * std::cbrt((double)n))));
  tg.g = std::max(ext / (float)cells, 1e-6f);
  tg.inv_g = 1.0f / tg.g;
  for (int k = 0; k < 3; ++k) {
    tg.lo[k] = m.val_raw_lo[k];
    tg.dim[k] = std::max(1, (int)std::floor((m.val_raw_hi[k] - m.val_raw_lo[k]) * tg.inv_g) + 1);
  }
  const size_t nc = (size_t)tg.dim[0] * tg.dim[1] * tg.dim[2];
  PGP_CUDA(ctx, m.tgrid_start.reserve((nc + 1) * 4));
  PGP_CUDA(ctx, m.tgrid_pts.reserve((size_t)n * 16));
  PGP_CUDA(ctx, ts.cell_of.reserve((size_t)n * 4));
  PGP_CUDA(ctx, ts.cursor.reserve((nc + 1) * 4));
  PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((nc + 1) / 2048 + 4096) * 4));
  uint32_t* st = m.tgrid_start.as<uint32_t>();
  PGP_CUDA(ctx, cudaMemsetAsync(st, 0, (nc + 1) * 4, ctx->stream));
  k5_tgrid_count<<<(n + 255) / 256, 256, 0, ctx->stream>>>(m.val_raw.as<float4>(), n, tg, ts.cell_of.as<uint32_t>(), st);
  ctx->launches++;
  int rc = pgp_scan_exclusive_u32(ctx, st, (int64_t)nc + 1, ctx->scene.scratch.as<uint32_t>());
  if (rc) return rc;
  PGP_CUDA(ctx, cudaMemcpyAsync(ts.cursor.p, st, (nc + 1) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  k5_tgrid_scatter<<<(n + 255) / 256, 256, 0, ctx->stream>>>(m.val_raw.as<float4>(), n, ts.cell_of.as<uint32_t>(), ts.cursor.as<uint32_t>(),
                                                            m.tgrid_pts.as<float4>());
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  memcpy(&m.tg_lo, tg.lo, 12); m.tg_g = tg.g; memcpy(m.tg_dim, tg.dim, 12);
  m.tgrid_ready = true;
  return PGP_OK;
}

// general 4x4 rigid inverse in double: [R t]^-1 = [R^T, -R^T t]
void invert_pose(const double* P, double* I) {
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) I[4 * r + c] = P[4 * c + r];
    I[4 * r + 3] = -(P[0 * 4 + r] * P[3] + P[1 * 4 + r] * P[7] + P[2 * 4 + r] * P[11]);
  }
  I[12] = I[13] = I[14] = 0; I[15] = 1;
}

}  // namespace

// host-callable copy of max_eigvec4 for the CPU test-suite (tests/test_host_arithmetic.py): N16 row-major symmetric 4x4; returns 1
// and the (unnormalised) eigenvector of the largest eigenvalue, or 0 when the kernel would fall back to Jacobi
extern "C" PGP_API int pgp_host_max_eigvec4(const double* N16, double* q4) {
  double N[4][4];
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) N[i][j] = N16[4 * i + j];
  return max_eigvec4(N, q4) ? 1 : 0;
}


int k5_tricp(pgp_ctx* ctx, Model& m, const float* seg_xyz_host, int ns, double* poses16_host, int k, float trim, float ratio, int max_iter,
             int* iters_out, float* energy_out) {
  TScratch& ts = tscratch_of(ctx);
  int rc = build_target_grid(ctx, m);
  if (rc) return rc;
  const float keep_f = fabsf(trim * (float)ns);                          // abs(numPoints) on a float, UCTState.cpp:181,194
  const int n_keep = keep_f < 2147483648.f ? std::min(ns, (int)keep_f) : ns;
  if (n_keep < 3) {
    for (int i = 0; i < k; ++i) { if (iters_out) iters_out[i] = 0; if (energy_out) energy_out[i] = 0.f; }
    return PGP_OK;
  }
  // The source cloud goes up in Morton order of its own bounding box: a rigid transform keeps neighbours together, so the 32
  // queries of a warp walk the same few grid rows of the target in every iteration of every pose (the ring searches of unrelated
  // points diverge: 4 of 32 lanes were active in the distance loop).  Sums are order-free up to double rounding; ties at the trim
  // threshold are admitted in this order.
  std::vector<float> seg4((size_t)ns * 4, 0.f), T((size_t)k * 12);
  {
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = 0; i < ns; ++i) for (int c = 0; c < 3; ++c) { lo[c] = std::min(lo[c], seg_xyz_host[3 * i + c]); hi[c] = std::max(hi[c], seg_xyz_host[3 * i + c]); }
    const float ext = std::max(std::max(hi[0] - lo[0], hi[1] - lo[1]), std::max(hi[2] - lo[2], 1e-12f));
    auto spread = [](uint32_t v) { uint64_t x = v & 0x1fffffu; x = (x | x << 32) & 0x1f00000000ffffull; x = (x | x << 16) & 0x1f0000ff0000ffull;
                                   x = (x | x << 8) & 0x100f00f00f00f00full; x = (x | x << 4) & 0x10c30c30c30c30c3ull; x = (x | x << 2) & 0x1249249249249249ull; return x; };
    std::vector<std::pair<uint64_t, int>> key((size_t)ns);
    for (int i = 0; i < ns; ++i) {
      uint64_t m = 0;
      for (int c = 0; c < 3; ++c) {
        const float u = (seg_xyz_host[3 * i + c] - lo[c]) / ext;
        const uint32_t q = (uint32_t)std::min(1023.0f, std::max(0.0f, u * 1024.0f));     // (NaN -> 0)
        m |= spread(q) << c;
      }
      key[(size_t)i] = std::make_pair(m, i);
    }
    std::sort(key.begin(), key.end());
    for (int i = 0; i < ns; ++i) for (int c = 0; c < 3; ++c) seg4[4 * (size_t)i + c] = seg_xyz_host[3 * key[(size_t)i].second + c];
  }
  for (int i = 0; i < k; ++i) {
    double inv[16];
    invert_pose(poses16_host + 16 * i, inv);                            // tform = inverse(object pose), UCTState.cpp:184-185
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) T[12 * (size_t)i + 4 * r + c] = (float)inv[4 * r + c];
  }
  PGP_CUDA(ctx, ts.seg.reserve((size_t)ns * 16));
  PGP_CUDA(ctx, ts.d2.reserve((size_t)k * ns * 4));
  PGP_CUDA(ctx, ts.nn.reserve((size_t)k * ns * 4));
  PGP_CUDA(ctx, ts.T.reserve((size_t)k * 48));
  PGP_CUDA(ctx, ts.iters.reserve((size_t)k * 4));
  PGP_CUDA(ctx, ts.energy.reserve((size_t)k * 4));
  PGP_CUDA(ctx, cudaMemcpyAsync(ts.seg.p, seg4.data(), (size_t)ns * 16, cudaMemcpyHostToDevice, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(ts.T.p, T.data(), (size_t)k * 48, cudaMemcpyHostToDevice, ctx->stream));
  TricpParams p{};
  p.src = ts.seg.as<float4>(); p.ns = ns;
  p.tgt = m.tgrid_pts.as<float4>(); p.tstart = m.tgrid_start.as<uint32_t>(); p.nt = m.nv; p.tgt_orig = m.val_raw.as<float4>();
  memcpy(p.tg.lo, m.tg_lo, 12); p.tg.g = m.tg_g; p.tg.inv_g = 1.0f / m.tg_g; memcpy(p.tg.dim, m.tg_dim, 12);
  p.d2 = ts.d2.as<float>(); p.nn = ts.nn.as<int>(); p.T = ts.T.as<float>();
  p.n_keep = n_keep; p.ratio = ratio; p.max_iter = std::max(1, max_iter);
  p.iters = ts.iters.as<int>(); p.energy = ts.energy.as<float>();
  k5_tricp_kernel<<<2 * k, TT, 0, ctx->stream>>>(p);      // one cluster of two CTAs per pose
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  PGP_CUDA(ctx, cudaMemcpyAsync(T.data(), ts.T.p, (size_t)k * 48, cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<int> it(k);
  std::vector<float> en(k);
  PGP_CUDA(ctx, cudaMemcpyAsync(it.data(), ts.iters.p, (size_t)k * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(en.data(), ts.energy.p, (size_t)k * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < k; ++i) {
    if (en[i] <= FLT_MAX) {                                              // (non-finite energy: the pose stays as it was given)
      double M[16] = {0}, inv[16];
      for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) M[4 * r + c] = (double)T[12 * (size_t)i + 4 * r + c];
      M[15] = 1;
      invert_pose(M, inv);                                               // pose = inverse(tform), UCTState.cpp:195-203
      memcpy(poses16_host + 16 * i, inv, sizeof(inv));
    }
    if (iters_out) iters_out[i] = it[i];
    if (energy_out) energy_out[i] = en[i];
  }
  return PGP_OK;
}

void k5_release(pgp_ctx* ctx) {
  if (!ctx->k5_scratch) return;
  TScratch* ts = static_cast<TScratch*>(ctx->k5_scratch);
  for (DevBuf* b : {&ts->seg, &ts->d2, &ts->nn, &ts->T, &ts->iters, &ts->energy, &ts->cell_of, &ts->cursor}) b->release();
  delete ts;
  ctx->k5_scratch = nullptr;
}
