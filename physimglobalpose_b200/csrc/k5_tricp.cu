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
// pgp_tricp_plane (utilities::pointToPlaneICP, utilities.cpp:709-739) runs the same kernel with the point-to-plane fit instead:
// 28 double sums in two passes, a 6x6 truncated pseudo-inverse solve, and PCL's Rz Ry Rx update (restated, parity unpinned).
#include <cooperative_groups.h>
#include <float.h>
#include <math.h>

#include <algorithm>
#include <type_traits>
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
  const float4* nrm_orig;        // unit normals of tgt_orig, same order (point-to-plane fit)
};

// One item of a batched refinement (pgp_refine_batch): its own TricpParams -- source, target grid, n_keep, d2 / nn rows; T, iters
// and energy point at its first pose -- and where its poses start in the launch.
struct K5Item {
  TricpParams p;
  int pose_lo;
};
struct K5Batch { const K5Item* items; const int* pose_item; };   // pose_item: launch pose -> item
template <bool BATCH> using K5Args = std::conditional_t<BATCH, K5Batch, TricpParams>;

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

// x = H^+ g for the 6x6 normal equations of the point-to-plane fit (symmetric positive semi-definite H, row-major): Jacobi scaling
// s_j = 1 / sqrt(H_jj) (0 where H_jj <= 0), M = S H S = V diag(lambda) V^T by cyclic Jacobi in double (rows p < q in order; stop
// when the off-diagonal norm is <= 1e-15 |M|_F, or after 30 sweeps), every lambda <= 1e-9 lambda_max dropped (all of them when
// lambda_max <= 0), x = S V diag(lambda^+) V^T S g.  The truncation gives the minimum-norm update when the kept points leave
// directions free (one face of a box: rank 3).  Returns the number of eigenvalues kept.
#ifdef __CUDA_ARCH__
#define K5_ROLLED _Pragma("unroll 1")      // one thread runs this: keep M and V in local memory rather than spill an unrolled copy
#else
#define K5_ROLLED
#endif
__host__ __device__ int solve_plane6(const double H[36], const double g[6], double x[6]) {
  double s[6], M[6][6], V[6][6];
  for (int j = 0; j < 6; ++j) s[j] = H[7 * j] > 0.0 ? 1.0 / sqrt(H[7 * j]) : 0.0;
  double f2 = 0.0;
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 6; ++j) { M[i][j] = (s[i] * H[6 * i + j]) * s[j]; V[i][j] = (i == j); f2 += M[i][j] * M[i][j]; }
  K5_ROLLED
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0;
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) if (i != j) off += M[i][j] * M[i][j];
    if (!(off > 1e-30 * f2)) break;
    K5_ROLLED
    for (int p = 0; p < 6; ++p)
      K5_ROLLED
      for (int q = p + 1; q < 6; ++q) {
        if (M[p][q] == 0.0) continue;
        const double theta = (M[q][q] - M[p][p]) / (2.0 * M[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
        for (int k = 0; k < 6; ++k) { const double mkp = M[k][p], mkq = M[k][q]; M[k][p] = cs * mkp - sn * mkq; M[k][q] = sn * mkp + cs * mkq; }
        for (int k = 0; k < 6; ++k) { const double mpk = M[p][k], mqk = M[q][k]; M[p][k] = cs * mpk - sn * mqk; M[q][k] = sn * mpk + cs * mqk; }
        for (int k = 0; k < 6; ++k) { const double vkp = V[k][p], vkq = V[k][q]; V[k][p] = cs * vkp - sn * vkq; V[k][q] = sn * vkp + cs * vkq; }
      }
  }
  double lmax = M[0][0];
  for (int k = 1; k < 6; ++k) lmax = fmax(lmax, M[k][k]);
  double w[6];
  int rank = 0;
  for (int k = 0; k < 6; ++k) {
    double u = 0.0;
    for (int i = 0; i < 6; ++i) u += V[i][k] * (s[i] * g[i]);
    const bool keep = lmax > 0.0 && M[k][k] > 1e-9 * lmax;
    w[k] = keep ? u / M[k][k] : 0.0;
    rank += keep;
  }
  for (int i = 0; i < 6; ++i) {
    double v = 0.0;
    for (int k = 0; k < 6; ++k) v += V[i][k] * w[k];
    x[i] = s[i] * v;
  }
  return rank;
}

// dR = Rz(gamma) Ry(beta) Rx(alpha) from x = (alpha, beta, gamma, ...): the construction of PCL's
// TransformationEstimationPointToPlaneLLS as recalled (not vendored: restated, parity unpinned), in this association.
__host__ __device__ void euler_zyx(const double x[3], double R[3][3]) {
  const double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
  R[0][0] = cg * cb; R[0][1] = -sg * ca + (cg * sb) * sa; R[0][2] = sg * sa + (cg * sb) * ca;
  R[1][0] = sg * cb; R[1][1] = cg * ca + (sg * sb) * sa;  R[1][2] = -cg * sa + (sg * sb) * ca;
  R[2][0] = -sb;     R[2][1] = cb * sa;                   R[2][2] = cb * ca;
}

// One Gauss-Newton step of the point-to-plane fit from the 28 sums S = {E, sum a r (6), H upper triangle row by row (21)}:
// x = H^+ g with g = -sum a r, T <- fp32(dR R_T, ((dR_0 t_T + dR_1 t_T) + dR_2 t_T) + dt) in double from the fp32 T.
// (one copy per kernel instance: a callee shared by the single and the batched kernel is register-allocated for both)
template <bool BATCH>
__device__ __noinline__ void plane_fit(const double* S, float* T) {
  double H[36], g[6], x[6], R[3][3];
  for (int i = 0, k = 7; i < 6; ++i)
    for (int j = i; j < 6; ++j, ++k) H[6 * i + j] = H[6 * j + i] = S[k];
  for (int j = 0; j < 6; ++j) g[j] = -S[1 + j];
  solve_plane6(H, g, x);
  euler_zyx(x, R);
  float Tn[12];
  for (int i = 0; i < 3; ++i)
    for (int c = 0; c < 4; ++c) {
      const double v = (R[i][0] * (double)T[c] + R[i][1] * (double)T[4 + c]) + R[i][2] * (double)T[8 + c];
      Tn[4 * i + c] = (float)(c == 3 ? v + x[3 + i] : v);
    }
  for (int k = 0; k < 12; ++k) T[k] = Tn[k];
}

// Sums over the kept correspondences of this CTA's half into acc[16]: d2 below tau, and the values equal to tau admitted in source
// order (CTA 0 holds the lower indices) until `rank` of them are in.  term(i, acc) adds point i's contributions.
template <class Term>
__device__ __forceinline__ void kept_sums(const float* d2, int i_lo, int i_hi, uint32_t tau, uint32_t rank, uint32_t eq_seen, bool all_eq,
                                          uint32_t* s_warp, int tid, int lane, int warp, double acc[16], Term term) {
#pragma unroll
  for (int k = 0; k < 16; ++k) acc[k] = 0.0;
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
    if (keep) term(i, acc);
    eq_seen += total;
    if (!all_eq) __syncthreads();
  }
}

// Block sum of acc[16] into out[16] (thread 0..15 write), in a fixed order: lanes by the butterfly below, warps in order.
__device__ __forceinline__ void block_sum16(double acc[16], double (*s_red)[16], double* out, int tid, int lane, int warp) {
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
  if (tid < 16) { double v = 0; for (int w = 0; w < TT / 32; ++w) v += s_red[w][tid]; out[tid] = v; }
}

// Point-to-plane sums of kept point i, pass PASS of two: entries [16 PASS, 16 PASS + 16) of
// {r^2, a r (6), a_j a_k for j <= k row by row (21), 0 (4)} with a = [p' x n, n], r = n . (p' - q), all in double.
template <int PASS>
__device__ __forceinline__ void plane_terms(const TricpParams& p, const float* sT, const int* nn, int i, double acc[16]) {
  const float4 s = p.src[i];
  const float qx = sT[0] * s.x + sT[1] * s.y + sT[2] * s.z + sT[3];
  const float qy = sT[4] * s.x + sT[5] * s.y + sT[6] * s.z + sT[7];
  const float qz = sT[8] * s.x + sT[9] * s.y + sT[10] * s.z + sT[11];
  const float4 n = p.nrm_orig[nn[i]];
  const double px = qx, py = qy, pz = qz, nx = n.x, ny = n.y, nz = n.z;
  const double a[6] = {py * nz - pz * ny, pz * nx - px * nz, px * ny - py * nx, nx, ny, nz};
  double v[32];
  if (PASS == 0) {
    const float4 g = p.tgt_orig[nn[i]];
    const double r = ((px - (double)g.x) * nx + (py - (double)g.y) * ny) + (pz - (double)g.z) * nz;
    v[0] = r * r;
#pragma unroll
    for (int j = 0; j < 6; ++j) v[1 + j] = a[j] * r;
  }
#pragma unroll
  for (int j = 0, k = 7; j < 6; ++j)
#pragma unroll
    for (int l = j; l < 6; ++l, ++k) v[k] = a[j] * a[l];
#pragma unroll
  for (int k = 0; k < 16; ++k)
    if (16 * PASS + k < 28) acc[k] += v[16 * PASS + k];
}

// Two CTAs (one thread-block cluster) per pose: CTA r owns the source points [r * ceil(ns / 2), ...) -- their correspondences, their
// share of the radix-select histograms and of the sums.  The halves meet through distributed shared memory: after a cluster
// barrier each CTA adds the partner's histogram (or partial sums) to its own IN THE SAME ORDER, so both take identical decisions
// and carry identical transforms -- nothing is broadcast, and the serial fit runs redundantly on both.  64 poses then fill 128 of
// the 148 SMs and the per-iteration critical path (the slowest pose decides the kernel's time) halves.
// PLANE = false: the point-to-point fit (16 sums, Horn).  PLANE = true: the point-to-plane fit; its 28 sums do not fit the
// 64-register budget of a 1024-thread CTA next to the search, so they take two passes of 16 over the kept set (the second one
// 12 sums and 4 zeros), each through the same butterfly into its own half of s_part.
// BATCH = false: one item, its TricpParams in the kernel arguments.  BATCH = true (pgp_refine_batch): many items in one launch;
// each cluster copies its item's K5Item into shared memory and runs the same code on it -- or returns at once when the item has
// n_keep < 3 (set so by k5_prep_items, or left at 0 by a refused call), before any cluster barrier: both CTAs read the same
// descriptor, so the pair leaves together and neither touches the other's shared memory.
template <bool PLANE, bool BATCH = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TT, 1) k5_tricp_kernel(const K5Args<BATCH> a) {
  namespace cg = cooperative_groups;
  cg::cluster_group cl = cg::this_cluster();
  constexpr int NS = PLANE ? 32 : 16;    // sums exchanged between the CTAs
  __shared__ K5Item s_item;
  if constexpr (BATCH) {
    static_assert(sizeof(K5Item) % 4 == 0 && sizeof(K5Item) / 4 <= TT, "K5Item is copied one word per thread");
    const K5Item* src = a.items + a.pose_item[blockIdx.x >> 1];
    if (threadIdx.x < sizeof(K5Item) / 4) reinterpret_cast<int*>(&s_item)[threadIdx.x] = reinterpret_cast<const int*>(src)[threadIdx.x];
    __syncthreads();
    if (s_item.p.n_keep < 3) return;
  }
  const TricpParams* pp;
  if constexpr (BATCH) pp = &s_item.p; else pp = &a;
  const TricpParams& p = *pp;
  const int pose = BATCH ? (int)(blockIdx.x >> 1) - s_item.pose_lo : (int)(blockIdx.x >> 1);
  __shared__ float sT[12];
  __shared__ uint32_t s_hist[2][256];    // double-buffered by pass parity: the partner may still read pass p while pass p+1 fills
  __shared__ uint32_t s_sel[4];          // prefix, remaining rank, CTA 0's count of values equal to tau
  __shared__ uint32_t s_warp[TT / 32];
  __shared__ double s_red[TT / 32][16];
  __shared__ double s_part[NS];
  __shared__ int s_cont;
  const unsigned cr = cl.block_rank();
  const uint32_t* r_hist = cl.map_shared_rank(&s_hist[0][0], cr ^ 1u);
  const double* r_part = cl.map_shared_rank(&s_part[0], cr ^ 1u);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
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
    const uint32_t eq_seen = cr ? s_sel[2] : 0u;
    const bool all_eq = s_sel[3] == rank;          // every value equal to tau is kept (the usual case: tau is unique): no ordering needed
    if constexpr (PLANE) {
      kept_sums(d2, i_lo, i_hi, tau, rank, eq_seen, all_eq, s_warp, tid, lane, warp, acc,
                [&](int i, double* a) { plane_terms<0>(p, sT, nn, i, a); });
      block_sum16(acc, s_red, s_part, tid, lane, warp);
      __syncthreads();                             // s_red is refilled by the second pass
      kept_sums(d2, i_lo, i_hi, tau, rank, eq_seen, all_eq, s_warp, tid, lane, warp, acc,
                [&](int i, double* a) { plane_terms<1>(p, sT, nn, i, a); });
      block_sum16(acc, s_red, s_part + 16, tid, lane, warp);
    } else {
      kept_sums(d2, i_lo, i_hi, tau, rank, eq_seen, all_eq, s_warp, tid, lane, warp, acc, [&](int i, double* acc) {
        const float4 s = p.src[i];
        const float4 g = p.tgt_orig[nn[i]];
        acc[0] += (double)d2[i];
        acc[1] += s.x; acc[2] += s.y; acc[3] += s.z;
        acc[4] += g.x; acc[5] += g.y; acc[6] += g.z;
        acc[7] += (double)s.x * g.x; acc[8] += (double)s.x * g.y; acc[9] += (double)s.x * g.z;
        acc[10] += (double)s.y * g.x; acc[11] += (double)s.y * g.y; acc[12] += (double)s.y * g.z;
        acc[13] += (double)s.z * g.x; acc[14] += (double)s.z * g.y; acc[15] += (double)s.z * g.z;
      });
      block_sum16(acc, s_red, s_part, tid, lane, warp);
    }
    cl.sync();
    if (tid == 0) {
      double S[NS];
      for (int k = 0; k < NS; ++k) S[k] = cr ? r_part[k] + s_part[k] : s_part[k] + r_part[k];      // CTA 0's half + CTA 1's half, in both
      old_energy = energy;
      energy = (float)S[0];
      if (PLANE && !(energy <= FLT_MAX)) energy = INFINITY;      // (a NaN residual reports +Inf, as an overflowing one does)
      if (energy <= FLT_MAX) {                     // a kept squared distance overflowed: no fit, and the ratio test below stops
        if constexpr (PLANE) {
          plane_fit<BATCH>(S, sT);
        } else {
          float Tn[12];
          rigid_fit((double)p.n_keep, S + 1, Tn);
          for (int k = 0; k < 12; ++k) sT[k] = Tn[k];
        }
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
// The batch (pgp_refine_batch[_dev]) adds: in4 / placed_T (its segments and placed rows converted on the device), flags (K6),
// keys (the sorts too large for shared memory), the host call's copies of its arguments (raw_*) and results (out), and pinned
// staging for the one upload of its host-built tables.
struct TScratch {
  DevBuf seg, d2, nn, T, iters, energy, cell_of, cursor, items;
  DevBuf in4, placed_T, flags, keys, raw_seg, raw_placed, raw_poses, out;
  StagingRing staging;
  bool prep_smem_set = false;
};
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

// general 4x4 rigid inverse in double: [R t]^-1 = [R^T, -R^T t] (the device copies run unfused like the host's: -fmad=false)
__host__ __device__ void invert_pose(const double* P, double* I) {
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) I[4 * r + c] = P[4 * c + r];
    I[4 * r + 3] = -(P[0 * 4 + r] * P[3] + P[1 * 4 + r] * P[7] + P[2 * 4 + r] * P[11]);
  }
  I[12] = I[13] = I[14] = 0; I[15] = 1;
}

// The host half of one refinement of pgp_tricp / pgp_tricp_plane / pgp_mcts_tricp: n_keep, the source in Morton order, the start
// transforms, and the poses from the refined transforms (the batch runs the same arithmetic on the device, k5_prep_items).

__host__ __device__ int n_keep_of(float trim, int ns) {
  const float keep_f = fabsf(trim * (float)ns);                          // abs(numPoints) on a float, UCTState.cpp:181,194
  return keep_f < 2147483648.f ? ((int)keep_f < ns ? (int)keep_f : ns) : ns;
}

// The source cloud goes up in Morton order of its own bounding box: a rigid transform keeps neighbours together, so the 32
// queries of a warp walk the same few grid rows of the target in every iteration of every pose (the ring searches of unrelated
// points diverge: 4 of 32 lanes were active in the distance loop).  Sums are order-free up to double rounding; ties at the trim
// threshold are admitted in this order.  The order is that of the (code, index) pairs; morton_source computes it on the host
// for the single calls, k5_prep_items on the device for the batch, both with the two functions below.

// edge of the bounding cube of the box [lo, hi]
__host__ __device__ inline float morton_extent(const float lo[3], const float hi[3]) {
  const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
  const float a = dx < dy ? dy : dx, b = dz < 1e-12f ? 1e-12f : dz;                  // std::max(u, v) = u < v ? v : u
  return a < b ? b : a;
}
// 30-bit code of p over the cube [lo, lo + ext]: per axis fp32 (p - lo) / ext, x 1024, clamped to [0, 1023] (NaN -> 0), the
// axes' bits interleaved x lowest
__host__ __device__ inline uint64_t morton_code(float x, float y, float z, const float lo[3], float ext) {
  const float p[3] = {x, y, z};
  uint64_t m = 0;
  for (int c = 0; c < 3; ++c) {
    const float v = (p[c] - lo[c]) / ext * 1024.0f;
    uint64_t q = (uint32_t)(v > 0.0f ? (v < 1023.0f ? v : 1023.0f) : 0.0f);    // std::min(1023, std::max(0, v))
    q = (q | q << 32) & 0x1f00000000ffffull; q = (q | q << 16) & 0x1f0000ff0000ffull; q = (q | q << 8) & 0x100f00f00f00f00full;
    q = (q | q << 4) & 0x10c30c30c30c30c3ull; q = (q | q << 2) & 0x1249249249249249ull;
    m |= q << c;
  }
  return m;
}

// seg4: ns x float4 (w = 0)
void morton_source(const float* seg_xyz_host, int ns, float* seg4) {
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = 0; i < ns; ++i) for (int c = 0; c < 3; ++c) { lo[c] = std::min(lo[c], seg_xyz_host[3 * i + c]); hi[c] = std::max(hi[c], seg_xyz_host[3 * i + c]); }
  const float ext = morton_extent(lo, hi);
  std::vector<std::pair<uint64_t, int>> key((size_t)ns);
  for (int i = 0; i < ns; ++i) {
    const float* p = seg_xyz_host + 3 * (size_t)i;
    key[(size_t)i] = std::make_pair(morton_code(p[0], p[1], p[2], lo, ext), i);
  }
  std::sort(key.begin(), key.end());
  for (int i = 0; i < ns; ++i) {
    for (int c = 0; c < 3; ++c) seg4[4 * (size_t)i + c] = seg_xyz_host[3 * key[(size_t)i].second + c];
    seg4[4 * (size_t)i + 3] = 0.f;
  }
}

// T12: k x 12 fp32, the inverse of each pose (tform = inverse(object pose), UCTState.cpp:184-185)
void start_transforms(const double* poses16_host, int k, float* T12) {
  for (int i = 0; i < k; ++i) {
    double inv[16];
    invert_pose(poses16_host + 16 * (size_t)i, inv);
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) T12[12 * (size_t)i + 4 * r + c] = (float)inv[4 * r + c];
  }
}

// pose = inverse(tform), UCTState.cpp:195-203; a non-finite energy leaves the pose as it was given
void finish_poses(const float* T12, const int* it, const float* en, int k, double* poses16_host, int* iters_out, float* energy_out) {
  for (int i = 0; i < k; ++i) {
    if (en[i] <= FLT_MAX) {
      double M[16] = {0}, inv[16];
      for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) M[4 * r + c] = (double)T12[12 * (size_t)i + 4 * r + c];
      M[15] = 1;
      invert_pose(M, inv);
      memcpy(poses16_host + 16 * (size_t)i, inv, sizeof(inv));
    }
    if (iters_out) iters_out[i] = it[i];
    if (energy_out) energy_out[i] = en[i];
  }
}

void zero_results(int k, int* iters_out, float* energy_out) {
  for (int i = 0; i < k; ++i) { if (iters_out) iters_out[i] = 0; if (energy_out) energy_out[i] = 0.f; }
}

// the TricpParams of one item whose source, d2 / nn rows and pose rows start at the given device addresses
TricpParams item_params(const Model& m, const float4* src, int ns, float* d2, int* nn, float* T, int* iters, float* energy, int n_keep, float ratio,
                        int max_iter) {
  TricpParams p{};
  p.src = src; p.ns = ns;
  p.tgt = m.tgrid_pts.as<float4>(); p.tstart = m.tgrid_start.as<uint32_t>(); p.nt = m.nv; p.tgt_orig = m.val_raw.as<float4>();
  p.nrm_orig = m.val_nrm_orig.as<float4>();
  memcpy(p.tg.lo, m.tg_lo, 12); p.tg.g = m.tg_g; p.tg.inv_g = 1.0f / m.tg_g; memcpy(p.tg.dim, m.tg_dim, 12);
  p.d2 = d2; p.nn = nn; p.T = T;
  p.n_keep = n_keep; p.ratio = ratio; p.max_iter = std::max(1, max_iter);
  p.iters = iters; p.energy = energy;
  return p;
}

// ---------------------------------------------------------------- the batch on the device (pgp_refine_batch[_dev])
// ingest -> K6 -> k5_prep_items -> K5 -> k5_finish, a fixed number of launches and no read-back.  Every row of the packed source
// and of the d2 / nn scratch is laid out by SEGMENT size (an upper bound of the survivors), so the host knows every offset.

// The survivors of an item whose segment has at most K5_SORT_SHARED points are sorted in the dynamic shared memory of its CTA
// (64 KB of keys at most); larger items sort in global memory (TScratch::keys), with the same code.
constexpr int K5_SORT_SHARED = 8192;

// One item as k5_prep_items reads it: its points in in4, its K6 flags (flag_lo < 0: nothing placed), its slot of the packed
// source (src_lo < 0: k = 0) and of the global sort keys (key_lo < 0: sorted in shared memory).
struct PrepItem { int64_t seg_lo, flag_lo, src_lo, key_lo; int ns, k; };

__host__ __device__ inline int pow2_at_least(int n) { int p = 1; while (p < n) p <<= 1; return p; }

// Step 1: segments to float4 (w = 0), placed rows to fp32 (pose16_to_f32x12, as K6 takes them), the start transforms (the fp32
// inverse of every pose, as start_transforms), and the finiteness of every value: a NaN or Inf anywhere sets *status to
// PGP_E_INVALID (PGP_OK was stored before the launch).  Index t < n_pts is a point, the next n_rows placed rows, then the poses.
__global__ void k5_ingest(const float* __restrict__ seg_xyz, int64_t n_pts, const double* __restrict__ placed16, int64_t n_rows,
                          const double* __restrict__ poses16, int64_t n_poses, float4* __restrict__ in4, float* __restrict__ placed_T,
                          float* __restrict__ T, int32_t* __restrict__ status) {
  bool ok = true;
  const int64_t n = n_pts + n_rows + n_poses;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    if (t < n_pts) {
      const float x = seg_xyz[3 * t], y = seg_xyz[3 * t + 1], z = seg_xyz[3 * t + 2];
      ok &= isfinite(x) && isfinite(y) && isfinite(z);
      in4[t] = make_float4(x, y, z, 0.f);
      continue;
    }
    const bool placed = t < n_pts + n_rows;
    const int64_t r = placed ? t - n_pts : t - n_pts - n_rows;
    const double* src = (placed ? placed16 : poses16) + 16 * r;
    double P[16];
    for (int k = 0; k < 16; ++k) { P[k] = src[k]; ok &= isfinite(P[k]); }
    if (placed) {
      pose16_to_f32x12(P, placed_T + 12 * r);
    } else {
      double inv[16];
      invert_pose(P, inv);
      for (int k = 0; k < 12; ++k) T[12 * r + k] = (float)inv[k];
    }
  }
  if (!ok) *status = PGP_E_INVALID;
}

// Step 3: the host half of one item, one CTA per item -- n_unexplained, n_keep and, for an item with k > 0 and n_keep >= 3, its
// survivors in Morton order into its slot of the packed source, with ns and n_keep written into its K5 descriptor.  The bounding
// box is exact (min / max), the codes are morton_code's.  A survivor keeps its segment index i, and the unique keys
// (code << 32 | i) are sorted: compaction keeps the original order, so this is the order std::sort gives morton_source's
// (code, survivor index) pairs.  Bitonic sort over the next power of two, with non-survivors and padding at ~0 (after every
// code of 30 bits); __syncthreads orders the global-memory passes as it does the shared ones.
__global__ void __launch_bounds__(TT) k5_prep_items(const float4* __restrict__ in4, const uint8_t* __restrict__ flags, const PrepItem* __restrict__ items,
                                                    K5Item* __restrict__ desc, float4* __restrict__ src, uint64_t* __restrict__ gkeys, float trim,
                                                    int* __restrict__ n_unexplained, const int32_t* __restrict__ status) {
  extern __shared__ uint64_t s_keys[];
  __shared__ float s_box[TT / 32][6];
  __shared__ int s_cnt[TT / 32];
  if (*status) return;
  const PrepItem P = items[blockIdx.x];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float4* seg = in4 + P.seg_lo;
  const uint8_t* fl = P.flag_lo >= 0 ? flags + P.flag_lo : nullptr;
  float b[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};      // lo, hi of the survivors
  int cnt = 0;
  for (int i = tid; i < P.ns; i += TT)
    if (!fl || !fl[i]) {
      const float4 s = seg[i];
      ++cnt;
      b[0] = fminf(b[0], s.x); b[1] = fminf(b[1], s.y); b[2] = fminf(b[2], s.z);
      b[3] = fmaxf(b[3], s.x); b[4] = fmaxf(b[4], s.y); b[5] = fmaxf(b[5], s.z);
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      b[c] = fminf(b[c], __shfl_xor_sync(0xffffffffu, b[c], o));
      b[3 + c] = fmaxf(b[3 + c], __shfl_xor_sync(0xffffffffu, b[3 + c], o));
    }
  }
  if (lane == 0) { s_cnt[warp] = cnt; for (int c = 0; c < 6; ++c) s_box[warp][c] = b[c]; }
  __syncthreads();
  cnt = 0;
  for (int w = 0; w < TT / 32; ++w) {
    cnt += s_cnt[w];
    for (int c = 0; c < 3; ++c) { b[c] = fminf(b[c], s_box[w][c]); b[3 + c] = fmaxf(b[3 + c], s_box[w][3 + c]); }
  }
  if (tid == 0 && n_unexplained) n_unexplained[blockIdx.x] = cnt;
  if (P.k == 0) return;
  const int n_keep = n_keep_of(trim, cnt);
  if (tid == 0) { desc[blockIdx.x].p.ns = cnt; desc[blockIdx.x].p.n_keep = n_keep; }
  if (n_keep < 3) return;
  const float lo[3] = {b[0], b[1], b[2]}, hi[3] = {b[3], b[4], b[5]};
  const float ext = morton_extent(lo, hi);
  const int n2 = pow2_at_least(P.ns);
  uint64_t* keys = P.key_lo >= 0 ? gkeys + P.key_lo : s_keys;
  for (int i = tid; i < n2; i += TT) {
    uint64_t key = ~0ull;
    if (i < P.ns && (!fl || !fl[i])) { const float4 s = seg[i]; key = morton_code(s.x, s.y, s.z, lo, ext) << 32 | (uint32_t)i; }
    keys[i] = key;
  }
  __syncthreads();
  for (int k = 2; k <= n2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n2; i += TT) {
        const int l = i ^ j;
        if (l > i) {
          const uint64_t x = keys[i], y = keys[l];
          if ((x > y) == ((i & k) == 0)) { keys[i] = y; keys[l] = x; }
        }
      }
      __syncthreads();
    }
  for (int r = tid; r < cnt; r += TT) src[P.src_lo + r] = seg[(uint32_t)keys[r]];
}

// Step 6, one thread per pose (finish_poses): pose = inverse(tform) when the energy is finite, and the iterations and energy; an
// item that K5 skipped (n_keep < 3) keeps its poses and gets 0 / 0.  Nothing is written when the call was refused.
__global__ void k5_finish(const K5Item* __restrict__ desc, const int* __restrict__ pose_item, const float* __restrict__ T, const int* __restrict__ it,
                          const float* __restrict__ en, int n_poses, double* __restrict__ poses16, int* __restrict__ iters_out,
                          float* __restrict__ energy_out, const int32_t* __restrict__ status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_poses || *status) return;
  int iv = 0;
  float ev = 0.f;
  if (desc[pose_item[i]].p.n_keep >= 3) {
    iv = it[i]; ev = en[i];
    if (ev <= FLT_MAX) {
      double M[16] = {0}, inv[16];
      for (int k = 0; k < 12; ++k) M[k] = (double)T[12 * (size_t)i + k];
      M[15] = 1;
      invert_pose(M, inv);
      for (int k = 0; k < 16; ++k) poses16[16 * (size_t)i + k] = inv[k];
    }
  }
  if (iters_out) iters_out[i] = iv;
  if (energy_out) energy_out[i] = ev;
}

}  // namespace

// host-callable copy of max_eigvec4 for the CPU test-suite (tests/test_host_arithmetic.py): N16 row-major symmetric 4x4; returns 1
// and the (unnormalised) eigenvector of the largest eigenvalue, or 0 when the kernel would fall back to Jacobi
extern "C" PGP_API int pgp_host_max_eigvec4(const double* N16, double* q4) {
  double N[4][4];
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) N[i][j] = N16[4 * i + j];
  return max_eigvec4(N, q4) ? 1 : 0;
}

// host-callable copy of solve_plane6 (the 6x6 solve of the point-to-plane fit) for the CPU test-suite: H36 row-major symmetric,
// x6 = H^+ g6 as the kernel computes it; returns the number of eigenvalues kept
extern "C" PGP_API int pgp_host_solve_plane6(const double* H36, const double* g6, double* x6) {
  return solve_plane6(H36, g6, x6);
}


int k5_tricp(pgp_ctx* ctx, Model& m, const float* seg_xyz_host, int ns, double* poses16_host, int k, float trim, float ratio, int max_iter,
             int* iters_out, float* energy_out, bool plane) {
  TScratch& ts = tscratch_of(ctx);
  int rc = build_target_grid(ctx, m);
  if (rc) return rc;
  const int n_keep = n_keep_of(trim, ns);
  if (n_keep < 3) { zero_results(k, iters_out, energy_out); return PGP_OK; }
  std::vector<float> seg4((size_t)ns * 4), T((size_t)k * 12);
  morton_source(seg_xyz_host, ns, seg4.data());
  start_transforms(poses16_host, k, T.data());
  PGP_CUDA(ctx, ts.seg.reserve((size_t)ns * 16));
  PGP_CUDA(ctx, ts.d2.reserve((size_t)k * ns * 4));
  PGP_CUDA(ctx, ts.nn.reserve((size_t)k * ns * 4));
  PGP_CUDA(ctx, ts.T.reserve((size_t)k * 48));
  PGP_CUDA(ctx, ts.iters.reserve((size_t)k * 4));
  PGP_CUDA(ctx, ts.energy.reserve((size_t)k * 4));
  PGP_CUDA(ctx, cudaMemcpyAsync(ts.seg.p, seg4.data(), (size_t)ns * 16, cudaMemcpyHostToDevice, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(ts.T.p, T.data(), (size_t)k * 48, cudaMemcpyHostToDevice, ctx->stream));
  const TricpParams p = item_params(m, ts.seg.as<float4>(), ns, ts.d2.as<float>(), ts.nn.as<int>(), ts.T.as<float>(), ts.iters.as<int>(),
                                    ts.energy.as<float>(), n_keep, ratio, max_iter);
  if (plane) k5_tricp_kernel<true><<<2 * k, TT, 0, ctx->stream>>>(p);     // one cluster of two CTAs per pose
  else k5_tricp_kernel<false><<<2 * k, TT, 0, ctx->stream>>>(p);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  PGP_CUDA(ctx, cudaMemcpyAsync(T.data(), ts.T.p, (size_t)k * 48, cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<int> it(k);
  std::vector<float> en(k);
  PGP_CUDA(ctx, cudaMemcpyAsync(it.data(), ts.iters.p, (size_t)k * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaMemcpyAsync(en.data(), ts.energy.p, (size_t)k * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  finish_poses(T.data(), it.data(), en.data(), k, poses16_host, iters_out, energy_out);
  return PGP_OK;
}

static size_t align16(size_t n) { return (n + 15) & ~(size_t)15; }

// pgp_refine_batch_dev after its checks (pgp_api.cu).  The host lays the batch out from the structure alone, builds the K5
// descriptors, the item table of k5_prep_items, K6's job table and the pose -> item map, and sends them up in ONE copy from pinned
// staging; the descriptors' ns and n_keep are filled in on the device.  Each item runs exactly the arithmetic of its single call.
int k5_refine_batch_dev(pgp_ctx* ctx, bool plane, const float* seg_xyz, const int64_t* seg_offsets, int n_segs, const double* placed16,
                        int64_t n_placed_rows, const pgp_refine_item* items, const int64_t* pose_offsets, int n_items, double* poses16,
                        float threshold, float trim, float ratio, int max_iter, int* iters_out, float* energy_out, int* n_unexplained_out,
                        int32_t* status) {
  TScratch& ts = tscratch_of(ctx);
  cudaStream_t st = ctx->stream;
  for (int i = 0; i < n_items; ++i) {                                   // (cached per model: built once for each distinct obj)
    int rc = build_target_grid(ctx, ctx->models[items[i].obj]);
    if (rc) return rc;
  }
  const int64_t n_pts = seg_offsets[n_segs], n_poses = pose_offsets[n_items];
  std::vector<PrepItem> prep((size_t)n_items);
  std::vector<K6Dev> jobs;
  int64_t n_flags = 0, n_blocks = 0, n_src = 0, n_keys = 0, n_scr = 0;
  int smem_keys = 0;
  for (int i = 0; i < n_items; ++i) {
    const pgp_refine_item& it = items[i];
    const int ns = (int)(seg_offsets[it.seg + 1] - seg_offsets[it.seg]);
    const int k = (int)(pose_offsets[i + 1] - pose_offsets[i]);
    PrepItem& P = prep[(size_t)i];
    P = PrepItem{seg_offsets[it.seg], -1, -1, -1, ns, k};
    if (it.n_placed > 0) {
      const Model& m = ctx->models[it.obj];
      jobs.push_back(K6Dev{m.val_raw.as<float4>(), m.nv, ns, it.n_placed, P.seg_lo, (int64_t)it.placed_lo, n_flags, n_blocks});
      P.flag_lo = n_flags;
      n_flags += ns; n_blocks += (ns + K6_T - 1) / K6_T;
    }
    if (k > 0) {
      P.src_lo = n_src;
      n_src += ns; n_scr += (int64_t)k * ns;
      if (ns > K5_SORT_SHARED) { P.key_lo = n_keys; n_keys += pow2_at_least(ns); }
      else smem_keys = std::max(smem_keys, pow2_at_least(ns));
    }
  }
  const size_t o_prep = align16((size_t)n_items * sizeof(K5Item)), o_jobs = o_prep + align16((size_t)n_items * sizeof(PrepItem));
  const size_t o_map = o_jobs + align16(jobs.size() * sizeof(K6Dev)), blob = o_map + (size_t)n_poses * 4;
  PGP_CUDA(ctx, ts.in4.reserve((size_t)n_pts * 16));
  PGP_CUDA(ctx, ts.placed_T.reserve((size_t)n_placed_rows * 48));
  PGP_CUDA(ctx, ts.flags.reserve((size_t)n_flags));
  PGP_CUDA(ctx, ts.seg.reserve((size_t)n_src * 16));
  PGP_CUDA(ctx, ts.keys.reserve((size_t)n_keys * 8));
  PGP_CUDA(ctx, ts.d2.reserve((size_t)n_scr * 4));
  PGP_CUDA(ctx, ts.nn.reserve((size_t)n_scr * 4));
  PGP_CUDA(ctx, ts.T.reserve((size_t)n_poses * 48));
  PGP_CUDA(ctx, ts.iters.reserve((size_t)n_poses * 4));
  PGP_CUDA(ctx, ts.energy.reserve((size_t)n_poses * 4));
  PGP_CUDA(ctx, ts.items.reserve(blob));
  // 1. ingest (also for n_items = 0: the values are checked all the same)
  PGP_CUDA(ctx, cudaMemsetAsync(status, 0, sizeof(int32_t), st));       // PGP_OK
  const int64_t n_in = n_pts + n_placed_rows + n_poses;
  if (n_in > 0) {
    k5_ingest<<<(unsigned)std::min<int64_t>((n_in + 255) / 256, 16 * ctx->sm_count), 256, 0, st>>>(
        seg_xyz, n_pts, placed16, n_placed_rows, poses16, n_poses, ts.in4.as<float4>(), ts.placed_T.as<float>(), ts.T.as<float>(), status);
    ctx->launches++;
    PGP_CUDA(ctx, cudaGetLastError());
  }
  if (n_items == 0) return PGP_OK;
  // the tables, staged in the next pinned buffer
  StagingRing::Stage* sg = nullptr;
  PGP_CUDA(ctx, ts.staging.acquire(blob, &sg));
  char* h = static_cast<char*>(sg->host);
  K5Item* desc = reinterpret_cast<K5Item*>(h);
  int* pose_item = reinterpret_cast<int*>(h + o_map);
  int64_t scr = 0;
  for (int i = 0; i < n_items; ++i) {
    const PrepItem& P = prep[(size_t)i];
    const int64_t lo = pose_offsets[i];
    desc[i] = K5Item{};
    if (P.k == 0) continue;
    desc[i].p = item_params(ctx->models[items[i].obj], ts.seg.as<float4>() + P.src_lo, 0, ts.d2.as<float>() + scr, ts.nn.as<int>() + scr,
                            ts.T.as<float>() + 12 * lo, ts.iters.as<int>() + lo, ts.energy.as<float>() + lo, 0, ratio, max_iter);
    desc[i].pose_lo = (int)lo;
    for (int j = 0; j < P.k; ++j) pose_item[lo + j] = i;
    scr += (int64_t)P.k * P.ns;
  }
  memcpy(h + o_prep, prep.data(), prep.size() * sizeof(PrepItem));
  if (!jobs.empty()) memcpy(h + o_jobs, jobs.data(), jobs.size() * sizeof(K6Dev));
  PGP_CUDA(ctx, StagingRing::upload(sg, ts.items.p, blob, st));
  const K5Item* desc_dev = ts.items.as<K5Item>();
  const int* map_dev = reinterpret_cast<const int*>(ts.items.as<char>() + o_map);
  // 2. explained points
  int rc = k6_mark_batch_dev(ctx, ts.in4.as<float4>(), reinterpret_cast<const K6Dev*>(ts.items.as<char>() + o_jobs), (int)jobs.size(), n_blocks,
                             ts.placed_T.as<float>(), threshold, ts.flags.as<uint8_t>());
  if (rc) return rc;
  // 3. compaction, n_keep, Morton order
  if (!ts.prep_smem_set) {
    PGP_CUDA(ctx, cudaFuncSetAttribute(k5_prep_items, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * K5_SORT_SHARED));
    ts.prep_smem_set = true;
  }
  k5_prep_items<<<n_items, TT, (size_t)smem_keys * 8, st>>>(ts.in4.as<float4>(), ts.flags.as<uint8_t>(),
                                                           reinterpret_cast<const PrepItem*>(ts.items.as<char>() + o_prep), ts.items.as<K5Item>(),
                                                           ts.seg.as<float4>(), ts.keys.as<uint64_t>(), trim, n_unexplained_out, status);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  if (n_poses == 0) return PGP_OK;
  // 5. one cluster of two CTAs per pose of every item; 6. the poses back
  const K5Batch b{desc_dev, map_dev};
  if (plane) k5_tricp_kernel<true, true><<<2 * (unsigned)n_poses, TT, 0, st>>>(b);
  else k5_tricp_kernel<false, true><<<2 * (unsigned)n_poses, TT, 0, st>>>(b);
  k5_finish<<<(unsigned)((n_poses + 255) / 256), 256, 0, st>>>(desc_dev, map_dev, ts.T.as<float>(), ts.iters.as<int>(), ts.energy.as<float>(), (int)n_poses,
                                                               poses16, iters_out, energy_out, status);
  ctx->launches += 2;
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

// pgp_refine_batch after its checks: its arguments up, the device pipeline, the results down, one synchronisation.
int k5_refine_batch(pgp_ctx* ctx, bool plane, const float* seg_xyz, const int64_t* seg_offsets, int n_segs, const double* placed16, int64_t n_placed_rows,
                    const pgp_refine_item* items, const int64_t* pose_offsets, int n_items, double* poses16, float threshold, float trim,
                    float ratio, int max_iter, int* iters_out, float* energy_out, int* n_unexplained_out) {
  if (n_items == 0) return PGP_OK;
  TScratch& ts = tscratch_of(ctx);
  cudaStream_t st = ctx->stream;
  const int64_t n_pts = seg_offsets[n_segs], n_poses = pose_offsets[n_items];
  PGP_CUDA(ctx, ts.raw_seg.reserve((size_t)n_pts * 12));
  PGP_CUDA(ctx, ts.raw_placed.reserve((size_t)n_placed_rows * 128));
  PGP_CUDA(ctx, ts.raw_poses.reserve((size_t)n_poses * 128));
  PGP_CUDA(ctx, ts.out.reserve((size_t)n_poses * 8 + (size_t)n_items * 4 + 4));
  int* it_dev = ts.out.as<int>();
  float* en_dev = reinterpret_cast<float*>(it_dev + n_poses);
  int* nun_dev = it_dev + 2 * n_poses;
  int32_t* status = nun_dev + n_items;
  if (n_pts) PGP_CUDA(ctx, cudaMemcpyAsync(ts.raw_seg.p, seg_xyz, (size_t)n_pts * 12, cudaMemcpyHostToDevice, st));
  if (n_placed_rows) PGP_CUDA(ctx, cudaMemcpyAsync(ts.raw_placed.p, placed16, (size_t)n_placed_rows * 128, cudaMemcpyHostToDevice, st));
  if (n_poses) PGP_CUDA(ctx, cudaMemcpyAsync(ts.raw_poses.p, poses16, (size_t)n_poses * 128, cudaMemcpyHostToDevice, st));
  int rc = k5_refine_batch_dev(ctx, plane, ts.raw_seg.as<float>(), seg_offsets, n_segs, ts.raw_placed.as<double>(), n_placed_rows, items, pose_offsets,
                               n_items, ts.raw_poses.as<double>(), threshold, trim, ratio, max_iter, it_dev, en_dev, nun_dev, status);
  if (rc) return rc;
  if (n_poses) {
    PGP_CUDA(ctx, cudaMemcpyAsync(poses16, ts.raw_poses.p, (size_t)n_poses * 128, cudaMemcpyDeviceToHost, st));
    if (iters_out) PGP_CUDA(ctx, cudaMemcpyAsync(iters_out, it_dev, (size_t)n_poses * 4, cudaMemcpyDeviceToHost, st));
    if (energy_out) PGP_CUDA(ctx, cudaMemcpyAsync(energy_out, en_dev, (size_t)n_poses * 4, cudaMemcpyDeviceToHost, st));
  }
  if (n_unexplained_out) PGP_CUDA(ctx, cudaMemcpyAsync(n_unexplained_out, nun_dev, (size_t)n_items * 4, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  return PGP_OK;
}

void k5_release(pgp_ctx* ctx) {
  if (!ctx->k5_scratch) return;
  TScratch* ts = static_cast<TScratch*>(ctx->k5_scratch);
  for (DevBuf* b : {&ts->seg, &ts->d2, &ts->nn, &ts->T, &ts->iters, &ts->energy, &ts->cell_of, &ts->cursor, &ts->items, &ts->in4, &ts->placed_T,
                    &ts->flags, &ts->keys, &ts->raw_seg, &ts->raw_placed, &ts->raw_poses, &ts->out})
    b->release();
  ts->staging.release();
  delete ts;
  ctx->k5_scratch = nullptr;
}
