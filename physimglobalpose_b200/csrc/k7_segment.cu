// K7 -- segment preparation on the device: the step in front of the PCS -> LCP path (SURVEY.md 8f-2).
//
//   depth decode     utilities::readDepthImage           PPE/src/misc/utilities.cpp:47-61    ((d << 13) | (d >> 3)) as u16, / 10000
//   mask             GTSegmentation::compute2dSegment    PPE/src/segmentation/Segmentation.cpp:187-207  (class id == object id)
//   back-projection  utilities::convert3dUnOrganizedRGB  PPE/src/misc/utilities.cpp:210-228   fp32 ((v - cx) * depth) / fx, 0.1 < depth < 2.0
//   voxel centroids  pcl::VoxelGrid, leaf 1 cm           Segmentation.cpp:226-229
//   normals          pcl::MovingLeastSquares, r = 2 cm   Segmentation.cpp:231-238  -- as local PCA (smallest eigenvector), towards the camera
//   outlier removal  pcl::RadiusOutlierRemoval 3 cm / 10 PPE/src/hypothesis_generation/ObjectPoseCandidateSet.cpp:28-32, flip + renormalise :39-51
//
// The byte / integer / fp32 parts (decode, mask, back-projection, pixel order) are exact.  The three PCL filters are
// un-vendored third-party code (PCL is neither in the reference tree nor installed): RESTATED, PARITY UNPINNED -- the kernels
// follow the numpy restatement the configs[0] fixture was prepared with, and are tested against it.
// All neighbourhood work runs on the dense voxel table of the centroids (one centroid per voxel), HBM-bound and tiny.
#include <math.h>

#include <algorithm>
#include <vector>

#include "pgp_internal.cuh"

namespace {

constexpr int T = 256;
constexpr int64_t K7_MAX_CELLS = 250000000;            // dense voxel table: 2.5e8 cells, 1 GB per uint32 array

// pass 1: validity flag per pixel; pass 2 (after the scan): emit points in row-major pixel order
__global__ void k7_flags(const uint16_t* __restrict__ depth, const uint8_t* __restrict__ mask, int n, int cls, uint32_t* __restrict__ flag) {
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= n) return;
  const float d = mask[i] == cls ? decode_depth(depth[i]) : 0.f;
  flag[i] = depth_valid(d) ? 1u : 0u;
}
__global__ void k7_emit(const uint16_t* __restrict__ depth, const uint8_t* __restrict__ mask, int n, int cols, int cls, float fx, float fy, float cx,
                        float cy, const uint32_t* __restrict__ off, float4* __restrict__ pts, int* __restrict__ ijk_min, float leaf) {
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= n || off[i + 1] == off[i]) return;
  const float d = decode_depth(depth[i]);
  const int u = i / cols, v = i % cols;
  const float x = __fdiv_rn(__fmul_rn(__fsub_rn((float)v, cx), d), fx);
  const float y = __fdiv_rn(__fmul_rn(__fsub_rn((float)u, cy), d), fy);
  pts[off[i]] = make_float4(x, y, d, __int_as_float(i));
  atomicMin(ijk_min + 0, (int)floorf(__fdiv_rn(x, leaf)));
  atomicMin(ijk_min + 1, (int)floorf(__fdiv_rn(y, leaf)));
  atomicMin(ijk_min + 2, (int)floorf(__fdiv_rn(d, leaf)));
  atomicMax(ijk_min + 3, (int)floorf(__fdiv_rn(x, leaf)));
  atomicMax(ijk_min + 4, (int)floorf(__fdiv_rn(y, leaf)));
  atomicMax(ijk_min + 5, (int)floorf(__fdiv_rn(d, leaf)));
}

struct VoxGrid { int mn[3]; int dim[3]; float leaf; };
__device__ __forceinline__ int vox_key(const VoxGrid& g, float4 p) {
  const int i = (int)floorf(__fdiv_rn(p.x, g.leaf)) - g.mn[0], j = (int)floorf(__fdiv_rn(p.y, g.leaf)) - g.mn[1],
            k = (int)floorf(__fdiv_rn(p.z, g.leaf)) - g.mn[2];
  return i + g.dim[0] * (j + g.dim[1] * k);
}
__global__ void k7_hist(const float4* __restrict__ pts, int n, VoxGrid g, uint32_t* __restrict__ key_of, uint32_t* __restrict__ cnt) {
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= n) return;
  const int k = vox_key(g, pts[i]);
  key_of[i] = (uint32_t)k;
  atomicAdd(cnt + k, 1u);
}
__global__ void k7_scatter(const float4* __restrict__ pts, int n, const uint32_t* __restrict__ key_of, uint32_t* __restrict__ cursor, float4* __restrict__ sorted) {
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= n) return;
  sorted[atomicAdd(cursor + key_of[i], 1u)] = pts[i];
}
// one thread per voxel: order its points by pixel index (deterministic sum order), centroid in double, occupancy flag
__global__ void k7_centroids(float4* __restrict__ sorted, const uint32_t* __restrict__ start, int n_vox, uint32_t* __restrict__ occ) {
  const int v = blockIdx.x * T + threadIdx.x;
  if (v >= n_vox) return;
  const uint32_t s = start[v], e = start[v + 1];
  occ[v] = e > s ? 1u : 0u;
  if (e == s) return;
  for (uint32_t i = s + 1; i < e; ++i) {
    const float4 x = sorted[i];
    const int key = __float_as_int(x.w);
    uint32_t j = i;
    while (j > s && __float_as_int(sorted[j - 1].w) > key) { sorted[j] = sorted[j - 1]; --j; }
    sorted[j] = x;
  }
  double sx = 0, sy = 0, sz = 0;
  for (uint32_t i = s; i < e; ++i) { sx += (double)sorted[i].x; sy += (double)sorted[i].y; sz += (double)sorted[i].z; }
  const double c = (double)(e - s);
  sorted[s] = make_float4((float)(sx / c), (float)(sy / c), (float)(sz / c), 0.f);      // the voxel's centroid parks in its first slot
}
// occupied voxels in key order -> centroid list + voxel -> centroid index table (-1 = empty)
__global__ void k7_compact(const float4* __restrict__ sorted, const uint32_t* __restrict__ start, const uint32_t* __restrict__ occ_scan, int n_vox,
                           float4* __restrict__ cen, int* __restrict__ vox_to_cen) {
  const int v = blockIdx.x * T + threadIdx.x;
  if (v >= n_vox) return;
  if (occ_scan[v + 1] == occ_scan[v]) { vox_to_cen[v] = -1; return; }
  cen[occ_scan[v]] = sorted[start[v]];
  vox_to_cen[v] = (int)occ_scan[v];
}

// smallest-eigenvalue eigenvector of a symmetric 3x3 matrix, cyclic Jacobi in double
__device__ void smallest_eigvec(double a[3][3], double n[3]) {
  double v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int sweep = 0; sweep < 32; ++sweep) {
    const double off = fabs(a[0][1]) + fabs(a[0][2]) + fabs(a[1][2]);
    if (off < 1e-300 || off <= 1e-18 * (fabs(a[0][0]) + fabs(a[1][1]) + fabs(a[2][2]))) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; ++k) { const double akp = a[k][p], akq = a[k][q]; a[k][p] = c * akp - s * akq; a[k][q] = s * akp + c * akq; }
        for (int k = 0; k < 3; ++k) { const double apk = a[p][k], aqk = a[q][k]; a[p][k] = c * apk - s * aqk; a[q][k] = s * apk + c * aqk; }
        for (int k = 0; k < 3; ++k) { const double vkp = v[k][p], vkq = v[k][q]; v[k][p] = c * vkp - s * vkq; v[k][q] = s * vkp + c * vkq; }
      }
  }
  int m = 0;
  if (a[1][1] < a[m][m]) m = 1;
  if (a[2][2] < a[m][m]) m = 2;
  n[0] = v[0][m]; n[1] = v[1][m]; n[2] = v[2][m];
}

// Eigen's Vector3d::unitOrthogonal() -- the local frame pcl::MovingLeastSquares fits its polynomial in
__device__ void unit_orthogonal(const double n[3], double v[3]) {
  if (!(fabs(n[0]) <= fabs(n[2]) * 1e-12) || !(fabs(n[1]) <= fabs(n[2]) * 1e-12)) {
    const double inv = 1.0 / sqrt(n[0] * n[0] + n[1] * n[1]);
    v[0] = -n[1] * inv; v[1] = n[0] * inv; v[2] = 0.0;
  } else {
    const double inv = 1.0 / sqrt(n[1] * n[1] + n[2] * n[2]);
    v[0] = 0.0; v[1] = -n[2] * inv; v[2] = n[1] * inv;
  }
}

// A x = b for a symmetric positive definite 6x6 A (lower triangle read), Cholesky in place.  False if a pivot is not above
// CHOL6_REL_PIVOT times its column's own diagonal: such a system is singular up to rounding (neighbours on one line or on two lines,
// as thin strips and mask edges give), and whether its rounding-level pivot comes out positive is an accident of summation order.
// The threshold makes the decision a property of the geometry, so oracle/segment_port.py::chol6_solve (this function, operation
// for operation) decides the same.
constexpr double CHOL6_REL_PIVOT = 1e-10;
__device__ bool chol6_solve(double A[6][6], double b[6]) {
  for (int j = 0; j < 6; ++j) {
    double d = A[j][j];
    for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k];
    if (!(d > CHOL6_REL_PIVOT * A[j][j])) return false;
    d = sqrt(d);
    A[j][j] = d;
    for (int i = j + 1; i < 6; ++i) {
      double v = A[i][j];
      for (int k = 0; k < j; ++k) v -= A[i][k] * A[j][k];
      A[i][j] = v / d;
    }
  }
  for (int i = 0; i < 6; ++i) { double v = b[i]; for (int k = 0; k < i; ++k) v -= A[i][k] * b[k]; b[i] = v / A[i][i]; }
  for (int i = 5; i >= 0; --i) { double v = b[i]; for (int k = i + 1; k < 6; ++k) v -= A[k][i] * b[k]; b[i] = v / A[i][i]; }
  return true;
}

// one thread per centroid: PCA plane over the neighbours within normal_r and the neighbour count within outlier_r (the point
// itself included).  mls = 0: the plane normal (towards the camera at the origin) is the output normal, the centroid the output
// point.  mls = 1: pcl::MovingLeastSquares as the reference configures it (polynomial fit of order 2, normals, no upsampling;
// PPE/src/segmentation/Segmentation.cpp:231-238) -- the query is projected onto the plane, a weighted (exp(-d^2 / r^2))
// least-squares polynomial [1, v, v^2, u, uv, u^2] in the plane's frame is fitted over the same neighbours, the point moves along
// the plane normal by its value at (0, 0) and the normal tilts by its gradient there; points with fewer than 3 neighbours are
// dropped (proj.w = 0), as PCL drops them.  Restated from PCL's published algorithm (mls.hpp): PARITY UNPINNED, == oracle/segment_port.py.
__global__ void k7_normals(const float4* __restrict__ cen, int nc, VoxGrid g, const int* __restrict__ vox_to_cen, double normal_r, double outlier_r,
                           int min_nb, int mls, float4* __restrict__ nrm, float4* __restrict__ proj, uint32_t* __restrict__ keep,
                           float* __restrict__ max_disp) {
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= nc) return;
  const float4 c = cen[i];
  const int ci = (int)floorf(__fdiv_rn(c.x, g.leaf)) - g.mn[0], cj = (int)floorf(__fdiv_rn(c.y, g.leaf)) - g.mn[1],
            ck = (int)floorf(__fdiv_rn(c.z, g.leaf)) - g.mn[2];
  const int R = (int)ceil(fmax(normal_r, outlier_r) / (double)g.leaf) + 1;
  const double nr2 = normal_r * normal_r, or2 = outlier_r * outlier_r;
  // two passes over the neighbourhood: mean, then covariance (like np.cov on the centred block)
  double mx = 0, my = 0, mz = 0;
  int cnt_n = 0, cnt_o = 0;
  for (int pass = 0; pass < 2; ++pass) {
    double cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int dk = -R; dk <= R; ++dk) {
      const int k = ck + dk;
      if (k < 0 || k >= g.dim[2]) continue;
      for (int dj = -R; dj <= R; ++dj) {
        const int j = cj + dj;
        if (j < 0 || j >= g.dim[1]) continue;
        for (int di = -R; di <= R; ++di) {
          const int ii = ci + di;
          if (ii < 0 || ii >= g.dim[0]) continue;
          const int q = vox_to_cen[ii + g.dim[0] * (j + g.dim[1] * k)];
          if (q < 0) continue;
          const float4 p = cen[q];
          const double dx = (double)p.x - (double)c.x, dy = (double)p.y - (double)c.y, dz = (double)p.z - (double)c.z;
          const double d2 = dx * dx + dy * dy + dz * dz;
          if (pass == 0) {
            if (d2 <= or2) ++cnt_o;
            if (d2 <= nr2) { ++cnt_n; mx += (double)p.x; my += (double)p.y; mz += (double)p.z; }
          } else if (d2 <= nr2) {
            const double ex = (double)p.x - mx, ey = (double)p.y - my, ez = (double)p.z - mz;
            cov[0][0] += ex * ex; cov[0][1] += ex * ey; cov[0][2] += ex * ez; cov[1][1] += ey * ey; cov[1][2] += ey * ez; cov[2][2] += ez * ez;
          }
        }
      }
    }
    if (pass == 0) {
      if (cnt_n > 0) { mx /= cnt_n; my /= cnt_n; mz /= cnt_n; }
    } else {
      double n[3];
      if (cnt_n >= 3) {
        cov[1][0] = cov[0][1]; cov[2][0] = cov[0][2]; cov[2][1] = cov[1][2];
        smallest_eigvec(cov, n);
      } else {
        n[0] = -(double)c.x; n[1] = -(double)c.y; n[2] = -(double)c.z;
      }
      double pt[3] = {(double)c.x, (double)c.y, (double)c.z};
      if (mls) {
        if (cnt_n < 3) { proj[i] = make_float4(c.x, c.y, c.z, 0.f); nrm[i] = make_float4(0.f, 0.f, 0.f, 0.f); keep[i] = 0u; return; }
        const double ln = sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
        n[0] /= ln; n[1] /= ln; n[2] /= ln;
        const double dist = (pt[0] - mx) * n[0] + (pt[1] - my) * n[1] + (pt[2] - mz) * n[2];
        pt[0] -= dist * n[0]; pt[1] -= dist * n[1]; pt[2] -= dist * n[2];
        if (cnt_n >= 6) {
          double va[3], ua[3];
          unit_orthogonal(n, va);
          ua[0] = n[1] * va[2] - n[2] * va[1]; ua[1] = n[2] * va[0] - n[0] * va[2]; ua[2] = n[0] * va[1] - n[1] * va[0];
          double A[6][6], b[6];
          for (int r = 0; r < 6; ++r) { b[r] = 0.0; for (int q = 0; q < 6; ++q) A[r][q] = 0.0; }
          const double inv_r2 = 1.0 / nr2;
          for (int dk = -R; dk <= R; ++dk) {
            const int k = ck + dk;
            if (k < 0 || k >= g.dim[2]) continue;
            for (int dj = -R; dj <= R; ++dj) {
              const int j = cj + dj;
              if (j < 0 || j >= g.dim[1]) continue;
              for (int di = -R; di <= R; ++di) {
                const int ii = ci + di;
                if (ii < 0 || ii >= g.dim[0]) continue;
                const int q = vox_to_cen[ii + g.dim[0] * (j + g.dim[1] * k)];
                if (q < 0) continue;
                const float4 p = cen[q];
                const double dx = (double)p.x - (double)c.x, dy = (double)p.y - (double)c.y, dz = (double)p.z - (double)c.z;
                if (!(dx * dx + dy * dy + dz * dz <= nr2)) continue;                       // the same neighbours as the plane
                const double ex = (double)p.x - pt[0], ey = (double)p.y - pt[1], ez = (double)p.z - pt[2];
                const double w = exp(-(ex * ex + ey * ey + ez * ez) * inv_r2);
                const double u = ex * ua[0] + ey * ua[1] + ez * ua[2], v = ex * va[0] + ey * va[1] + ez * va[2];
                const double f = ex * n[0] + ey * n[1] + ez * n[2];
                const double phi[6] = {1.0, v, v * v, u, u * v, u * u};
                for (int r = 0; r < 6; ++r) {
                  const double wr = w * phi[r];
                  b[r] += wr * f;
                  for (int q2 = 0; q2 <= r; ++q2) A[r][q2] += wr * phi[q2];
                }
              }
            }
          }
          if (chol6_solve(A, b)) {
            pt[0] += b[0] * n[0]; pt[1] += b[0] * n[1]; pt[2] += b[0] * n[2];
            for (int a = 0; a < 3; ++a) n[a] = n[a] - b[3] * ua[a] - b[1] * va[a];
          }
        }
      }
      if (n[0] * pt[0] + n[1] * pt[1] + n[2] * pt[2] > 0) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; }
      const double l = sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
      nrm[i] = make_float4((float)(n[0] / l), (float)(n[1] / l), (float)(n[2] / l), 0.f);
      const float4 out = make_float4((float)pt[0], (float)pt[1], (float)pt[2], 1.f);
      proj[i] = out;
      keep[i] = cnt_o >= min_nb ? 1u : 0u;                   // (mls: overwritten by k7_outlier_count on the projected cloud)
      if (mls) {                                             // |proj - cen| of the stored floats, rounded up: k7_outlier_count's window
        const double ex = (double)out.x - (double)c.x, ey = (double)out.y - (double)c.y, ez = (double)out.z - (double)c.z;
        const float disp = __double2float_ru(sqrt(ex * ex + ey * ey + ez * ez));
        atomicMax(reinterpret_cast<int*>(max_disp), __float_as_int(disp));      // non-negative floats order as their bits
      }
    }
  }
}

// mls = 1: the radius-outlier filter runs on the PROJECTED cloud (ObjectPoseCandidateSet.cpp:28-32 filters what MLS returned), but
// the voxel table holds the centroids.  Two projected points within outlier_r have centroids within outlier_r + 2 * max_disp (the
// largest |proj - cen| of the call, recorded by k7_normals), so a window of ceil((outlier_r + 2 * max_disp) / leaf) + 1 voxels
// around the centroid's voxel holds every neighbour; the + 1 absorbs the rounding of the voxel indices.  The displacement is not
// bounded by normal_r (the polynomial's value at the origin is not), hence the measured bound.  Clamped to the table.
__global__ void k7_outlier_count(const float4* __restrict__ cen, const float4* __restrict__ proj, int nc, VoxGrid g, const int* __restrict__ vox_to_cen,
                                 double outlier_r, int min_nb, const float* __restrict__ max_disp, uint32_t* __restrict__ keep) {
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= nc) return;
  const float4 me = proj[i];
  if (me.w == 0.f) { keep[i] = 0u; return; }
  const float4 c = cen[i];
  const int ci = (int)floorf(__fdiv_rn(c.x, g.leaf)) - g.mn[0], cj = (int)floorf(__fdiv_rn(c.y, g.leaf)) - g.mn[1],
            ck = (int)floorf(__fdiv_rn(c.z, g.leaf)) - g.mn[2];
  const int span = max(g.dim[0], max(g.dim[1], g.dim[2]));
  const double Rd = ceil((outlier_r + 2.0 * (double)*max_disp) / (double)g.leaf) + 1.0;
  const int R = Rd < (double)span ? (int)Rd : span;
  const double or2 = outlier_r * outlier_r;
  int cnt = 0;
  for (int dk = -R; dk <= R; ++dk) {
    const int k = ck + dk;
    if (k < 0 || k >= g.dim[2]) continue;
    for (int dj = -R; dj <= R; ++dj) {
      const int j = cj + dj;
      if (j < 0 || j >= g.dim[1]) continue;
      for (int di = -R; di <= R; ++di) {
        const int ii = ci + di;
        if (ii < 0 || ii >= g.dim[0]) continue;
        const int q = vox_to_cen[ii + g.dim[0] * (j + g.dim[1] * k)];
        if (q < 0) continue;
        const float4 p = proj[q];
        if (p.w == 0.f) continue;
        const double dx = (double)p.x - (double)me.x, dy = (double)p.y - (double)me.y, dz = (double)p.z - (double)me.z;
        if (dx * dx + dy * dy + dz * dz <= or2) ++cnt;
      }
    }
  }
  keep[i] = cnt >= min_nb ? 1u : 0u;
}
__global__ void k7_keep(const float4* __restrict__ cen, const float4* __restrict__ nrm, const uint32_t* __restrict__ keep_scan, int nc,
                        float* __restrict__ xyz, float* __restrict__ nxyz) {
  const int i = blockIdx.x * T + threadIdx.x;
  if (i >= nc || keep_scan[i + 1] == keep_scan[i]) return;
  const uint32_t o = keep_scan[i];
  xyz[3 * o] = cen[i].x; xyz[3 * o + 1] = cen[i].y; xyz[3 * o + 2] = cen[i].z;
  nxyz[3 * o] = nrm[i].x; nxyz[3 * o + 1] = nrm[i].y; nxyz[3 * o + 2] = nrm[i].z;
}

// device scratch of the segment preparation: owned by the context (k7_release)
struct K7Scratch { DevBuf depth, mask, flag, pts, key_of, cnt, cursor, sorted, occ, cen, vox_to_cen, nrm, proj, keep, xyz, nxyz, max_disp; };
K7Scratch& k7_scratch_of(pgp_ctx* ctx) {
  if (!ctx->k7_scratch) ctx->k7_scratch = new K7Scratch();
  return *static_cast<K7Scratch*>(ctx->k7_scratch);
}

int scan_total(pgp_ctx* ctx, uint32_t* data, int64_t n, uint32_t* total) {
  PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((n + 1) / 2048 + 4096) * 4));
  int rc = pgp_scan_exclusive_u32(ctx, data, n + 1, ctx->scene.scratch.as<uint32_t>());
  if (rc) return rc;
  PGP_CUDA(ctx, cudaMemcpyAsync(total, data + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PGP_OK;
}

}  // namespace

int k7_prepare_segment(pgp_ctx* ctx, const uint16_t* depth_host, const uint8_t* mask_host, int rows, int cols, int cls, const float* K9, float leaf,
                       float normal_r, float outlier_r, int min_nb, float* xyz_host, float* nrm_host, int cap, int* n_out, int* n_raw_out) {
  K7Scratch& sc = k7_scratch_of(ctx);
  cudaStream_t st = ctx->stream;
  const int npx = rows * cols;
  *n_out = 0;
  if (n_raw_out) *n_raw_out = 0;
  PGP_CUDA(ctx, sc.depth.reserve((size_t)npx * 2));
  PGP_CUDA(ctx, sc.mask.reserve((size_t)npx));
  PGP_CUDA(ctx, sc.flag.reserve((size_t)(npx + 1) * 4));
  PGP_CUDA(ctx, ctx->work.reserve(4096));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.depth.p, depth_host, (size_t)npx * 2, cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.mask.p, mask_host, (size_t)npx, cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.flag.as<uint32_t>() + npx, 0, 4, st));
  k7_flags<<<(npx + T - 1) / T, T, 0, st>>>(sc.depth.as<uint16_t>(), sc.mask.as<uint8_t>(), npx, cls, sc.flag.as<uint32_t>());
  ctx->launches++;
  uint32_t n_raw = 0;
  int rc = scan_total(ctx, sc.flag.as<uint32_t>(), npx, &n_raw);
  if (rc) return rc;
  if (n_raw_out) *n_raw_out = (int)n_raw;
  if (n_raw == 0) return PGP_OK;
  PGP_CUDA(ctx, sc.pts.reserve((size_t)n_raw * 16));
  int* d_mm = ctx->work.as<int>() + 96;                               // 6 ints: voxel index min / max per axis
  const int init[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000};
  PGP_CUDA(ctx, cudaMemcpyAsync(d_mm, init, sizeof(init), cudaMemcpyHostToDevice, st));
  k7_emit<<<(npx + T - 1) / T, T, 0, st>>>(sc.depth.as<uint16_t>(), sc.mask.as<uint8_t>(), npx, cols, cls, K9[0], K9[4], K9[2], K9[5],
                                          sc.flag.as<uint32_t>(), sc.pts.as<float4>(), d_mm, leaf);
  ctx->launches++;
  int mm[6];
  PGP_CUDA(ctx, cudaMemcpyAsync(mm, d_mm, sizeof(mm), cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  // the index span in int64: max - min + 1 of two ints can exceed INT_MAX (the leaf refusal of pgp_prepare_segment keeps every index
  // within +-2^30, this keeps the table size honest regardless); each factor is checked before the next multiplication, so the
  // product never exceeds 2.5e8 * 2^32
  VoxGrid g{};
  g.leaf = leaf;
  int64_t dim[3], cells = 1;
  for (int k = 0; k < 3; ++k) {
    g.mn[k] = mm[k];
    dim[k] = (int64_t)mm[3 + k] - (int64_t)mm[k] + 1;
    cells *= dim[k];
    if (cells > K7_MAX_CELLS)
      return pgp_fail(ctx, PGP_E_TOO_LARGE, "segment voxel table needs more than %lld cells (span %lld x %lld x %lld voxels so far)", (long long)K7_MAX_CELLS,
                      (long long)dim[0], (long long)(k > 0 ? dim[1] : 1), (long long)(k > 1 ? dim[2] : 1));
  }
  for (int k = 0; k < 3; ++k) g.dim[k] = (int)dim[k];
  const int n_vox = (int)cells;
  PGP_CUDA(ctx, sc.key_of.reserve((size_t)n_raw * 4));
  PGP_CUDA(ctx, sc.cnt.reserve((size_t)(n_vox + 1) * 4));
  PGP_CUDA(ctx, sc.cursor.reserve((size_t)(n_vox + 1) * 4));
  PGP_CUDA(ctx, sc.sorted.reserve((size_t)n_raw * 16));
  PGP_CUDA(ctx, sc.occ.reserve((size_t)(n_vox + 1) * 4));
  PGP_CUDA(ctx, sc.vox_to_cen.reserve((size_t)n_vox * 4));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.cnt.p, 0, (size_t)(n_vox + 1) * 4, st));
  const int nb = ((int)n_raw + T - 1) / T, vb = (n_vox + T - 1) / T;
  k7_hist<<<nb, T, 0, st>>>(sc.pts.as<float4>(), (int)n_raw, g, sc.key_of.as<uint32_t>(), sc.cnt.as<uint32_t>());
  ctx->launches++;
  PGP_CUDA(ctx, ctx->scene.scratch.reserve((size_t)((n_vox + 1) / 2048 + 4096) * 4));
  rc = pgp_scan_exclusive_u32(ctx, sc.cnt.as<uint32_t>(), (int64_t)n_vox + 1, ctx->scene.scratch.as<uint32_t>());
  if (rc) return rc;
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.cursor.p, sc.cnt.p, (size_t)(n_vox + 1) * 4, cudaMemcpyDeviceToDevice, st));
  k7_scatter<<<nb, T, 0, st>>>(sc.pts.as<float4>(), (int)n_raw, sc.key_of.as<uint32_t>(), sc.cursor.as<uint32_t>(), sc.sorted.as<float4>());
  PGP_CUDA(ctx, cudaMemsetAsync(sc.occ.as<uint32_t>() + n_vox, 0, 4, st));
  k7_centroids<<<vb, T, 0, st>>>(sc.sorted.as<float4>(), sc.cnt.as<uint32_t>(), n_vox, sc.occ.as<uint32_t>());
  ctx->launches += 2;
  uint32_t nc = 0;
  rc = scan_total(ctx, sc.occ.as<uint32_t>(), n_vox, &nc);
  if (rc) return rc;
  PGP_CUDA(ctx, sc.cen.reserve((size_t)nc * 16));
  PGP_CUDA(ctx, sc.nrm.reserve((size_t)nc * 16));
  PGP_CUDA(ctx, sc.proj.reserve((size_t)nc * 16));
  PGP_CUDA(ctx, sc.keep.reserve((size_t)(nc + 1) * 4));
  PGP_CUDA(ctx, sc.xyz.reserve((size_t)nc * 12));
  PGP_CUDA(ctx, sc.nxyz.reserve((size_t)nc * 12));
  k7_compact<<<vb, T, 0, st>>>(sc.sorted.as<float4>(), sc.cnt.as<uint32_t>(), sc.occ.as<uint32_t>(), n_vox, sc.cen.as<float4>(), sc.vox_to_cen.as<int>());
  PGP_CUDA(ctx, cudaMemsetAsync(sc.keep.as<uint32_t>() + nc, 0, 4, st));
  PGP_CUDA(ctx, sc.max_disp.reserve(4));
  PGP_CUDA(ctx, cudaMemsetAsync(sc.max_disp.p, 0, 4, st));                // +0.0f: the atomicMax identity of non-negative float bits
  k7_normals<<<((int)nc + T - 1) / T, T, 0, st>>>(sc.cen.as<float4>(), (int)nc, g, sc.vox_to_cen.as<int>(), (double)normal_r, (double)outlier_r, min_nb,
                                                 ctx->k7_mls, sc.nrm.as<float4>(), sc.proj.as<float4>(), sc.keep.as<uint32_t>(), sc.max_disp.as<float>());
  ctx->launches += 2;
  if (ctx->k7_mls) {
    k7_outlier_count<<<((int)nc + T - 1) / T, T, 0, st>>>(sc.cen.as<float4>(), sc.proj.as<float4>(), (int)nc, g, sc.vox_to_cen.as<int>(), (double)outlier_r, min_nb,
                                                         sc.max_disp.as<float>(), sc.keep.as<uint32_t>());
    ctx->launches++;
  }
  uint32_t n_keep = 0;
  rc = scan_total(ctx, sc.keep.as<uint32_t>(), nc, &n_keep);
  if (rc) return rc;
  if ((int)n_keep > cap) return pgp_fail(ctx, PGP_E_CAPACITY, "segment has %u points, capacity %d", n_keep, cap);
  if (n_keep) {
    k7_keep<<<((int)nc + T - 1) / T, T, 0, st>>>(sc.proj.as<float4>(), sc.nrm.as<float4>(), sc.keep.as<uint32_t>(), (int)nc, sc.xyz.as<float>(), sc.nxyz.as<float>());
    ctx->launches++;
    PGP_CUDA(ctx, cudaMemcpyAsync(xyz_host, sc.xyz.p, (size_t)n_keep * 12, cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaMemcpyAsync(nrm_host, sc.nxyz.p, (size_t)n_keep * 12, cudaMemcpyDeviceToHost, st));
  }
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  PGP_CUDA(ctx, cudaGetLastError());
  *n_out = (int)n_keep;
  return PGP_OK;
}

void k7_release(pgp_ctx* ctx) {
  if (!ctx->k7_scratch) return;
  K7Scratch* sc = static_cast<K7Scratch*>(ctx->k7_scratch);
  for (DevBuf* b : {&sc->depth, &sc->mask, &sc->flag, &sc->pts, &sc->key_of, &sc->cnt, &sc->cursor, &sc->sorted, &sc->occ, &sc->cen, &sc->vox_to_cen, &sc->nrm,
                    &sc->proj, &sc->keep, &sc->xyz, &sc->nxyz, &sc->max_disp})
    b->release();
  delete sc;
  ctx->k7_scratch = nullptr;
}
