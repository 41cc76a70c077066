/*
 * lcp_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C CPU restatement of the reference's PCS -> LCP -> TrICP hot path.  It exists to CHECK
 * the CUDA kernels (tests/, __graft_entry__.smoke(), bench.py's cpu_baseline / --impl reference
 * legs).  Nothing in the product path may import, link or execute it.
 *
 * Parity status
 *   LCP (count + weighted), centring, priors, kd-tree, improving chain, rigid-from-quad, pair
 *   extraction: PINNED.  tests/test_oracle_golden.py (test_port_equals_reference_live) checks this file against the
 *   reference engine itself (oracle/_ref/libs4ref.so, compiled in place from /root/reference by
 *   oracle/Makefile) on seeded inputs, and tests/golden/ holds vectors minted from that build
 *   (tests/golden/make_golden.py) for machines where /root/reference does not exist.
 *   The reference's own test-suite holds no golden vectors for this path (SURVEY.md 8c).
 *   TrICP: RESTATED, PARITY UNPINNED (independently cross-checked against scipy cKDTree + numpy SVD,
 *   tests/test_tricp_crosscheck.py) -- pcl::recognition::TrimmedICP is not vendored in
 *   /root/reference and PCL is not installed; lo_tricp follows the call sites
 *   (PPE/src/hypothesis_verification/mcts/UCTState.cpp:121-204, PPE/src/misc/utilities.cpp:651-680)
 *   and PCL's published algorithm (pcl/recognition/ransac_based/trimmed_icp.h, PCL 1.7/1.8, the
 *   distro versions of the README's Ubuntu 14.04/16.04).
 *
 * Citations: S4 = /root/reference/src/3rdparty/super4pcs/src/super4pcs,
 *            PPE = /root/reference/src/physim_pose_estimation.
 *
 * Arithmetic: every fp32 operation is individually rounded (compile with -ffp-contract=off) in
 * the association Eigen 3.3.90 + SSE2 produces for the reference (SURVEY.md 7 "Hard parts"):
 *   point transform   t_r = ((M_r0*x + M_r1*y) + M_r2*z) + M_r3           (match4pcsBase.cc:1717)
 *   squared distance  d2  = dx*dx + (dy*dy + dz*dz)                        (kdtree.h:423)
 *   normal rotation   r_i = M_i0*n0 + (M_i1*n1 + M_i2*n2)                  (match4pcsBase.cc:1755)
 *   3-vector dot      a0*b0 + (a1*b1 + a2*b2)                              (match4pcsBase.cc:1756)
 */
#define _GNU_SOURCE
#include <float.h>
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#define LO_LEAF_MAX 64   /* KD_POINT_PER_CELL, S4/accelerators/kdtree.h:63 */
#define LO_DEPTH_MAX 32  /* KD_MAX_DEPTH,      S4/accelerators/kdtree.h:60 */

typedef struct {
  float split;        /* inner: split coordinate                */
  uint32_t child;     /* inner: index of the left child (right = +1) */
  uint32_t start;     /* leaf: first slot in pts/ids            */
  uint32_t count;     /* leaf: number of slots (the reference stores this in 16 bits) */
  uint8_t axis;
  uint8_t is_leaf;
} lo_node;

typedef struct {
  float* pts;     /* permuted copy of the centred scene, 3 floats per slot */
  int32_t* ids;   /* original index of each slot */
  lo_node* nodes;
  uint32_t n_nodes, cap_nodes;
  uint32_t n;
} lo_tree;

typedef struct lo_ctx {
  int nP, nQ, nV;
  float *P, *Pn;          /* centred scene segment + unit normals (engine's "P")      */
  float *Q, *Qn;          /* centred search model ("Q")                               */
  float *V, *Vn;          /* centred validation model ("Q_validation")                */
  float cP[3], cQ[3];
  float* prior;           /* per scene point, orig_probabilities_                     */
  double delta;
  lo_tree tree;
} lo_ctx;

/* ------------------------------------------------------------------------------------------ */
/* kd-tree: S4/accelerators/kdtree.h:355-370 (finalize), :560-641 (createTree), :522-538 (split) */

static uint32_t lo_tree_new_pair(lo_tree* t) {
  if (t->n_nodes + 2 > t->cap_nodes) {
    t->cap_nodes = t->cap_nodes * 2 + 64;
    t->nodes = (lo_node*)realloc(t->nodes, sizeof(lo_node) * t->cap_nodes);
  }
  uint32_t first = t->n_nodes;
  memset(&t->nodes[first], 0, 2 * sizeof(lo_node));
  t->n_nodes += 2;
  return first;
}

/* Partition slots [lo,hi) so that coordinate < sv comes first; returns the boundary.  The
 * exact sweep order is kept because it fixes the order of points inside a leaf, which decides
 * which of two EQUIDISTANT points a query reports (kdtree.h:424 accepts on <=). */
static uint32_t lo_partition(lo_tree* t, int lo, int hi, int axis, float sv) {
  int l = lo, r = hi - 1;
  while (l < r) {
    while (l < hi && t->pts[3 * l + axis] < sv) ++l;
    while (r >= lo && t->pts[3 * r + axis] >= sv) --r;
    if (l > r) break;
    for (int k = 0; k < 3; ++k) {
      float tmp = t->pts[3 * l + k];
      t->pts[3 * l + k] = t->pts[3 * r + k];
      t->pts[3 * r + k] = tmp;
    }
    int32_t ti = t->ids[l]; t->ids[l] = t->ids[r]; t->ids[r] = ti;
    ++l; --r;
  }
  return (uint32_t)(t->pts[3 * l + axis] < sv ? l + 1 : l);
}

static void lo_tree_build_node(lo_tree* t, uint32_t node, uint32_t lo, uint32_t hi, unsigned level) {
  float mn[3], mx[3];
  for (int k = 0; k < 3; ++k) { mn[k] = FLT_MAX / 2; mx[k] = -FLT_MAX / 2; } /* bbox.h:63-64 */
  for (uint32_t i = lo; i < hi; ++i)
    for (int k = 0; k < 3; ++k) {
      float v = t->pts[3 * i + k];
      if (v < mn[k]) mn[k] = v;
      if (v > mx[k]) mx[k] = v;
    }
  int axis = 0;
  float best = 0.5f * (mx[0] - mn[0]);
  for (int k = 1; k < 3; ++k) {
    float h = 0.5f * (mx[k] - mn[k]);
    if (h > best) { best = h; axis = k; }   /* first maximum wins, as Eigen's maxCoeff visitor */
  }
  float sv = mn[axis] + ((mx[axis] - mn[axis]) / 2.0f);   /* bbox.h:91-92 center() */
  uint32_t mid = lo_partition(t, (int)lo, (int)hi, axis, sv);
  uint32_t first = lo_tree_new_pair(t);
  t->nodes[node].axis = (uint8_t)axis;
  t->nodes[node].split = sv;
  t->nodes[node].child = first;
  t->nodes[node].is_leaf = 0;
  uint32_t seg[2][2] = {{lo, mid}, {mid, hi}};
  for (int side = 0; side < 2; ++side) {
    uint32_t a = seg[side][0], b = seg[side][1];
    uint32_t c = first + (uint32_t)side;
    if (b - a <= LO_LEAF_MAX || level >= LO_DEPTH_MAX) {
      t->nodes[c].is_leaf = 1;
      t->nodes[c].start = a;
      t->nodes[c].count = b - a;
    } else {
      lo_tree_build_node(t, c, a, b, level + 1);
    }
  }
}

static void lo_tree_build(lo_tree* t, const float* pts, uint32_t n) {
  memset(t, 0, sizeof(*t));
  t->n = n;
  t->pts = (float*)malloc(sizeof(float) * 3 * (n ? n : 1));
  t->ids = (int32_t*)malloc(sizeof(int32_t) * (n ? n : 1));
  memcpy(t->pts, pts, sizeof(float) * 3 * n);
  for (uint32_t i = 0; i < n; ++i) t->ids[i] = (int32_t)i;
  t->cap_nodes = 4 * n / LO_LEAF_MAX + 64;
  t->nodes = (lo_node*)calloc(t->cap_nodes, sizeof(lo_node));
  t->n_nodes = 1;
  if (n == 0) { t->nodes[0].is_leaf = 1; return; }
  lo_tree_build_node(t, 0, 0, n, 1);
}

static void lo_tree_free(lo_tree* t) { free(t->pts); free(t->ids); free(t->nodes); }

/* Closest point within sqrt(r2): S4/accelerators/kdtree.h:394-459.  Accept on d2 <= best
 * (:424), descend the near child first, visit the far child only while plane^2 < best (:416).
 * Re-entrant (own stack) unlike the reference (member stack, :311). */
static int32_t lo_tree_closest_within(const lo_tree* t, const float q[3], float r2) {
  struct { uint32_t node; float sq; } stack[2 * LO_DEPTH_MAX + 8];
  int top = 0;
  stack[top].node = 0; stack[top].sq = 0.f; ++top;
  int32_t best_id = -1;
  float best = r2;
  while (top) {
    uint32_t nid = stack[top - 1].node;
    float sq = stack[top - 1].sq;
    const lo_node* nd = &t->nodes[nid];
    if (!(sq < best)) { --top; continue; }
    if (nd->is_leaf) {
      --top;
      uint32_t end = nd->start + nd->count;
      for (uint32_t i = nd->start; i < end; ++i) {
        float dx = q[0] - t->pts[3 * i], dy = q[1] - t->pts[3 * i + 1], dz = q[2] - t->pts[3 * i + 2];
        float d2 = dx * dx + (dy * dy + dz * dz);
        if (d2 <= best) { best = d2; best_id = t->ids[i]; }
      }
    } else {
      float off = q[nd->axis] - nd->split;
      uint32_t near_c, far_c;
      if (off < 0.f) { near_c = nd->child; far_c = nd->child + 1; }
      else           { near_c = nd->child + 1; far_c = nd->child; }
      /* the far child inherits the parent's bound, the near child is pushed on top */
      stack[top - 1].node = far_c;
      stack[top - 1].sq = off * off;
      /* NOTE: the reference assigns the parent's sq to the pushed (near) entry and
       * off^2 to the entry that stays (far): */
      stack[top].node = near_c;
      stack[top].sq = sq;
      ++top;
    }
  }
  return best_id;
}

/* ------------------------------------------------------------------------------------------ */
/* init: S4/algorithms/match4pcsBase.cc:216-345 */

static void lo_centroid(const float* xyz, int n, float c[3]) {
  c[0] = c[1] = c[2] = 0.f;
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < 3; ++k) c[k] += xyz[3 * i + k];      /* :242-250, sequential fp32 sums */
  float fn = (float)n;
  for (int k = 0; k < 3; ++k) c[k] /= fn;
}

static float* lo_dup_centred(const float* xyz, int n, const float c[3]) {
  float* out = (float*)malloc(sizeof(float) * 3 * (n ? n : 1));
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < 3; ++k) out[3 * i + k] = xyz[3 * i + k] - c[k];   /* :253-261 */
  return out;
}

/* Point3D::set_normal normalises (S4/shared4pcs.h:85-87); zero / tiny normals are zeroed by the
 * reader (S4/utils/geometry.h:56-82).  Eigen's normalized() = v / sqrt(v.squaredNorm()), with
 * squaredNorm summed as x*x + (y*y + z*z)... the 3-element redux is ((x*x + y*y) + z*z) for the
 * non-vectorised 3-vector; both orders are tried by the pinning test, this is the one that matches. */
static float* lo_dup_normals(const float* nrm, int n) {
  float* out = (float*)calloc((size_t)3 * (n ? n : 1), sizeof(float));
  if (!nrm) return out;
  for (int i = 0; i < n; ++i) {
    float x = nrm[3 * i], y = nrm[3 * i + 1], z = nrm[3 * i + 2];
    float s = x * x + y * y + z * z;
    if (s < 0.01f) continue;
    float len = sqrtf(s);
    out[3 * i] = x / len; out[3 * i + 1] = y / len; out[3 * i + 2] = z / len;
  }
  return out;
}

lo_ctx* lo_create(const float* P_xyz, const float* P_nrm, int nP,
                  const float* Q_xyz, const float* Q_nrm, int nQ,
                  const float* V_xyz, const float* V_nrm, int nV,
                  double delta, const float* K9,
                  const uint16_t* prior_img, int rows, int cols) {
  lo_ctx* c = (lo_ctx*)calloc(1, sizeof(lo_ctx));
  c->nP = nP; c->nQ = nQ; c->nV = nV; c->delta = delta;
  lo_centroid(P_xyz, nP, c->cP);
  lo_centroid(Q_xyz, nQ, c->cQ);                 /* centroid of the SEARCH model, :248-251 */
  c->P = lo_dup_centred(P_xyz, nP, c->cP);
  c->Q = lo_dup_centred(Q_xyz, nQ, c->cQ);
  c->V = lo_dup_centred(V_xyz, nV, c->cQ);       /* validation set is centred on cQ too, :259-261 */
  c->Pn = lo_dup_normals(P_nrm, nP);
  c->Qn = lo_dup_normals(Q_nrm, nQ);
  c->Vn = lo_dup_normals(V_nrm, nV);
  lo_tree_build(&c->tree, c->P, (uint32_t)nP);   /* initKdTree, :1046-1056 */

  /* priors by pin-hole projection of the un-centred scene point, :327-340.  Without an image the
   * harness' imread stand-in returns all-10000 => prior 1.0. */
  c->prior = (float*)malloc(sizeof(float) * (nP ? nP : 1));
  for (int i = 0; i < nP; ++i) {
    if (!prior_img || rows <= 0 || cols <= 0) { c->prior[i] = 1.0f; continue; }
    /* b_ii.pos() += centroid_P_ in fp32, then widened to double and narrowed back (:329-334) */
    float x = c->P[3 * i] + c->cP[0], y = c->P[3 * i + 1] + c->cP[1], z = c->P[3 * i + 2] + c->cP[2];
    float u, v, w;
    if (K9) {
      /* camIntrinsic * Vector3f : 3x3 * 3x1 lazy product, row redux a0*b0 + (a1*b1 + a2*b2)?  The
       * dense 3x3*3x1 product in Eigen 3.3 evaluates column-wise: (K_r0*x + K_r1*y) + K_r2*z. */
      u = (K9[0] * x + K9[1] * y) + K9[2] * z;
      v = (K9[3] * x + K9[4] * y) + K9[5] * z;
      w = (K9[6] * x + K9[7] * y) + K9[8] * z;
    } else { u = x; v = y; w = z; }
    int col = (int)(u / w);
    int row = (int)(v / w);
    if (row < 0) row = 0;
    if (col < 0) col = 0;
    if (row >= rows) row = rows - 1;
    if (col >= cols) col = cols - 1;
    c->prior[i] = (float)prior_img[(size_t)row * cols + col] / 10000;   /* :321-323 */
  }
  return c;
}

void lo_destroy(lo_ctx* c) {
  if (!c) return;
  free(c->P); free(c->Pn); free(c->Q); free(c->Qn); free(c->V); free(c->Vn); free(c->prior);
  lo_tree_free(&c->tree);
  free(c);
}

void lo_get_centroids(const lo_ctx* c, float* cP, float* cQ) {
  memcpy(cP, c->cP, sizeof(float) * 3); memcpy(cQ, c->cQ, sizeof(float) * 3);
}
void lo_get_priors(const lo_ctx* c, float* out) { memcpy(out, c->prior, sizeof(float) * c->nP); }
void lo_get_centred(const lo_ctx* c, int which, float* xyz, float* nrm) {
  const float* s = which == 0 ? c->P : which == 1 ? c->Q : c->V;
  const float* sn = which == 0 ? c->Pn : which == 1 ? c->Qn : c->Vn;
  int n = which == 0 ? c->nP : which == 1 ? c->nQ : c->nV;
  if (xyz) memcpy(xyz, s, sizeof(float) * 3 * n);
  if (nrm) memcpy(nrm, sn, sizeof(float) * 3 * n);
}

/* ------------------------------------------------------------------------------------------ */
/* LCP scoring */

static inline void lo_xform(const float* T, const float* p, float* out) {
  /* T = row-major 3x4.  (mat * p.homogeneous()).head<3>(), match4pcsBase.cc:1717 */
  for (int r = 0; r < 3; ++r)
    out[r] = ((T[4 * r] * p[0] + T[4 * r + 1] * p[1]) + T[4 * r + 2] * p[2]) + T[4 * r + 3];
}

/* Verify with best_LCP_ == 0 (no early termination): match4pcsBase.cc:1699-1731 */
static uint32_t lo_verify_one(const lo_ctx* c, const float* T) {
  const float eps = (float)c->delta;          /* const Scalar epsilon = options_.delta; :1703 */
  const float r2 = eps * eps;                 /* :1710 */
  uint32_t good = 0;
  for (int i = 0; i < c->nV; ++i) {
    float t[3];
    lo_xform(T, c->V + 3 * i, t);
    if (lo_tree_closest_within(&c->tree, t, r2) >= 0) ++good;
  }
  return good;
}

void lo_verify_batch(const lo_ctx* c, const float* T, int64_t n, uint32_t* counts) {
  for (int64_t i = 0; i < n; ++i) counts[i] = lo_verify_one(c, T + 12 * i);
}

/* Verify as Perform_N_steps drives it: running best + early termination (:1708,:1725-1727).
 * frac[i] is what the reference would store in allPose[i].second. */
void lo_verify_running_best(const lo_ctx* c, const float* T, int64_t n, float* frac, int64_t* best_index) {
  const float eps = (float)c->delta, r2 = eps * eps;
  float best_lcp = 0.f;
  int64_t best = -1;
  for (int64_t h = 0; h < n; ++h) {
    int good = 0;
    const size_t np = (size_t)c->nV;
    const int terminate_value = (int)(best_lcp * np);
    for (int i = 0; i < c->nV; ++i) {
      float t[3];
      lo_xform(T + 12 * h, c->V + 3 * i, t);
      if (lo_tree_closest_within(&c->tree, t, r2) >= 0) ++good;
      /* size_t arithmetic exactly as written in the reference: np - i + good < terminate_value */
      if (np - (size_t)i + (size_t)good < (size_t)terminate_value) break;
    }
    float f = (float)good / (float)np;
    frac[h] = f;
    if (f > best_lcp) { best_lcp = f; best = h; }
  }
  *best_index = best;
}

/* WeightedVerify: match4pcsBase.cc:1733-1766.  Returns the score; appends the registered scene
 * indices to reg (if non-NULL, capacity nV) and their number to *nreg. */
static float lo_weighted_one(const lo_ctx* c, const float* T, int32_t* reg, int32_t* nreg) {
  const float eps = (float)c->delta, r2 = eps * eps;
  float acc = 0.f;
  int32_t k = 0;
  for (int i = 0; i < c->nV; ++i) {
    float t[3];
    lo_xform(T, c->V + 3 * i, t);
    int32_t id = lo_tree_closest_within(&c->tree, t, r2);
    if (id < 0) continue;
    const float* n = c->Vn + 3 * i;
    float nq[3];
    for (int r = 0; r < 3; ++r)    /* mat.block<3,3>(0,0) * normal, :1755 */
      nq[r] = T[4 * r] * n[0] + (T[4 * r + 1] * n[1] + T[4 * r + 2] * n[2]);
    const float* ns = c->Pn + 3 * id;
    float d = ns[0] * nq[0] + (ns[1] * nq[1] + ns[2] * nq[2]);
    /* float angle_n = std::acos(dot)*180/M_PI : acosf, float*180, then a double division */
    float angle = (float)((double)(acosf(d) * 180.0f) / M_PI);
    float other = fabsf(180.0f - angle);
    float m = other < angle ? other : angle;   /* std::min(a,b): (b < a) ? b : a -- NaN => a */
    if (m < 30.0f) {
      acc += c->prior[id];
      if (reg) reg[k] = id;
      ++k;
    }
  }
  if (nreg) *nreg = k;
  return acc / (float)c->nV;
}

void lo_weighted_verify_batch(const lo_ctx* c, const float* T, int64_t n, float* scores, int32_t* nreg,
                              int64_t reg_of, int32_t* reg_out) {
  for (int64_t i = 0; i < n; ++i) {
    int32_t k = 0;
    scores[i] = lo_weighted_one(c, T + 12 * i, (reg_out && i == reg_of) ? reg_out : NULL, &k);
    if (nreg) nreg[i] = k;
  }
}

/* multi-threaded count scoring for the CPU baseline (the port's tree query is re-entrant, so one
 * context serves all threads).  Static interleaved partition.  Returns wall seconds. */
typedef struct { const lo_ctx* c; const float* T; int64_t n; uint32_t* counts; int tid, nt; } lo_job;
static void* lo_worker(void* arg) {
  lo_job* j = (lo_job*)arg;
  for (int64_t i = j->tid; i < j->n; i += j->nt) j->counts[i] = lo_verify_one(j->c, j->T + 12 * i);
  return NULL;
}
double lo_verify_batch_mt(const lo_ctx* c, int nthreads, const float* T, int64_t n, uint32_t* counts) {
  struct timespec a, b;
  clock_gettime(CLOCK_MONOTONIC, &a);
  pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * nthreads);
  lo_job* jobs = (lo_job*)malloc(sizeof(lo_job) * nthreads);
  for (int t = 0; t < nthreads; ++t) {
    jobs[t].c = c; jobs[t].T = T; jobs[t].n = n; jobs[t].counts = counts; jobs[t].tid = t; jobs[t].nt = nthreads;
    pthread_create(&th[t], NULL, lo_worker, &jobs[t]);
  }
  for (int t = 0; t < nthreads; ++t) pthread_join(th[t], NULL);
  clock_gettime(CLOCK_MONOTONIC, &b);
  free(th); free(jobs);
  return (double)(b.tv_sec - a.tv_sec) + 1e-9 * (double)(b.tv_nsec - a.tv_nsec);
}

/* Nearest-neighbour id (or -1) of every transformed validation point for ONE hypothesis: the
 * per-point view of WeightedVerify's kd-tree query, for debugging device disagreements. */
void lo_nn_ids(const lo_ctx* c, const float* T, int32_t* ids) {
  const float eps = (float)c->delta, r2 = eps * eps;
  for (int i = 0; i < c->nV; ++i) {
    float t[3];
    lo_xform(T, c->V + 3 * i, t);
    ids[i] = lo_tree_closest_within(&c->tree, t, r2);
  }
}

/* ------------------------------------------------------------------------------------------ */
/* Result shaping: the strictly-improving chain Perform_N_steps returns
 * (match4pcsBase.cc:1888-1914).  idx_out receives the generation indices of the improving
 * hypotheses; the last one is bestHypothesis.  Returns the chain length (may exceed cap). */
int64_t lo_improving_chain(const float* scores, int64_t n, int64_t* idx_out, int64_t cap) {
  float best = 0.f;      /* best_LCP_ starts at 0: a score of exactly 0 never enters the chain */
  int64_t k = 0;
  for (int64_t i = 0; i < n; ++i) {
    if (scores[i] > best) {
      best = scores[i];
      if (k < cap) idx_out[k] = i;
      ++k;
    }
  }
  return k;
}

/* ------------------------------------------------------------------------------------------ */
/* Rigid transform from a congruent (base, quad): ComputeRigidTransformFromCongruentPair
 * (match4pcsBase.cc:1411-1488) + ComputeRigidTransformation (:1504-1614).  Float math in the
 * same sequence of steps; Eigen's exact association inside normalized()/cross()/3x3 products is
 * not reproduced bit-for-bit, so tests compare to the reference within 2e-6 (abs).  Degenerate
 * bases (zero / collinear edges), for which the reference returns `true` with an UNINITIALISED
 * matrix (:1533-1544, SURVEY.md 7), are rejected here: return 0.
 * T16 = centred 4x4 column-major; pose16 = un-centred pose, column-major doubles. */
static void v3_sub(const float* a, const float* b, float* o) { for (int k = 0; k < 3; ++k) o[k] = a[k] - b[k]; }
static float v3_dot(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static void v3_cross(const float* a, const float* b, float* o) {
  o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}
static int v3_normalize(float* a) {
  float s = v3_dot(a, a);
  if (s == 0.f) return 0;
  float l = sqrtf(s);
  for (int k = 0; k < 3; ++k) a[k] /= l;
  return 1;
}
static int lo_frame(const float* p0, const float* p1, const float* p2, float f[3][3]) {
  float e1[3], e2[3];
  v3_sub(p1, p0, f[0]);
  if (!v3_normalize(f[0])) return 0;
  v3_sub(p2, p0, e1);
  float d = v3_dot(e1, f[0]);
  for (int k = 0; k < 3; ++k) e2[k] = e1[k] - d * f[0][k];
  memcpy(f[1], e2, sizeof(e2));
  if (!v3_normalize(f[1])) return 0;
  v3_cross(f[0], f[1], f[2]);
  return 1;
}

int lo_rigid_from_quad(const lo_ctx* c, const int* base, const int* quad, float* T16, double* pose16) {
  const float *b0 = c->P + 3 * base[0], *b1 = c->P + 3 * base[1], *b2 = c->P + 3 * base[2];
  const float *q0 = c->Q + 3 * quad[0], *q1 = c->Q + 3 * quad[1], *q2 = c->Q + 3 * quad[2];
  float c1[3], c2[3];
  for (int k = 0; k < 3; ++k) {
    c1[k] = (b0[k] + b1[k] + b2[k]) / 3.0f;      /* :1428 */
    c2[k] = (q0[k] + q1[k] + q2[k]) / 3.0f;      /* :1452-1454 */
  }
  float fp[3][3], fq[3][3];
  if (!lo_frame(b0, b1, b2, fp)) return 0;
  if (!lo_frame(q0, q1, q2, fq)) return 0;
  float R[3][3];                                  /* rotate_p^T * rotate_q, :1560 */
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) R[i][j] = fp[0][i] * fq[0][j] + fp[1][i] * fq[1][j] + fp[2][i] * fq[2][j];
  /* "rotation should be orthogonal": diag(R*R) - 1 > 1e-6 on any entry rejects (:1563; note R*R,
   * not R*R^T -- restated as written) */
  for (int i = 0; i < 3; ++i) {
    float s = R[i][0] * R[0][i] + R[i][1] * R[1][i] + R[i][2] * R[2][i];
    if (s - 1.0f > 1e-6f) return 0;
  }
  /* translation of Tr(c1) * R * Tr(-c2), :1601-1610 */
  float t[3];
  for (int i = 0; i < 3; ++i) t[i] = c1[i] + (R[i][0] * (-c2[0]) + R[i][1] * (-c2[1]) + R[i][2] * (-c2[2]));
  memset(T16, 0, sizeof(float) * 16);
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) T16[4 * j + i] = R[i][j];
    T16[12 + i] = t[i];
  }
  T16[15] = 1.f;
  /* un-centred: col3 = c1 + cP - R*(c2 + cQ), :1474-1482 */
  for (int k = 0; k < 16; ++k) pose16[k] = (double)T16[k];
  for (int i = 0; i < 3; ++i) {
    float s0 = c2[0] + c->cQ[0], s1 = c2[1] + c->cQ[1], s2 = c2[2] + c->cQ[2];
    float rt = R[i][0] * s0 + R[i][1] * s1 + R[i][2] * s2;
    pose16[12 + i] = (double)((c1[i] + c->cP[i]) - rt);
  }
  return 1;
}

/* ------------------------------------------------------------------------------------------ */
/* Pair extraction: the brute-force specification Match4PCS::ExtractPairs (S4/algorithms/4pcs.cc:
 * 109-192) with the shipped options (no normal / colour / angle gates, super4pcs_test.cc:26,32).
 * For j < i with | ||q_i - q_j|| - d | <= eps emit (j,i) then (i,j).  The comparison is done in
 * double on an fp32 distance, as in pairCreationFunctor.h:38-39,177-179 (pair_distance and
 * pair_distance_epsilon are stored as double there).  Returns the number of ordered pairs. */
int64_t lo_extract_pairs(const lo_ctx* c, float pair_distance, float eps, int32_t* pairs, int64_t cap) {
  int64_t k = 0;
  const double d = (double)pair_distance, e = (double)eps;
  for (int j = 0; j < c->nQ; ++j) {
    const float* p = c->Q + 3 * j;
    for (int i = j + 1; i < c->nQ; ++i) {
      const float* q = c->Q + 3 * i;
      float dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
      float dist = sqrtf(dx * dx + (dy * dy + dz * dz));
      if (fabs((double)dist - d) > e) continue;
      if (k + 2 <= cap) { pairs[2 * k] = j; pairs[2 * k + 1] = i; pairs[2 * k + 2] = i; pairs[2 * k + 3] = j; }
      k += 2;
    }
  }
  return k;
}

/* ------------------------------------------------------------------------------------------ */
/* Trimmed ICP -- RESTATED, PARITY UNPINNED (see header).
 *
 * Call-site conventions (UCTState.cpp:121-204; utilities.cpp:651-680): target = model cloud,
 * source = scene segment, guess = inverse(object pose) i.e. scene->model, n_keep = |trim * N_src|
 * truncated to int, new-to-old energy ratio passed as 1.0 (PCL's setter is believed to clamp any
 * ratio >= 1 to 0.99; `ratio` is therefore a parameter here, default 0.99 at the call sites of
 * this repo).  PCL algorithm: do { transform every source point by T; exact 1-NN in the target;
 * sort correspondences by squared distance; keep the n_keep smallest; energy = sum of kept d2;
 * T <- closed-form rigid fit (SVD / Umeyama without scale) of kept (ORIGINAL source, target)
 * pairs; } while (energy/old_energy < ratio), energy initialised to FLT_MAX.
 * T, in/out: row-major 3x4 float (source->target).  Returns the number of iterations. */
typedef struct { float d2; int32_t src, tgt; } lo_corr;
static int lo_corr_cmp(const void* a, const void* b) {
  const lo_corr *x = (const lo_corr*)a, *y = (const lo_corr*)b;
  if (x->d2 < y->d2) return -1;
  if (x->d2 > y->d2) return 1;
  return (x->src > y->src) - (x->src < y->src);   /* deterministic tie-break (PCL: unspecified) */
}

/* Horn's closed-form absolute orientation via the 4x4 symmetric eigenproblem (double Jacobi).
 * Mathematically identical to the SVD/Umeyama solution for non-degenerate inputs. */
static void lo_jacobi4(double A[4][4], double V[4][4]) {
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) V[i][j] = (i == j);
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0;
    for (int i = 0; i < 4; ++i) for (int j = i + 1; j < 4; ++j) off += A[i][j] * A[i][j];
    if (off < 1e-300) break;
    for (int p = 0; p < 4; ++p)
      for (int q = p + 1; q < 4; ++q) {
        if (fabs(A[p][q]) < 1e-300) continue;
        double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
        double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
        for (int k = 0; k < 4; ++k) {
          double akp = A[k][p], akq = A[k][q];
          A[k][p] = cs * akp - sn * akq; A[k][q] = sn * akp + cs * akq;
        }
        for (int k = 0; k < 4; ++k) {
          double apk = A[p][k], aqk = A[q][k];
          A[p][k] = cs * apk - sn * aqk; A[q][k] = sn * apk + cs * aqk;
        }
        for (int k = 0; k < 4; ++k) {
          double vkp = V[k][p], vkq = V[k][q];
          V[k][p] = cs * vkp - sn * vkq; V[k][q] = sn * vkp + cs * vkq;
        }
      }
  }
}

/* fit R,t minimising sum || R*s_i + t - g_i ||^2 from the 15 sums (two centroids + 3x3
 * cross-covariance); inputs accumulated in double. */
void lo_rigid_fit_from_sums(const double cs[3], const double cg[3], double H[3][3], float* T) {
  /* H[a][b] = sum (s - cs)[a] * (g - cg)[b] */
  double N[4][4];
  double Sxx = H[0][0], Sxy = H[0][1], Sxz = H[0][2];
  double Syx = H[1][0], Syy = H[1][1], Syz = H[1][2];
  double Szx = H[2][0], Szy = H[2][1], Szz = H[2][2];
  N[0][0] = Sxx + Syy + Szz; N[0][1] = Syz - Szy;       N[0][2] = Szx - Sxz;        N[0][3] = Sxy - Syx;
  N[1][0] = N[0][1];        N[1][1] = Sxx - Syy - Szz;  N[1][2] = Sxy + Syx;        N[1][3] = Szx + Sxz;
  N[2][0] = N[0][2];        N[2][1] = N[1][2];          N[2][2] = -Sxx + Syy - Szz; N[2][3] = Syz + Szy;
  N[3][0] = N[0][3];        N[3][1] = N[1][3];          N[3][2] = N[2][3];          N[3][3] = -Sxx - Syy + Szz;
  double V[4][4];
  lo_jacobi4(N, V);
  int best = 0;
  for (int k = 1; k < 4; ++k) if (N[k][k] > N[best][best]) best = k;
  double qw = V[0][best], qx = V[1][best], qy = V[2][best], qz = V[3][best];
  double nrm = sqrt(qw * qw + qx * qx + qy * qy + qz * qz);
  qw /= nrm; qx /= nrm; qy /= nrm; qz /= nrm;
  double R[3][3] = {
      {1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw)},
      {2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw)},
      {2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)}};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) T[4 * i + j] = (float)R[i][j];
    T[4 * i + 3] = (float)(cg[i] - (R[i][0] * cs[0] + R[i][1] * cs[1] + R[i][2] * cs[2]));
  }
}

int lo_tricp(const float* src, int ns, const float* tgt, int nt, float* T, float trim, float ratio,
             int max_iter, float* final_energy) {
  int n_keep = (int)fabsf(trim * (float)ns);       /* abs(numPoints) on a float, UCTState.cpp:181,194 */
  if (n_keep > ns) n_keep = ns;
  if (n_keep < 3 || nt < 1) { if (final_energy) *final_energy = 0.f; return 0; }
  lo_tree tree;
  lo_tree_build(&tree, tgt, (uint32_t)nt);
  lo_corr* corr = (lo_corr*)malloc(sizeof(lo_corr) * ns);
  float energy = FLT_MAX, old_energy;
  int it = 0;
  do {
    for (int i = 0; i < ns; ++i) {
      const float* p = src + 3 * i;
      float q[3];
      for (int r = 0; r < 3; ++r) q[r] = T[4 * r] * p[0] + T[4 * r + 1] * p[1] + T[4 * r + 2] * p[2] + T[4 * r + 3];
      /* exact unbounded 1-NN: restricted query with an infinite radius */
      int32_t id = lo_tree_closest_within(&tree, q, FLT_MAX);
      if (id >= 0) {
        float dx = q[0] - tgt[3 * id], dy = q[1] - tgt[3 * id + 1], dz = q[2] - tgt[3 * id + 2];
        corr[i].d2 = dx * dx + dy * dy + dz * dz;
      } else {
        /* no squared distance below FLT_MAX (NaN or overflowing query): target 0 at FLT_MAX, as K5 */
        id = 0;
        corr[i].d2 = FLT_MAX;
      }
      corr[i].src = i; corr[i].tgt = id;
    }
    qsort(corr, (size_t)ns, sizeof(lo_corr), lo_corr_cmp);
    old_energy = energy;
    double e = 0, cs[3] = {0, 0, 0}, cg[3] = {0, 0, 0};
    for (int k = 0; k < n_keep; ++k) {
      e += corr[k].d2;
      for (int a = 0; a < 3; ++a) { cs[a] += src[3 * corr[k].src + a]; cg[a] += tgt[3 * corr[k].tgt + a]; }
    }
    energy = (float)e;
    if (!(energy <= FLT_MAX)) { ++it; break; }     /* a kept squared distance overflowed: T stays, as K5 */
    for (int a = 0; a < 3; ++a) { cs[a] /= n_keep; cg[a] /= n_keep; }
    double H[3][3] = {{0}};
    for (int k = 0; k < n_keep; ++k)
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b)
          H[a][b] += ((double)src[3 * corr[k].src + a] - cs[a]) * ((double)tgt[3 * corr[k].tgt + b] - cg[b]);
    lo_rigid_fit_from_sums(cs, cg, H, T);
    ++it;
  } while ((energy / old_energy) < ratio && it < max_iter);
  if (final_energy) *final_energy = energy;
  free(corr);
  lo_tree_free(&tree);
  return it;
}

/* Explained-point removal of UCTState::performTrICP (PPE/src/hypothesis_verification/mcts/UCTState.cpp:149-174):
 * explained cloud = the model cloud transformed by every placed pose (pcl::transformPointCloud, fp32, each output
 * coordinate ((m0 x + m1 y) + m2 z) + m3), one FLANN radius search per segment point (L2_Simple squared distance summed
 * left to right; RadiusResultSet keeps dist < radius^2).  RESTATED, PARITY UNPINNED: PCL / FLANN are not vendored.
 * placed: n_placed x 12 row-major fp32 (utilities::convertToMatrix narrows the Isometry3d to Matrix4f).
 * flags[i] = 1 when segment point i is explained.  Returns the number of points that remain. */
int lo_remove_explained(const float* seg, int ns, const float* model, int nm, const float* placed, int n_placed, float threshold,
                        unsigned char* flags) {
  const float r2 = threshold * threshold;
  float* ex = (float*)malloc(sizeof(float) * 3 * (size_t)nm * (size_t)(n_placed > 0 ? n_placed : 1));
  for (int k = 0; k < n_placed; ++k) {
    const float* T = placed + 12 * k;
    for (int j = 0; j < nm; ++j) {
      const float x = model[3 * j], y = model[3 * j + 1], z = model[3 * j + 2];
      float* o = ex + 3 * ((size_t)k * nm + j);
      for (int r = 0; r < 3; ++r) o[r] = ((T[4 * r] * x + T[4 * r + 1] * y) + T[4 * r + 2] * z) + T[4 * r + 3];
    }
  }
  int kept = 0;
  const size_t ne = (size_t)nm * (size_t)n_placed;
  for (int i = 0; i < ns; ++i) {
    unsigned char hit = 0;
    for (size_t j = 0; j < ne && !hit; ++j) {
      const float dx = seg[3 * i] - ex[3 * j], dy = seg[3 * i + 1] - ex[3 * j + 1], dz = seg[3 * i + 2] - ex[3 * j + 2];
      const float d2 = (dx * dx + dy * dy) + dz * dz;
      if (d2 < r2) hit = 1;
    }
    flags[i] = hit;
    kept += hit ? 0 : 1;
  }
  free(ex);
  return kept;
}
