// The C ABI of include/pgp.h: context, host-side preparation (the O(n) part of
// Match4PCSBase::init, S4/algorithms/match4pcsBase.cc:216-345) and the thin wrappers that order
// the kernels of k1..k5 on the context's stream.  No CPU scoring path exists in this library.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <numeric>

#include "pgp_internal.cuh"

static std::string g_create_error;

int pgp_fail(pgp_ctx* ctx, int code, const char* fmt, ...) {
  char buf[768];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_create_error = buf;
  return code;
}

#define CHECK_CTX(ctx) do { if (!(ctx)) return PGP_E_INVALID; cudaSetDevice((ctx)->device); } while (0)

namespace {

// centroid exactly as match4pcsBase.cc:242-251: sequential fp32 accumulation, then / Scalar(n)
void seq_centroid(const float* xyz, int n, float c[3]) {
  volatile float sx = 0.f, sy = 0.f, sz = 0.f;   // volatile: keep the compiler from re-associating / vectorising the sum
  for (int i = 0; i < n; ++i) { sx = sx + xyz[3 * i]; sy = sy + xyz[3 * i + 1]; sz = sz + xyz[3 * i + 2]; }
  const float fn = (float)n;
  c[0] = sx / fn; c[1] = sy / fn; c[2] = sz / fn;
}

// Point3D::set_normal (S4/shared4pcs.h:85-87) + CleanInvalidNormals (S4/utils/geometry.h:56-82)
void unit_normal(const float* n, float out[3]) {
  out[0] = out[1] = out[2] = 0.f;
  if (!n) return;
  volatile float s = n[0] * n[0];
  s = s + n[1] * n[1];
  s = s + n[2] * n[2];
  if (s < 0.01f) return;
  float len = sqrtf(s);
  out[0] = n[0] / len; out[1] = n[1] / len; out[2] = n[2] / len;
}

int upload_cloud4(pgp_ctx* ctx, DevBuf& buf, const std::vector<float>& v4) {
  PGP_CUDA(ctx, buf.reserve(std::max<size_t>(v4.size() * 4, 64)));
  if (!v4.empty()) PGP_CUDA(ctx, cudaMemcpyAsync(buf.p, v4.data(), v4.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  return PGP_OK;
}

Model* get_model(pgp_ctx* ctx, int obj) {
  if (obj < 0 || obj >= (int)ctx->models.size() || !ctx->models[obj].ready) return nullptr;
  return &ctx->models[obj];
}

}  // namespace

extern "C" {

const char* pgp_version(void) { return "pgp-b200 0.1 (sm_100a)"; }

pgp_ctx* pgp_create(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    pgp_fail(nullptr, PGP_E_CUDA, "no CUDA device (%s); this library has no CPU path", e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    return nullptr;
  }
  if (device < 0 || device >= n) { pgp_fail(nullptr, PGP_E_INVALID, "device %d out of range (%d devices)", device, n); return nullptr; }
  if ((e = cudaSetDevice(device)) != cudaSuccess) { pgp_fail(nullptr, PGP_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e)); return nullptr; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major < 10) { pgp_fail(nullptr, PGP_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); return nullptr; }
  pgp_ctx* ctx = new pgp_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->back_stream, cudaStreamNonBlocking) != cudaSuccess) {
    pgp_fail(nullptr, PGP_E_CUDA, "cudaStreamCreate failed");
    delete ctx;
    return nullptr;
  }
  for (BatchSlot& bs : ctx->batch) {
    cudaEventCreateWithFlags(&bs.ev_start, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&bs.ev_first, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&bs.ev_scored, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&bs.ev_done, cudaEventDisableTiming);
  }
  ctx->stream = ctx->own_stream;
  ctx->models.resize(PGP_MAX_OBJECTS);
  // `work` holds the counters kernel parameters point at (K3's work / ready counters, K4's histograms and records): it is sized
  // once for its largest user (K4, ~350 KB) so that it is never reallocated while a launch that references it is in flight
  if (ctx->work.reserve(PGP_WORK_BYTES) != cudaSuccess) {
    pgp_fail(nullptr, PGP_E_NOMEM, "cudaMalloc of the %d-byte work buffer failed", PGP_WORK_BYTES);
    pgp_destroy(ctx);
    return nullptr;
  }
  return ctx;
}

void pgp_destroy(pgp_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  Scene& s = ctx->scene;
  for (DevBuf* b : {&s.xyz_raw, &s.nrm_raw, &s.unsorted, &s.cursor, &s.pts, &s.aux, &s.cell_start, &s.cell_of, &s.bitmap, &s.bmrank,
                    &s.block_cell, &s.codes, &s.near_cnt, &s.hdr, &s.region, &s.hdrw, &s.adesc, &s.arec, &s.wvox, &s.wbase, &s.wcnt, &s.wword, &s.wlists, &s.vrec, &s.aux_orig, &s.dist, &s.dist_tmp, &s.prior, &s.scratch, &ctx->work, &ctx->topk_out})
    b->release();
  for (BatchSlot& bs : ctx->batch) {
    bs.T.release(); bs.counts.release(); bs.scores.release();
    for (cudaEvent_t e : {bs.ev_start, bs.ev_first, bs.ev_scored, bs.ev_done}) if (e) cudaEventDestroy(e);
  }
  for (Model& m : ctx->models)
    for (DevBuf* b : {&m.search, &m.search_nrm, &m.search_unit, &m.val, &m.val_nrm, &m.val_orig, &m.val_nrm_orig, &m.gen_T, &m.gen_counts, &m.gen_scores,
                      &m.tgrid_pts, &m.tgrid_start, &m.val_raw, &m.val_groups, &m.ppf_keys, &m.ppf_offsets, &m.ppf_pairs, &m.ppf_bits})
      b->release();
  pgp_comm_release(ctx);
  k2_release(ctx);
  k5_release(ctx);
  k6_release(ctx);
  k7_release(ctx);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  cudaStreamDestroy(ctx->own_stream);
  cudaStreamDestroy(ctx->copy_stream);
  cudaStreamDestroy(ctx->back_stream);
  delete ctx;
}

const char* pgp_last_error(const pgp_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int pgp_set_stream(pgp_ctx* ctx, void* cuda_stream) {
  CHECK_CTX(ctx);
  ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return PGP_OK;
}

int pgp_synchronize(pgp_ctx* ctx) {
  CHECK_CTX(ctx);
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PGP_OK;
}

int64_t pgp_launch_count(const pgp_ctx* ctx) { return ctx ? ctx->launches : 0; }

int pgp_set_option(pgp_ctx* ctx, const char* name, int value) {
  CHECK_CTX(ctx);
  if (name && !strcmp(name, "force_coarse")) { ctx->force_coarse = value; return PGP_OK; }
  if (name && (!strcmp(name, "k3_warps_count") || !strcmp(name, "k3_warps_weighted"))) {
    if (value != 16 && value != 24 && value != 32 && !(value == 28 && !strcmp(name, "k3_warps_weighted")))
      return pgp_fail(ctx, PGP_E_INVALID, "%s must be 16, 24 or 32 (weighted: also 28)", name);
    (strcmp(name, "k3_warps_count") ? ctx->k3_warps_weighted : ctx->k3_warps_count) = value;
    return PGP_OK;
  }
  if (name && !strcmp(name, "k3_smem_table")) { ctx->k3_smem_table = value < 0 ? -1 : (value ? 1 : 0); return PGP_OK; }
  if (name && !strcmp(name, "k7_mls")) { ctx->k7_mls = value ? 1 : 0; return PGP_OK; }
  if (name && !strcmp(name, "group_cull")) { ctx->group_cull = value ? 1 : 0; return PGP_OK; }
  if (name && !strcmp(name, "stream_upload")) { ctx->stream_upload = value ? 1 : 0; return PGP_OK; }
  if (name && !strcmp(name, "tail_split")) { ctx->tail_split = value < 1 ? 1 : (value > 16 ? 16 : value); return PGP_OK; }
  return pgp_fail(ctx, PGP_E_INVALID, "unknown option %s", name ? name : "(null)");
}

int pgp_set_scene(pgp_ctx* ctx, const float* xyz, const float* nrm, int n, float delta) {
  CHECK_CTX(ctx);
  if (!xyz || n <= 0) return pgp_fail(ctx, PGP_E_INVALID, "pgp_set_scene: empty cloud");
  if (!(delta > 0.f) || !std::isfinite(delta)) return pgp_fail(ctx, PGP_E_INVALID, "pgp_set_scene: delta must be > 0");
  Scene& s = ctx->scene;
  s.ready = false;
  s.n = n;
  s.delta = delta;
  s.has_nrm = nrm != nullptr;
  seq_centroid(xyz, n, s.cP);
  PGP_CUDA(ctx, s.xyz_raw.reserve((size_t)n * 12));
  PGP_CUDA(ctx, cudaMemcpyAsync(s.xyz_raw.p, xyz, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
  if (nrm) {
    PGP_CUDA(ctx, s.nrm_raw.reserve((size_t)n * 12));
    PGP_CUDA(ctx, cudaMemcpyAsync(s.nrm_raw.p, nrm, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
  }
  PGP_CUDA(ctx, ctx->work.reserve(4096));
  int rc = k1_fill_priors(ctx, 1.0f);
  if (rc) return rc;
  ctx->last = LastBatch();
  return k1_build_grid(ctx);
}

int pgp_set_scene_priors(pgp_ctx* ctx, const float* prior) {
  CHECK_CTX(ctx);
  Scene& s = ctx->scene;
  if (!s.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (!prior) return pgp_fail(ctx, PGP_E_INVALID, "null priors");
  // Any finite value is a valid prior, negative ones included (the reference does not restrict orig_probabilities_, and the ordered
  // weighted sum handles them exactly).  A NaN or an infinity would make scores that have no order, so it is refused here.
  for (int i = 0; i < s.n; ++i)
    if (!std::isfinite(prior[i])) return pgp_fail(ctx, PGP_E_INVALID, "prior %d is not finite (%g)", i, (double)prior[i]);
  PGP_CUDA(ctx, cudaMemcpyAsync(s.prior.p, prior, (size_t)s.n * 4, cudaMemcpyHostToDevice, ctx->stream));
  return k1_refresh_sorted_priors(ctx);
}

int pgp_get_scene_priors(pgp_ctx* ctx, float* prior) {
  CHECK_CTX(ctx);
  Scene& s = ctx->scene;
  if (!s.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  PGP_CUDA(ctx, cudaMemcpyAsync(prior, s.prior.p, (size_t)s.n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PGP_OK;
}

int pgp_set_scene_prior_image(pgp_ctx* ctx, const uint16_t* img, int rows, int cols, const float* K9) {
  CHECK_CTX(ctx);
  Scene& s = ctx->scene;
  if (!s.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (!img || rows <= 0 || cols <= 0 || !K9) return pgp_fail(ctx, PGP_E_INVALID, "bad prior image");
  PGP_CUDA(ctx, s.scratch.reserve((size_t)rows * cols * 2));
  PGP_CUDA(ctx, cudaMemcpyAsync(s.scratch.p, img, (size_t)rows * cols * 2, cudaMemcpyHostToDevice, ctx->stream));
  return k1_project_priors(ctx, s.scratch.as<uint16_t>(), rows, cols, K9);
}

int pgp_set_model(pgp_ctx* ctx, int obj, const float* sx, const float* sn, int nq, const float* vx, const float* vn, int nv) {
  CHECK_CTX(ctx);
  if (obj < 0 || obj >= PGP_MAX_OBJECTS) return pgp_fail(ctx, PGP_E_INVALID, "object slot %d out of range", obj);
  if (!sx || nq <= 0 || !vx || nv <= 0) return pgp_fail(ctx, PGP_E_INVALID, "pgp_set_model: empty cloud");
  Model& m = ctx->models[obj];
  m.ready = false;
  m.nq = nq; m.nv = nv; m.n_gen = 0; m.tgrid_ready = false; m.val_rinf = 0.f;
  seq_centroid(sx, nq, m.cQ);   // centroid of the SEARCH cloud centres both clouds (:248-261)
  std::vector<float> s4((size_t)nq * 4), sn4((size_t)nq * 4), v4((size_t)nv * 4), vn4((size_t)nv * 4);
  for (int i = 0; i < nq; ++i) {
    for (int k = 0; k < 3; ++k) s4[4 * (size_t)i + k] = sx[3 * i + k] - m.cQ[k];
    int idx = i; memcpy(&s4[4 * (size_t)i + 3], &idx, 4);
    unit_normal(sn ? sn + 3 * i : nullptr, &sn4[4 * (size_t)i]);
  }
  // unit-cube copy of the search cloud for the quad join: bbox centre and ratio as synch3DContent
  // (pairCreationFunctor.h:102-138; AABB::center = min + (max - min)/2, accelerators/bbox.h:91-92)
  {
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = 0; i < nq; ++i)
      for (int k = 0; k < 3; ++k) { mn[k] = std::min(mn[k], s4[4 * (size_t)i + k]); mx[k] = std::max(mx[k], s4[4 * (size_t)i + k]); }
    double ratio = 0.0;
    for (int k = 0; k < 3; ++k) {
      m.unit_center[k] = mn[k] + ((mx[k] - mn[k]) / 2.0f);
      ratio = std::max(ratio, (double)(mx[k] - mn[k]) + 0.001);
    }
    m.unit_ratio = (float)ratio;
    std::vector<float> u4((size_t)nq * 4, 0.f);
    for (int i = 0; i < nq; ++i)
      for (int k = 0; k < 3; ++k) {
        volatile float t = s4[4 * (size_t)i + k] - m.unit_center[k];
        t = t / m.unit_ratio;
        u4[4 * (size_t)i + k] = t + 0.5f;
      }
    int rc0 = upload_cloud4(ctx, m.search_unit, u4);
    if (rc0) return rc0;
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // diameter estimate from 1000 pseudo-random pairs, like init() (:274-283) but with a fixed hash instead of rand()
    m.search_diameter = 0.f;
    uint64_t st = 0x1234567ull;
    for (int t = 0; t < 1000; ++t) {
      st = st * 6364136223846793005ull + 1442695040888963407ull; const int a = (int)((st >> 33) % (uint64_t)nq);
      st = st * 6364136223846793005ull + 1442695040888963407ull; const int b = (int)((st >> 33) % (uint64_t)nq);
      float d2 = 0.f;
      for (int k = 0; k < 3; ++k) { float d = s4[4 * (size_t)b + k] - s4[4 * (size_t)a + k]; d2 += d * d; }
      m.search_diameter = std::max(m.search_diameter, sqrtf(d2));
    }
  }
  for (int i = 0; i < nv; ++i) {
    for (int k = 0; k < 3; ++k) {
      float c = vx[3 * i + k] - m.cQ[k];
      v4[4 * (size_t)i + k] = c;
      m.val_rinf = std::max(m.val_rinf, fabsf(c));
    }
    int idx = i; memcpy(&v4[4 * (size_t)i + 3], &idx, 4);
    unit_normal(vn ? vn + 3 * i : nullptr, &vn4[4 * (size_t)i]);
  }
  // scoring order of the validation cloud: leaves of a balanced kd split (widest axis, cut at a multiple of 32 points), so every
  // aligned run of 32 points -- what a warp handles per step -- is a compact patch: its queries fall into neighbouring cells, and
  // its bounding sphere is small enough for K3's group cull to fire (counts are order-free).
  std::vector<int> order(nv);
  std::iota(order.begin(), order.end(), 0);
  {
    struct Range { int b, e; };
    std::vector<Range> stack{{0, nv}};
    while (!stack.empty()) {
      const Range r = stack.back(); stack.pop_back();
      const int n = r.e - r.b;
      if (n <= 32) continue;
      float rlo[3] = {INFINITY, INFINITY, INFINITY}, rhi[3] = {-INFINITY, -INFINITY, -INFINITY};
      for (int i = r.b; i < r.e; ++i)
        for (int k = 0; k < 3; ++k) { const float c = v4[4 * (size_t)order[i] + k]; rlo[k] = std::min(rlo[k], c); rhi[k] = std::max(rhi[k], c); }
      int ax = 0;
      for (int k = 1; k < 3; ++k) if (rhi[k] - rlo[k] > rhi[ax] - rlo[ax]) ax = k;
      const int half = ((n + 31) / 32 / 2) * 32;
      std::nth_element(order.begin() + r.b, order.begin() + r.b + half, order.begin() + r.e, [&](int a, int b) {
        const float ca = v4[4 * (size_t)a + ax], cb = v4[4 * (size_t)b + ax];
        return ca < cb || (ca == cb && a < b);
      });
      stack.push_back({r.b, r.b + half});
      stack.push_back({r.b + half, r.e});
    }
    for (int b = 0; b < nv; b += 32) std::sort(order.begin() + b, order.begin() + std::min(nv, b + 32));   // deterministic inside a leaf
  }
  // bounding sphere of each run of 32 points (centre = AABB centre, radius rounded up)
  std::vector<float> grp((size_t)((nv + 31) / 32) * 4);
  for (int b = 0, gi = 0; b < nv; b += 32, ++gi) {
    const int e = std::min(nv, b + 32);
    double glo[3] = {1e300, 1e300, 1e300}, ghi[3] = {-1e300, -1e300, -1e300};
    for (int i = b; i < e; ++i)
      for (int k = 0; k < 3; ++k) { const double c = v4[4 * (size_t)order[i] + k]; glo[k] = std::min(glo[k], c); ghi[k] = std::max(ghi[k], c); }
    float cf[3];
    for (int k = 0; k < 3; ++k) cf[k] = (float)(0.5 * (glo[k] + ghi[k]));
    double r2 = 0.0;
    for (int i = b; i < e; ++i) {
      double d2 = 0.0;
      for (int k = 0; k < 3; ++k) { const double d = (double)v4[4 * (size_t)order[i] + k] - (double)cf[k]; d2 += d * d; }
      r2 = std::max(r2, d2);
    }
    for (int k = 0; k < 3; ++k) grp[4 * (size_t)gi + k] = cf[k];
    grp[4 * (size_t)gi + 3] = (float)(sqrt(r2) * (1.0 + 1e-6)) + 1e-12f;
  }
  std::vector<float> vs4((size_t)nv * 4), vsn4((size_t)nv * 4);
  for (int i = 0; i < nv; ++i) {
    memcpy(&vs4[4 * (size_t)i], &v4[4 * (size_t)order[i]], 16);
    memcpy(&vsn4[4 * (size_t)i], &vn4[4 * (size_t)order[i]], 16);
  }
  int rc;
  if ((rc = upload_cloud4(ctx, m.search, s4))) return rc;
  if ((rc = upload_cloud4(ctx, m.search_nrm, sn4))) return rc;
  {
    std::vector<float> raw4((size_t)nv * 4, 0.f);
    for (int k = 0; k < 3; ++k) { m.val_raw_lo[k] = INFINITY; m.val_raw_hi[k] = -INFINITY; }
    for (int i = 0; i < nv; ++i)
      for (int k = 0; k < 3; ++k) {
        raw4[4 * (size_t)i + k] = vx[3 * i + k];
        m.val_raw_lo[k] = std::min(m.val_raw_lo[k], vx[3 * i + k]); m.val_raw_hi[k] = std::max(m.val_raw_hi[k], vx[3 * i + k]);
      }
    if ((rc = upload_cloud4(ctx, m.val_raw, raw4))) return rc;
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  if ((rc = upload_cloud4(ctx, m.val_orig, v4))) return rc;
  if ((rc = upload_cloud4(ctx, m.val_nrm_orig, vn4))) return rc;
  if ((rc = upload_cloud4(ctx, m.val, vs4))) return rc;
  if ((rc = upload_cloud4(ctx, m.val_groups, grp))) return rc;
  if ((rc = upload_cloud4(ctx, m.val_nrm, vsn4))) return rc;
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the staging vectors die here
  m.ready = true;
  if (ctx->last.obj == obj) ctx->last = LastBatch();
  return PGP_OK;
}

int pgp_get_centroids(pgp_ctx* ctx, int obj, float* cP, float* cQ) {
  CHECK_CTX(ctx);
  if (cP) { if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first"); memcpy(cP, ctx->scene.cP, 12); }
  if (cQ) { Model* m = get_model(ctx, obj); if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj); memcpy(cQ, m->cQ, 12); }
  return PGP_OK;
}

// T_c = Tr(-c_P) . T . Tr(c_Q)
int pgp_pose_to_centred(pgp_ctx* ctx, int obj, const double* P, float* T) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  for (int r = 0; r < 3; ++r) {
    double t = P[4 * r + 3];
    for (int c = 0; c < 3; ++c) { T[4 * r + c] = (float)P[4 * r + c]; t += P[4 * r + c] * (double)m->cQ[c]; }
    T[4 * r + 3] = (float)(t - (double)ctx->scene.cP[r]);
  }
  return PGP_OK;
}

// camera-frame pose of a centred transform: rotation unchanged, translation t_c + c_P - R c_Q, which
// is what match4pcsBase.cc:1474-1482 builds (c1 + cP - R (c2 + cQ) with t_c = c1 - R c2).
int pgp_centred_to_pose(pgp_ctx* ctx, int obj, const float* T, double* P) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  for (int r = 0; r < 3; ++r) {
    double t = (double)T[4 * r + 3] + (double)ctx->scene.cP[r];
    for (int c = 0; c < 3; ++c) { P[4 * r + c] = (double)T[4 * r + c]; t -= (double)T[4 * r + c] * (double)m->cQ[c]; }
    P[4 * r + 3] = t;
  }
  P[12] = P[13] = P[14] = 0.0; P[15] = 1.0;
  return PGP_OK;
}

int pgp_grid_info(pgp_ctx* ctx, int* dims3, int64_t* n_cells, int64_t* n_occupied, float* cell, int64_t* bytes) {
  CHECK_CTX(ctx);
  const Scene& s = ctx->scene;
  if (!s.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (dims3) memcpy(dims3, s.g.dim, 12);
  if (n_cells) *n_cells = s.g.n_cells;
  if (n_occupied) *n_occupied = s.n_occupied;
  if (cell) *cell = s.g.h;
  if (bytes) {
    *bytes = (int64_t)s.n * 32 + (s.g.n_cells + 1) * 4 + s.bitmap_words * 4;
    if (s.g.fine) *bytes += s.bitmap_words * 8 + (int64_t)s.g.n_blocks * (128 + 128) + s.n_ambig_voxels * 8 + s.n_list_words * 16 + s.g.n_cells * 4 * s.dist_r * s.dist_r * s.dist_r;   // K1b: bmrank, codes, hdrw, adesc, arec; K1d: dist
    if (s.wlists_ready) *bytes += (int64_t)s.g.n_blocks * (2052 + 640 + 2048) + s.n_wlist_entries * 4 + (int64_t)s.n * 16;       // K1c: wvox, wbase, wcnt, wword, vrec, wlists, aux_orig
  }
  return PGP_OK;
}

int pgp_label_stats(pgp_ctx* ctx, int64_t* out8) {
  CHECK_CTX(ctx);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (!out8) return pgp_fail(ctx, PGP_E_INVALID, "null output");
  return k1_fine_stats(ctx, out8);
}

static int check_score_args(pgp_ctx* ctx, int obj, int64_t n, int mode, Model** m) {
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  *m = get_model(ctx, obj);
  if (!*m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (n < 0) return pgp_fail(ctx, PGP_E_INVALID, "negative hypothesis count");
  if (mode != PGP_LCP_COUNT && mode != PGP_LCP_WEIGHTED) return pgp_fail(ctx, PGP_E_INVALID, "unknown LCP mode %d", mode);
  if (mode == PGP_LCP_WEIGHTED && !ctx->scene.has_nrm) return pgp_fail(ctx, PGP_E_INVALID, "weighted LCP needs scene normals");
  return PGP_OK;
}

int pgp_score_lcp_dev(pgp_ctx* ctx, int obj, const float* T_dev, int64_t n, int mode, uint32_t* counts_dev, float* scores_dev) {
  CHECK_CTX(ctx);
  Model* m = nullptr;
  int rc = check_score_args(ctx, obj, n, mode, &m);
  if (rc) return rc;
  if (n > 0 && (!T_dev || !counts_dev)) return pgp_fail(ctx, PGP_E_INVALID, "null device buffer");
  if (mode == PGP_LCP_WEIGHTED && n > 0 && !scores_dev) return pgp_fail(ctx, PGP_E_INVALID, "weighted LCP needs the score buffer");
  rc = k3_score(ctx, *m, T_dev, n, mode, counts_dev, scores_dev);
  if (rc) return rc;
  ctx->last.T = T_dev; ctx->last.counts = counts_dev; ctx->last.scores = scores_dev; ctx->last.n = n; ctx->last.mode = mode; ctx->last.obj = obj;
  return PGP_OK;
}

// Host-buffer scoring, split in two so that the caller can queue more work (top-k, the all-gather) behind the scoring launch
// before it waits: pgp_score_lcp_begin enqueues upload + K3 + the downloads and returns, pgp_score_lcp_end waits for them.
// PGP_BATCH_SLOTS batches may be in flight; _end ends the oldest.
int pgp_score_lcp_begin(pgp_ctx* ctx, int obj, const float* T, int64_t n, int mode, uint32_t* counts, float* scores) {
  CHECK_CTX(ctx);
  Model* m = nullptr;
  int rc = check_score_args(ctx, obj, n, mode, &m);
  if (rc) return rc;
  if (ctx->batch_head - ctx->batch_tail >= PGP_BATCH_SLOTS)
    return pgp_fail(ctx, PGP_E_INVALID, "pgp_score_lcp_begin: %d batches are in flight already, end one first", PGP_BATCH_SLOTS);
  if (n > 0 && !T) return pgp_fail(ctx, PGP_E_INVALID, "null transforms");
  const int si = ctx->batch_head % PGP_BATCH_SLOTS;
  BatchSlot& bs = ctx->batch[si];
  bs.pending = PendingBatch();
  bs.pending.active = true; bs.pending.obj = obj; bs.pending.n = n; bs.pending.mode = mode;
  bs.pending.counts = counts; bs.pending.scores = scores;
  ctx->batch_head++;
  if (n == 0) { ctx->last = LastBatch(); return PGP_OK; }
  auto fail = [&](int code) { bs.pending.active = false; ctx->batch_head--; return code; };
  if (bs.T.reserve((size_t)n * 48) != cudaSuccess || bs.counts.reserve((size_t)n * 4) != cudaSuccess || bs.scores.reserve((size_t)n * 4) != cudaSuccess)
    return fail(pgp_fail(ctx, PGP_E_NOMEM, "cudaMalloc of a %lld-hypothesis batch failed", (long long)n));
  // Large batches are uploaded in four chunks on the copy stream while ONE scoring launch is already consuming them: the kernel
  // hands out hypotheses in index order and, before touching hypothesis h, checks a device counter that the copy engine bumps
  // after every chunk (k3_fine_kernel, LcpParams::ready).  Chunk boundaries are multiples of 8 hypotheses = 384 bytes, so no
  // 128-byte line of T spans two chunks.  Only the first chunk's upload is exposed.
  float* dT = bs.T.as<float>();
  uint32_t* dC = bs.counts.as<uint32_t>();
  float* dS = bs.scores.as<float>();
  const int chunks = 4;
  if (!ctx->pinned) { PGP_CUDA(ctx, cudaMallocHost(&ctx->pinned, 256)); ctx->pinned_cap = 256; }
  bs.marks = static_cast<uint32_t*>(ctx->pinned) + 16 * si;                     // [0] = 0, [1..4] = hypotheses uploaded after chunk c
  uint32_t* marks = bs.marks;
  marks[8] = 0;                                                                 // abort flag read back by pgp_score_lcp_end
  uint32_t* ready = reinterpret_cast<uint32_t*>(ctx->work.as<char>() + 320 + 16 * si);      // this slot's {uploaded, abort}
  const bool streamed = ctx->stream_upload && n >= 32768 && n < (1ll << 31) && k3_streams_upload(ctx, mode);
  if (streamed) {
    marks[0] = 0;
    for (int c = 0; c < chunks; ++c) marks[c + 1] = (uint32_t)(c + 1 == chunks ? n : ((n * (c + 1) / chunks) & ~7ll));
    // The upload overwrites this slot's buffers, last used by the batch TWO begins ago (its K3, and the K4 the caller queued
    // behind it): everything that was on the caller's stream at the PREVIOUS begin covers that, while the previous batch's
    // scoring launch -- the one this upload is meant to run under -- is not waited for.  With no batch in flight there is
    // nothing to overlap with and the upload simply follows everything queued so far.
    PGP_CUDA(ctx, cudaEventRecord(bs.ev_start, ctx->stream));                   // everything queued on the caller's stream so far
    const bool overlap_prev = ctx->batch_head - ctx->batch_tail >= 2;           // (head already counts this batch)
    PGP_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, overlap_prev ? ctx->batch[(si + PGP_BATCH_SLOTS - 1) % PGP_BATCH_SLOTS].ev_start : bs.ev_start, 0));
    marks[6] = 0; marks[7] = 0;
    PGP_CUDA(ctx, cudaMemcpyAsync(ready, marks + 6, 8, cudaMemcpyHostToDevice, ctx->copy_stream));      // {uploaded = 0, abort = 0}
    for (int c = 0; c < chunks; ++c) {
      const int64_t lo = marks[c], hi = marks[c + 1];
      PGP_CUDA(ctx, cudaMemcpyAsync(dT + 12 * lo, T + 12 * lo, (size_t)(hi - lo) * 48, cudaMemcpyHostToDevice, ctx->copy_stream));
      PGP_CUDA(ctx, cudaMemcpyAsync(ready, marks + c + 1, 4, cudaMemcpyHostToDevice, ctx->copy_stream));
      if (c == 0) {
        PGP_CUDA(ctx, cudaEventRecord(bs.ev_first, ctx->copy_stream));
        PGP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, bs.ev_first, 0));
        rc = k3_score(ctx, *m, dT, n, mode, dC, dS, ready);
        if (rc) return fail(rc);
      }
    }
    ctx->last.T = dT; ctx->last.counts = dC; ctx->last.scores = dS; ctx->last.n = n; ctx->last.mode = mode; ctx->last.obj = obj;
  } else {
    PGP_CUDA(ctx, cudaMemcpyAsync(dT, T, (size_t)n * 48, cudaMemcpyHostToDevice, ctx->stream));
    rc = pgp_score_lcp_dev(ctx, obj, dT, n, mode, dC, dS);
    if (rc) return fail(rc);
  }
  // downloads on their own stream (PCIe is full duplex, and the caller's stream stays free for K4 / the next batch)
  PGP_CUDA(ctx, cudaEventRecord(bs.ev_scored, ctx->stream));
  PGP_CUDA(ctx, cudaStreamWaitEvent(ctx->back_stream, bs.ev_scored, 0));
  if (streamed) PGP_CUDA(ctx, cudaMemcpyAsync(marks + 8, ready + 1, 4, cudaMemcpyDeviceToHost, ctx->back_stream));
  if (counts) PGP_CUDA(ctx, cudaMemcpyAsync(counts, dC, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->back_stream));
  if (scores) PGP_CUDA(ctx, cudaMemcpyAsync(scores, dS, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->back_stream));
  PGP_CUDA(ctx, cudaEventRecord(bs.ev_done, ctx->back_stream));                // what pgp_score_lcp_end waits for
  bs.pending.streamed = streamed;
  return PGP_OK;
}

int pgp_score_lcp_end(pgp_ctx* ctx) {
  CHECK_CTX(ctx);
  if (ctx->batch_head == ctx->batch_tail) return PGP_OK;
  BatchSlot& bs = ctx->batch[ctx->batch_tail % PGP_BATCH_SLOTS];
  ctx->batch_tail++;
  if (!bs.pending.active) return PGP_OK;
  bs.pending.active = false;
  if (bs.pending.n == 0) return PGP_OK;
  PGP_CUDA(ctx, cudaEventSynchronize(bs.ev_done));           // this batch's downloads (and with them its upload and scoring) are done
  if (bs.pending.streamed && bs.marks[8]) {
    // the kernel gave up waiting for the upload (see k3_fine_kernel); the copies are done by now: score again, plainly
    Model* m = get_model(ctx, bs.pending.obj);
    if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", bs.pending.obj);
    const int64_t n = bs.pending.n;
    uint32_t* dC = bs.counts.as<uint32_t>();
    float* dS = bs.scores.as<float>();
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    int rc = k3_score(ctx, *m, bs.T.as<float>(), n, bs.pending.mode, dC, dS, nullptr);
    if (rc) return rc;
    if (bs.pending.counts) PGP_CUDA(ctx, cudaMemcpyAsync(bs.pending.counts, dC, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (bs.pending.scores) PGP_CUDA(ctx, cudaMemcpyAsync(bs.pending.scores, dS, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->last.T = bs.T.as<float>(); ctx->last.counts = dC; ctx->last.scores = dS; ctx->last.n = n; ctx->last.mode = bs.pending.mode; ctx->last.obj = bs.pending.obj;
    return 1;        // > 0: the batch was re-scored; anything the caller queued behind the first launch (pgp_topk_begin) must be redone
  }
  return PGP_OK;
}

int pgp_score_lcp(pgp_ctx* ctx, int obj, const float* T, int64_t n, int mode, uint32_t* counts, float* scores) {
  if (!ctx) return PGP_E_INVALID;
  if (ctx->batch_head != ctx->batch_tail) return pgp_fail(ctx, PGP_E_INVALID, "pgp_score_lcp with batches of pgp_score_lcp_begin still in flight");
  int rc = pgp_score_lcp_begin(ctx, obj, T, n, mode, counts, scores);
  if (rc) return rc;
  rc = pgp_score_lcp_end(ctx);
  if (rc < 0) return rc;
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PGP_OK;
}

static int nearest_common(pgp_ctx* ctx, int obj, const float* T12, int32_t* idx_host, int gate) {
  Model* m = nullptr;
  int rc = check_score_args(ctx, obj, 1, gate ? PGP_LCP_WEIGHTED : PGP_LCP_COUNT, &m);
  if (rc) return rc;
  PGP_CUDA(ctx, ctx->topk_out.reserve((size_t)m->nv * 4 + 64));
  float* dT = ctx->topk_out.as<float>();
  int32_t* didx = reinterpret_cast<int32_t*>(ctx->topk_out.as<char>() + 64);
  PGP_CUDA(ctx, cudaMemcpyAsync(dT, T12, 48, cudaMemcpyHostToDevice, ctx->stream));
  rc = k3_nearest(ctx, *m, dT, didx, gate);
  if (rc) return rc;
  PGP_CUDA(ctx, cudaMemcpyAsync(idx_host, didx, (size_t)m->nv * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PGP_OK;
}

int pgp_nearest_in_range(pgp_ctx* ctx, int obj, const float* T12, int32_t* idx_host) {
  CHECK_CTX(ctx);
  if (!T12 || !idx_host) return pgp_fail(ctx, PGP_E_INVALID, "null argument");
  return nearest_common(ctx, obj, T12, idx_host, 0);
}

int pgp_registered_points(pgp_ctx* ctx, int obj, const float* T12, int32_t* idx_host, int cap) {
  CHECK_CTX(ctx);
  if (!T12 || !idx_host) return pgp_fail(ctx, PGP_E_INVALID, "null argument");
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  std::vector<int32_t> tmp(m->nv);
  int rc = nearest_common(ctx, obj, T12, tmp.data(), 1);
  if (rc) return rc;
  int k = 0;
  for (int i = 0; i < m->nv; ++i)
    if (tmp[i] >= 0) {
      if (k >= cap) return pgp_fail(ctx, PGP_E_CAPACITY, "more than %d registered points", cap);
      idx_host[k++] = tmp[i];
    }
  return k;
}

int pgp_topk(pgp_ctx* ctx, int obj, int k, int64_t index_base, pgp_hyp* out) {
  CHECK_CTX(ctx);
  if (pgp_comm_active(ctx)) {        // collective: K4 -> all-gather -> merge (pgp_comm.cu)
    if (k < 0 || (k > 0 && !out)) return pgp_fail(ctx, PGP_E_INVALID, "bad k / output");
    if (k == 0) return 0;
    const int t = pgp_topk_begin(ctx, obj, k, index_base);
    return t < 0 ? t : pgp_topk_end(ctx, t, out);
  }
  if (index_base == PGP_INDEX_AUTO) index_base = 0;
  if (ctx->last.obj != obj || ctx->last.n <= 0) return pgp_fail(ctx, PGP_E_NO_SCORES, "no scored batch for object %d", obj);
  if (k < 0 || (k > 0 && !out)) return pgp_fail(ctx, PGP_E_INVALID, "bad k / output");
  int n_out = 0;
  int rc = k4_topk(ctx, ctx->last, k, index_base, out, &n_out);
  return rc ? rc : n_out;
}

int pgp_topk_dev(pgp_ctx* ctx, int obj, int k, int64_t index_base, pgp_hyp* out_dev) {
  CHECK_CTX(ctx);
  if (ctx->last.obj != obj || ctx->last.n <= 0) return pgp_fail(ctx, PGP_E_NO_SCORES, "no scored batch for object %d", obj);
  if (k <= 0 || !out_dev) return pgp_fail(ctx, PGP_E_INVALID, "bad k / output");
  if (index_base == PGP_INDEX_AUTO) index_base = 0;     // a local selection, like pgp_topk without a communicator
  return k4_topk_dev(ctx, ctx->last, k, index_base, out_dev);
}

int pgp_improving_chain(pgp_ctx* ctx, int obj, int64_t index_base, pgp_hyp* out, int cap) {
  CHECK_CTX(ctx);
  if (pgp_comm_active(ctx)) return pgp_comm_improving_chain(ctx, obj, index_base, out, cap);
  if (index_base == PGP_INDEX_AUTO) index_base = 0;
  if (ctx->last.obj != obj || ctx->last.n <= 0) return pgp_fail(ctx, PGP_E_NO_SCORES, "no scored batch for object %d", obj);
  if (cap <= 0 || !out) return pgp_fail(ctx, PGP_E_INVALID, "bad capacity / output");
  int n_out = 0;
  int rc = k4_chain(ctx, ctx->last, index_base, out, cap, &n_out);
  if (rc) return rc;
  if (n_out > cap) {
    // up to 4096 candidates the kernel sorts the whole chain and writes its last cap elements; beyond that the compaction kept an
    // arbitrary subset (in atomic order), so nothing written can be used
    if (n_out > K4_MAX_K)
      return pgp_fail(ctx, PGP_E_CAPACITY, "improving chain has %d elements, more than %d: the output is unusable", n_out, K4_MAX_K);
    return pgp_fail(ctx, PGP_E_CAPACITY, "improving chain has %d elements, capacity %d (the last %d were written)", n_out, cap, cap);
  }
  return n_out;
}

// (score desc, index asc) over the concatenated lists; records with index < 0 are padding.
int pgp_topk_merge(const pgp_hyp* lists, int n_lists, int k_each, int k, pgp_hyp* out) {
  if (!lists || !out || n_lists <= 0 || k_each < 0 || k < 0) return PGP_E_INVALID;
  std::vector<const pgp_hyp*> v;
  v.reserve((size_t)n_lists * k_each);
  for (int i = 0; i < n_lists * k_each; ++i)
    if (lists[i].index >= 0) v.push_back(lists + i);
  std::sort(v.begin(), v.end(), [](const pgp_hyp* a, const pgp_hyp* b) {
    if (a->score != b->score) return a->score > b->score;
    return a->index < b->index;
  });
  int m = std::min<int>(k, (int)v.size());
  for (int i = 0; i < m; ++i) out[i] = *v[i];
  return m;
}

void pgp_pcs_default_opts(pgp_pcs_opts* o) {
  if (!o) return;
  o->n_bases = 100; o->max_quads_per_base = 100; o->max_base_diameter = -1.f; o->overlap = 0.5f; o->base_trials = 1000; o->mode = 0;
}

int pgp_extract_pairs(pgp_ctx* ctx, int obj, float dist, float eps, int32_t* pairs, int64_t cap, int64_t* n_pairs) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!n_pairs) return pgp_fail(ctx, PGP_E_INVALID, "null n_pairs");
  return k2_extract_pairs(ctx, *m, dist, eps, pairs, cap, n_pairs);
}

int pgp_find_quads(pgp_ctx* ctx, int obj, const int32_t* base4, float inv1, float inv2, float eps, const int32_t* p1, int64_t n1,
                   const int32_t* p2, int64_t n2, int32_t* quads, int64_t cap, int64_t* n_quads) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (!base4 || !n_quads || n1 < 0 || n2 < 0) return pgp_fail(ctx, PGP_E_INVALID, "bad argument");
  return k2_find_quads(ctx, *m, base4, inv1, inv2, eps, p1, n1, p2, n2, quads, cap, n_quads);
}

int pgp_find_quads_v4pcs(pgp_ctx* ctx, int obj, const int32_t* base4, float eps, int32_t* quads, int64_t cap, int64_t* n_quads) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (!base4 || !n_quads || cap < 0) return pgp_fail(ctx, PGP_E_INVALID, "bad argument");
  return k2_find_quads_v4pcs(ctx, *m, base4, eps, quads, cap, n_quads);
}

int pgp_rigid_from_quads(pgp_ctx* ctx, int obj, const int32_t* base4, const int32_t* quads, int64_t n, float* T, uint8_t* ok) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (!base4 || !quads || !T || !ok || n < 0) return pgp_fail(ctx, PGP_E_INVALID, "bad argument");
  return k2_rigid_from_quads(ctx, *m, base4, quads, n, T, ok);
}

int pgp_generate_pcs_range(pgp_ctx* ctx, int obj, const pgp_pcs_opts* opts, uint64_t seed, int base_lo, int base_hi, int64_t max_hyp, int64_t* n_hyp) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  pgp_pcs_opts o;
  if (opts) o = *opts; else pgp_pcs_default_opts(&o);
  if (!n_hyp || max_hyp <= 0) return pgp_fail(ctx, PGP_E_INVALID, "bad argument");
  const int nb = std::max(1, o.n_bases);
  if (base_lo < 0 || base_hi > nb || base_lo > base_hi) return pgp_fail(ctx, PGP_E_INVALID, "base range [%d, %d) outside [0, %d)", base_lo, base_hi, nb);
  m->gen_index_base = -1;
  return k2_generate(ctx, *m, &o, seed, base_lo, base_hi, max_hyp, n_hyp);
}

int pgp_generate_pcs(pgp_ctx* ctx, int obj, const pgp_pcs_opts* opts, uint64_t seed, int64_t max_hyp, int64_t* n_hyp) {
  const int nb = opts ? std::max(1, opts->n_bases) : 100;
  int rc = pgp_generate_pcs_range(ctx, obj, opts, seed, 0, nb, max_hyp, n_hyp);
  if (rc == PGP_OK) ctx->models[obj].gen_index_base = 0;
  return rc;
}

int pgp_score_generated(pgp_ctx* ctx, int obj, int mode) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (m->n_gen <= 0) return pgp_fail(ctx, PGP_E_NO_SCORES, "pgp_generate_pcs produced no hypotheses for object %d", obj);
  PGP_CUDA(ctx, m->gen_counts.reserve((size_t)m->n_gen * 4));
  PGP_CUDA(ctx, m->gen_scores.reserve((size_t)m->n_gen * 4));
  int rc = pgp_score_lcp_dev(ctx, obj, m->gen_T.as<float>(), m->n_gen, mode, m->gen_counts.as<uint32_t>(), m->gen_scores.as<float>());
  m->gen_scored = rc == PGP_OK;
  return rc;
}

int pgp_get_generated(pgp_ctx* ctx, int obj, float* T, uint32_t* counts, float* scores, int64_t cap) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  int64_t n = std::min<int64_t>(cap, m->n_gen);
  if (n > 0) {
    if (T) PGP_CUDA(ctx, cudaMemcpyAsync(T, m->gen_T.p, (size_t)n * 48, cudaMemcpyDeviceToHost, ctx->stream));
    if (counts && m->gen_scored) PGP_CUDA(ctx, cudaMemcpyAsync(counts, m->gen_counts.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (scores && m->gen_scored) PGP_CUDA(ctx, cudaMemcpyAsync(scores, m->gen_scores.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return (int)std::min<int64_t>(n, 0x7fffffff);
}

int pgp_set_ppf_map(pgp_ctx* ctx, int obj, const int32_t* keys4, const int64_t* offsets, const int32_t* pairs, int64_t n_keys) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (n_keys < 0 || (n_keys > 0 && (!keys4 || !offsets || !pairs))) return pgp_fail(ctx, PGP_E_INVALID, "bad PPF map");
  return k2_set_ppf_map(ctx, *m, keys4, offsets, pairs, n_keys);
}

int pgp_build_ppf_map(pgp_ctx* ctx, int obj) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  return k2_build_ppf_map(ctx, *m);
}

int pgp_get_ppf_map(pgp_ctx* ctx, int obj, int32_t* keys4, int64_t cap_keys, int64_t* offsets, int32_t* pairs, int64_t cap_pairs,
                    int64_t* n_keys, int64_t* n_pairs) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (n_keys) *n_keys = m->n_ppf_keys;
  if (n_pairs) *n_pairs = m->n_ppf_pairs;
  const int64_t nk = std::min<int64_t>(cap_keys, m->n_ppf_keys);
  for (int64_t k = 0; k < nk; ++k) {
    const uint32_t pk = m->h_ppf_keys[k];
    if (keys4) { keys4[4 * k] = (int32_t)(pk >> 15) * 5; keys4[4 * k + 1] = (int32_t)((pk >> 10) & 31) * 10; keys4[4 * k + 2] = (int32_t)((pk >> 5) & 31) * 10; keys4[4 * k + 3] = (int32_t)(pk & 31) * 10; }
    if (offsets) { offsets[k] = m->h_ppf_offsets[k]; offsets[k + 1] = m->h_ppf_offsets[k + 1]; }
  }
  if (pairs) memcpy(pairs, m->h_ppf_pairs.data(), (size_t)std::min<int64_t>(cap_pairs, m->n_ppf_pairs) * 8);
  return PGP_OK;
}

int pgp_scene_ppf_keys(pgp_ctx* ctx, const int32_t* pairs, int64_t n, int32_t* keys4) {
  CHECK_CTX(ctx);
  if (!ctx->scene.ready) return pgp_fail(ctx, PGP_E_NO_SCENE, "pgp_set_scene first");
  if (n < 0 || (n > 0 && (!pairs || !keys4))) return pgp_fail(ctx, PGP_E_INVALID, "null argument");
  return k2_scene_ppf_keys(ctx, pairs, n, keys4);
}

uint32_t pgp_stocs_engine_seed(uint64_t seed, int base, int attempt) { return k2_stocs_engine_seed(seed, base, attempt); }

int pgp_get_bases(pgp_ctx* ctx, int obj, int32_t* ids, float* inv, uint8_t* ok, int cap) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!ids || !inv || !ok) return pgp_fail(ctx, PGP_E_INVALID, "null output");
  const int n = std::min(cap, m->n_gen_bases);
  if (n <= 0) return 0;
  int rc = k2_get_bases(ctx, *m, n, ids, inv, ok);
  return rc ? rc : n;
}

// trimmed ICP inputs: every segment coordinate and every pose entry finite
static bool tricp_inputs_finite(const float* seg, int ns, const double* poses, int k) {
  for (size_t i = 0; i < (size_t)ns * 3; ++i) if (!std::isfinite(seg[i])) return false;
  for (size_t i = 0; i < (size_t)k * 16; ++i) if (!std::isfinite(poses[i])) return false;
  return true;
}

int pgp_tricp(pgp_ctx* ctx, int obj, const float* seg, int ns, double* poses, int k, float trim, float ratio, int max_iter, int* iters, float* energy) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!seg || ns <= 0 || !poses || k < 0) return pgp_fail(ctx, PGP_E_INVALID, "bad argument");
  if (!(trim > 0.f) || !(ratio > 0.f)) return pgp_fail(ctx, PGP_E_INVALID, "pgp_tricp: trim and ratio must be > 0");
  if (!tricp_inputs_finite(seg, ns, poses, k)) return pgp_fail(ctx, PGP_E_INVALID, "pgp_tricp: non-finite segment point or pose");
  if (k == 0) return PGP_OK;
  return k5_tricp(ctx, *m, seg, ns, poses, k, trim, ratio, max_iter, iters, energy);
}

}  // extern "C"

int pgp_remove_explained(pgp_ctx* ctx, int obj, const float* seg, int ns, const double* placed16, int n_placed, float threshold, uint8_t* explained) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (ns < 0 || n_placed < 0 || (ns > 0 && (!seg || !explained)) || (n_placed > 0 && !placed16) || !(threshold >= 0.f))
    return pgp_fail(ctx, PGP_E_INVALID, "pgp_remove_explained: bad argument");
  int kept = 0;
  int rc = k6_remove_explained(ctx, *m, seg, ns, placed16, n_placed, threshold, explained, &kept);
  return rc ? rc : kept;
}

int pgp_mcts_tricp(pgp_ctx* ctx, int obj, const float* seg, int ns, const double* placed16, int n_placed, float threshold, double* poses, int k,
                   float trim, float ratio, int max_iter, int* iters, float* energy, int* n_unexplained) {
  CHECK_CTX(ctx);
  Model* m = get_model(ctx, obj);
  if (!m) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  if (!seg || ns <= 0 || !poses || k <= 0) return pgp_fail(ctx, PGP_E_INVALID, "pgp_mcts_tricp: empty input");
  if (!(trim > 0.f) || !(ratio > 0.f)) return pgp_fail(ctx, PGP_E_INVALID, "pgp_mcts_tricp: trim and ratio must be > 0");
  if (!tricp_inputs_finite(seg, ns, poses, k)) return pgp_fail(ctx, PGP_E_INVALID, "pgp_mcts_tricp: non-finite segment point or pose");
  std::vector<uint8_t> flag((size_t)ns, 0);
  int kept = ns;
  if (n_placed > 0) {
    int rc = k6_remove_explained(ctx, *m, seg, ns, placed16, n_placed, threshold, flag.data(), &kept);
    if (rc) return rc;
  }
  std::vector<float> un((size_t)std::max(kept, 1) * 3);
  int w = 0;
  for (int i = 0; i < ns; ++i)                       // extract.setNegative(true): the survivors in their original order
    if (!flag[i]) { memcpy(&un[3 * (size_t)w], seg + 3 * (size_t)i, 12); ++w; }
  if (n_unexplained) *n_unexplained = kept;
  if (kept == 0) { for (int i = 0; i < k; ++i) { if (iters) iters[i] = 0; if (energy) energy[i] = 0.f; } return PGP_OK; }
  return k5_tricp(ctx, *m, un.data(), kept, poses, k, trim, ratio, max_iter, iters, energy);
}

int pgp_prepare_segment(pgp_ctx* ctx, const uint16_t* depth_raw, const uint8_t* class_mask, int rows, int cols, int class_id, const float* K9,
                        float leaf, float normal_radius, float outlier_radius, int min_neighbors, float* xyz_out, float* nrm_out, int cap,
                        int* n_valid_pixels) {
  CHECK_CTX(ctx);
  if (!depth_raw || !class_mask || rows <= 0 || cols <= 0 || !K9 || !xyz_out || !nrm_out || cap < 0)
    return pgp_fail(ctx, PGP_E_INVALID, "pgp_prepare_segment: bad argument");
  if (!(leaf > 0.f) || !(normal_radius > 0.f) || !(outlier_radius > 0.f) || !(K9[0] != 0.f) || !(K9[4] != 0.f))
    return pgp_fail(ctx, PGP_E_INVALID, "pgp_prepare_segment: leaf, radii and focal lengths must be non-zero");
  if ((double)normal_radius / leaf > 16.0 || (double)outlier_radius / leaf > 16.0)
    return pgp_fail(ctx, PGP_E_INVALID, "pgp_prepare_segment: radius / leaf > 16");
  int n = 0;
  int rc = k7_prepare_segment(ctx, depth_raw, class_mask, rows, cols, class_id, K9, leaf, normal_radius, outlier_radius, min_neighbors, xyz_out, nrm_out,
                              cap, &n, n_valid_pixels);
  return rc ? rc : n;
}
