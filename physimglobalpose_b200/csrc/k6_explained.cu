// K6 -- explained-point removal before the per-node trimmed ICP of the MCTS search.
//
// UCTState::performTrICP (PPE/src/hypothesis_verification/mcts/UCTState.cpp:121-204): before an object's pose is refined
// against its segment, every segment point within pointRemovalThreshold (8 mm, UCTSearch.cpp) of the objects ALREADY PLACED
// is dropped (:149-174).  The reference builds the "explained" cloud by transforming the CURRENT object's model cloud with
// each placed object's pose (sic, :150-155: pcl::transformPointCloud in float) and runs one FLANN radius search per segment
// point.  Here: the same transformed cloud (fp32, row-wise left to right like pcl::transformPointCloud), then an exact
// all-pairs sweep over shared-memory tiles -- segment x explained is at most a few 10^8 distance tests, and it keeps the
// reference's arithmetic (squared distance summed left to right, strict d2 < r^2 as FLANN's radius result set).
// RESTATED, PARITY UNPINNED: PCL / FLANN are not vendored in the reference tree (SURVEY.md 8c); the CPU restatement the tests
// check this against is lo_remove_explained in the test infrastructure.
#include "pgp_internal.cuh"

namespace {

__global__ void k6_transform(const float4* __restrict__ model, int nv, const float* __restrict__ T12, int n_placed, float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nv * n_placed) return;
  const float* T = T12 + 12 * (i / nv);
  const float4 p = model[i % nv];
  out[i] = make_float4(xf_row(T[0], T[1], T[2], T[3], p.x, p.y, p.z), xf_row(T[4], T[5], T[6], T[7], p.x, p.y, p.z),
                       xf_row(T[8], T[9], T[10], T[11], p.x, p.y, p.z), 0.f);
}

// whether any of the m tile points lies strictly within r of s
__device__ __forceinline__ bool tile_hit(const float4 s, const float4* tile, int m, float r2) {
  for (int t = 0; t < m; ++t) {
    const float4 q = tile[t];
    const float dx = __fsub_rn(s.x, q.x), dy = __fsub_rn(s.y, q.y), dz = __fsub_rn(s.z, q.z);
    const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));   // L2_Simple: left to right
    if (d2 < r2) return true;
  }
  return false;
}

__global__ void __launch_bounds__(K6_T) k6_mark(const float4* __restrict__ seg, int ns, const float4* __restrict__ expl, int ne, float r2,
                                                uint8_t* __restrict__ flag) {
  __shared__ float4 tile[K6_T];
  const int i = blockIdx.x * K6_T + threadIdx.x;
  const float4 s = i < ns ? seg[i] : make_float4(0, 0, 0, 0);
  bool hit = false;
  for (int j0 = 0; j0 < ne; j0 += K6_T) {
    __syncthreads();
    if (j0 + (int)threadIdx.x < ne) tile[threadIdx.x] = expl[j0 + threadIdx.x];
    __syncthreads();
    if (__syncthreads_and(hit || i >= ns)) break;          // the whole CTA is done
    if (!hit && i < ns) hit = tile_hit(s, tile, min(K6_T, ne - j0), r2);
  }
  if (i < ns) flag[i] = hit ? 1 : 0;
}

// k6_mark for many (segment, placed set) jobs at once.  The explained cloud is not materialised: the tile loader transforms the
// model point with k6_transform's arithmetic, in k6_transform's order (placed row major, model point minor), so every job gets
// the flags k6_mark gives it.
__global__ void __launch_bounds__(K6_T) k6_mark_batch(const float4* __restrict__ seg, const K6Dev* __restrict__ jobs, int n_jobs,
                                                      const float* __restrict__ T12, float r2, uint8_t* __restrict__ flag) {
  __shared__ float4 tile[K6_T];
  int lo = 0, hi = n_jobs - 1;                               // last job whose first block is <= this one
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (jobs[mid].block_lo <= (int64_t)blockIdx.x) lo = mid; else hi = mid - 1; }
  const K6Dev J = jobs[lo];
  const int i = (int)(blockIdx.x - J.block_lo) * K6_T + threadIdx.x;
  const float4 s = i < J.ns ? seg[J.seg_lo + i] : make_float4(0, 0, 0, 0);
  const int64_t ne = (int64_t)J.nv * J.n_placed;
  bool hit = false;
  for (int64_t j0 = 0; j0 < ne; j0 += K6_T) {
    __syncthreads();
    const int64_t j = j0 + threadIdx.x;
    if (j < ne) {
      const float* T = T12 + 12 * (J.placed_lo + j / J.nv);
      const float4 p = J.model[j % J.nv];
      tile[threadIdx.x] = make_float4(xf_row(T[0], T[1], T[2], T[3], p.x, p.y, p.z), xf_row(T[4], T[5], T[6], T[7], p.x, p.y, p.z),
                                      xf_row(T[8], T[9], T[10], T[11], p.x, p.y, p.z), 0.f);
    }
    __syncthreads();
    if (__syncthreads_and(hit || i >= J.ns)) break;        // the whole CTA is done
    if (!hit && i < J.ns) hit = tile_hit(s, tile, (int)min((int64_t)K6_T, ne - j0), r2);
  }
  if (i < J.ns) flag[J.flag_lo + i] = hit ? 1 : 0;
}

// owned by the context, released by k6_release (pgp_destroy)
struct K6Scratch { DevBuf seg, expl, T, flag; };
K6Scratch& k6_scratch_of(pgp_ctx* ctx) {
  if (!ctx->k6_scratch) ctx->k6_scratch = new K6Scratch();
  return *static_cast<K6Scratch*>(ctx->k6_scratch);
}

}  // namespace

// flags_host[i] = 1 when segment point i is explained by a placed object.  Returns the number of UNEXPLAINED points.
int k6_remove_explained(pgp_ctx* ctx, Model& m, const float* seg_xyz_host, int ns, const double* placed16_host, int n_placed, float threshold,
                        uint8_t* flags_host, int* n_unexplained) {
  K6Scratch& sc = k6_scratch_of(ctx);
  *n_unexplained = ns;
  if (ns <= 0) return PGP_OK;
  if (n_placed <= 0) { memset(flags_host, 0, (size_t)ns); return PGP_OK; }
  cudaStream_t st = ctx->stream;
  std::vector<float> seg4((size_t)ns * 4, 0.f), T((size_t)n_placed * 12);
  for (int i = 0; i < ns; ++i) for (int c = 0; c < 3; ++c) seg4[4 * (size_t)i + c] = seg_xyz_host[3 * i + c];
  for (int k = 0; k < n_placed; ++k) pose16_to_f32x12(placed16_host + 16 * (size_t)k, &T[12 * (size_t)k]);
  const int ne = m.nv * n_placed;
  PGP_CUDA(ctx, sc.seg.reserve((size_t)ns * 16));
  PGP_CUDA(ctx, sc.expl.reserve((size_t)ne * 16));
  PGP_CUDA(ctx, sc.T.reserve((size_t)n_placed * 48));
  PGP_CUDA(ctx, sc.flag.reserve((size_t)ns));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.seg.p, seg4.data(), (size_t)ns * 16, cudaMemcpyHostToDevice, st));
  PGP_CUDA(ctx, cudaMemcpyAsync(sc.T.p, T.data(), (size_t)n_placed * 48, cudaMemcpyHostToDevice, st));
  k6_transform<<<(ne + 255) / 256, 256, 0, st>>>(m.val_raw.as<float4>(), m.nv, sc.T.as<float>(), n_placed, sc.expl.as<float4>());
  k6_mark<<<(ns + K6_T - 1) / K6_T, K6_T, 0, st>>>(sc.seg.as<float4>(), ns, sc.expl.as<float4>(), ne, threshold * threshold, sc.flag.as<uint8_t>());
  ctx->launches += 2;
  PGP_CUDA(ctx, cudaGetLastError());
  PGP_CUDA(ctx, cudaMemcpyAsync(flags_host, sc.flag.p, (size_t)ns, cudaMemcpyDeviceToHost, st));
  PGP_CUDA(ctx, cudaStreamSynchronize(st));
  int kept = 0;
  for (int i = 0; i < ns; ++i) kept += flags_host[i] ? 0 : 1;
  *n_unexplained = kept;
  return PGP_OK;
}

int k6_mark_batch_dev(pgp_ctx* ctx, const float4* seg4, const K6Dev* jobs_dev, int n_jobs, int64_t n_blocks, const float* T12, float threshold,
                      uint8_t* flags_dev) {
  if (n_blocks == 0) return PGP_OK;                          // (pgp_refine_batch bounds the flags, so n_blocks < 2^31)
  k6_mark_batch<<<(unsigned)n_blocks, K6_T, 0, ctx->stream>>>(seg4, jobs_dev, n_jobs, T12, threshold * threshold, flags_dev);
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  return PGP_OK;
}

int k6_compact(const float* seg_xyz_host, int ns, const uint8_t* flags, float* out_xyz) {
  int w = 0;
  for (int i = 0; i < ns; ++i)
    if (!flags[i]) { memcpy(out_xyz + 3 * (size_t)w, seg_xyz_host + 3 * (size_t)i, 12); ++w; }
  return w;
}

void k6_release(pgp_ctx* ctx) {
  if (!ctx->k6_scratch) return;
  K6Scratch* sc = static_cast<K6Scratch*>(ctx->k6_scratch);
  for (DevBuf* b : {&sc->seg, &sc->expl, &sc->T, &sc->flag}) b->release();
  delete sc;
  ctx->k6_scratch = nullptr;
}
