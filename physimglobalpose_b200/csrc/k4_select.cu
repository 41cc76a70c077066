// K4 -- selection over a scored batch: top-k and the strictly-improving chain.
//
// Replaces the serial best-so-far scan of Perform_N_steps (S4/algorithms/match4pcsBase.cc:1888-1901)
// and the result shaping of :1903-1914 / ComputeTransformation :1787-1796.
//
// Order: (score desc, generation index asc).  The pair is packed into ONE unique 64-bit key
//   key = key32(score) << ibits | (n - 1 - i)
// where key32 is the count itself (COUNT mode) or the fp32 score mapped to an unsigned integer of the same order
// (WEIGHTED mode, float_key below: negative scores rank below +0, -0 ties with +0), so "top-k" = the k largest
// keys; an MSB-first radix select (11-bit digits) finds the k-th key exactly, a compaction gathers the k
// survivors, one CTA sorts them.  Everything runs in ONE cooperative launch (one CTA per SM, software grid
// barrier between the passes), because at the benchmark size the whole selection is a few hundred KB of L2
// reads and would otherwise be launch-latency bound.
#include <algorithm>
#include <math.h>

#include "pgp_internal.cuh"

namespace {

constexpr int ST = 1024;          // threads per CTA
constexpr int DIGIT = 11;
constexpr int BINS = 1 << DIGIT;
constexpr int MAX_PASSES = 6;
constexpr int KMAX = K4_MAX_K;

struct SelParams {
  const uint32_t* key32;     // counts, or the bits of the fp32 scores (float_keys: mapped by float_key before any comparison)
  bool float_keys;
  const float* scores;       // may be null
  const uint32_t* counts;    // may be null
  const float* T;
  long long n;
  int nv;
  int k;
  int ibits, kbits;
  long long index_base;
  uint32_t* hist;            // MAX_PASSES x BINS, zeroed before launch
  unsigned* barrier;         // zeroed before launch
  unsigned* n_cand;          // zeroed before launch
  unsigned long long* cand;  // KMAX keys
  pgp_hyp* out;              // device, k records
  pgp_hyp* hdr;              // may be null: one more record {index = batch size, count = records written} in front of the k
                             // records, for the multi-GPU exchange (pgp_comm.cu)
  int* n_out;
  int mode;                  // 0: top-k, 1: improving chain
  unsigned long long* seg_max;   // chain: per-CTA segment maxima
};

__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned& epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(bar, 1u);
    const unsigned target = (epoch + 1) * gridDim.x;
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
    } while (v < target);
  }
  epoch++;
  __syncthreads();
}

// fp32 bits -> unsigned key with the order of the float values.  Priors may be negative (pgp_set_scene_priors), so a weighted score
// may be too: -0 is folded into +0 (they compare equal, the index decides), negative values are bit-inverted (below 0x80000000, the
// more negative the smaller), non-negative ones get the top bit set.
__device__ __forceinline__ uint32_t float_key(uint32_t bits) {
  const uint32_t u = bits == 0x80000000u ? 0u : bits;
  return (u >> 31) ? ~u : (u | 0x80000000u);
}
constexpr uint32_t FLOAT_KEY_ZERO = 0x80000000u;   // float_key(+0.f)

__device__ __forceinline__ uint32_t key32_at(const SelParams& p, long long i) {
  const uint32_t v = p.key32[i];
  return p.float_keys ? float_key(v) : v;
}

__device__ __forceinline__ unsigned long long make_key(const SelParams& p, long long i) {
  return ((unsigned long long)key32_at(p, i) << p.ibits) | (unsigned long long)(p.n - 1 - i);
}

__device__ void write_record(const SelParams& p, int slot, unsigned long long key) {
  long long i = p.n - 1 - (long long)(key & ((1ull << p.ibits) - 1ull));
  pgp_hyp r;
  r.index = i + p.index_base;
  r.count = p.counts ? p.counts[i] : 0u;
  r.score = p.scores ? p.scores[i] : __fdiv_rn((float)r.count, (float)p.nv);
#pragma unroll
  for (int c = 0; c < 12; ++c) r.T[c] = p.T[12 * i + c];
  p.out[slot] = r;
}

// sorts m (<= KMAX) keys held in shared memory, descending
__device__ void bitonic_desc(unsigned long long* s, int m_pow2) {
  for (int k = 2; k <= m_pow2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < m_pow2; t += blockDim.x) {
        int ixj = t ^ j;
        if (ixj > t) {
          unsigned long long a = s[t], b = s[ixj];
          bool up = (t & k) == 0;      // descending overall
          if (up ? (a < b) : (a > b)) { s[t] = b; s[ixj] = a; }
        }
      }
      __syncthreads();
    }
}

__global__ void __launch_bounds__(ST, 1) k4_select_kernel(const SelParams p) {
  __shared__ uint32_t s_hist[BINS];
  __shared__ unsigned long long s_keys[KMAX];
  __shared__ unsigned long long s_prefix;
  __shared__ int s_kk;
  unsigned epoch = 0;
  const long long stride = (long long)gridDim.x * ST;
  const long long tid = (long long)blockIdx.x * ST + threadIdx.x;
  const int total_bits = p.ibits + p.kbits;
  const int passes = (total_bits + DIGIT - 1) / DIGIT;

  if (p.mode == 0) {
    const int k = (int)min((long long)p.k, p.n);
    unsigned long long prefix = 0;   // the decided high bits of the k-th largest key
    int kk = k;                      // rank still to find inside the prefix bucket
    int hi = total_bits;             // bits [hi, total_bits) are decided
    for (int pass = 0; pass < passes; ++pass) {
      const int lo = max(hi - DIGIT, 0);
      const int nb = 1 << (hi - lo);
      for (int b = threadIdx.x; b < BINS; b += ST) s_hist[b] = 0;
      __syncthreads();
      for (long long i = tid; i < p.n; i += stride) {
        unsigned long long key = make_key(p, i);
        if ((key >> hi) == prefix) atomicAdd(&s_hist[(unsigned)(key >> lo) & (nb - 1)], 1u);
      }
      __syncthreads();
      uint32_t* gh = p.hist + pass * BINS;
      for (int b = threadIdx.x; b < nb; b += ST) { uint32_t v = s_hist[b]; if (v) atomicAdd(gh + b, v); }
      grid_barrier(p.barrier, epoch);
      // every CTA finds the digit of the k-th largest key: scan bins from the top
      for (int b = threadIdx.x; b < nb; b += ST) s_hist[b] = __ldcg(gh + b);
      __syncthreads();
      if (threadIdx.x < 32) {
        // warp-cooperative descending scan over nb bins
        int remaining = kk, found = -1, found_rem = 0;
        for (int top = nb - 1; top >= 0 && found < 0; top -= 32) {
          int b = top - (int)threadIdx.x;
          uint32_t v = b >= 0 ? s_hist[b] : 0u;
          uint32_t incl = v;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += t; }
          unsigned hit = __ballot_sync(0xffffffffu, incl >= (uint32_t)remaining);
          if (hit) {
            int l = __ffs(hit) - 1;
            found = top - l;
            uint32_t before = __shfl_sync(0xffffffffu, incl - v, l);
            found_rem = remaining - (int)before;
          } else {
            remaining -= (int)__shfl_sync(0xffffffffu, incl, 31);
          }
        }
        if (threadIdx.x == 0) { s_prefix = (prefix << (hi - lo)) | (unsigned long long)max(found, 0); s_kk = found_rem; }
      }
      __syncthreads();
      prefix = s_prefix; kk = s_kk; hi = lo;
      __syncthreads();
    }
    // prefix is now the k-th largest key itself
    const unsigned long long tau = prefix;
    if (k > 0)
      for (long long i = tid; i < p.n; i += stride) {
        unsigned long long key = make_key(p, i);
        if (key >= tau) { unsigned pos = atomicAdd(p.n_cand, 1u); if (pos < KMAX) p.cand[pos] = key; }
      }
    grid_barrier(p.barrier, epoch);
    if (blockIdx.x == 0) {
      int m = 1; while (m < k) m <<= 1;
      for (int t = threadIdx.x; t < m; t += ST) s_keys[t] = t < k ? __ldcg(p.cand + t) : 0ull;
      __syncthreads();
      bitonic_desc(s_keys, m);
      for (int t = threadIdx.x; t < k; t += ST) write_record(p, t, s_keys[t]);
      for (int t = k + threadIdx.x; t < p.k; t += ST) {      // pad: the merge skips index < 0
        pgp_hyp r;
        r.index = -1; r.count = 0; r.score = 0.f;
#pragma unroll
        for (int c = 0; c < 12; ++c) r.T[c] = 0.f;
        p.out[t] = r;
      }
      if (threadIdx.x == 0) {
        *p.n_out = k;
        if (p.hdr) { pgp_hyp r{}; r.index = p.n; r.count = (uint32_t)k; *p.hdr = r; }
      }
    }
  } else {
    // improving chain: i is kept iff key32[i] > max(key32[0..i)) and score i > 0 (best_LCP_ starts at 0, strict '>' at
    // match4pcsBase.cc:1891: a score <= 0 never enters, a later positive one still does).  Contiguous segment per CTA.
    const uint32_t floor = p.float_keys ? FLOAT_KEY_ZERO : 0u;
    const long long seg = (p.n + gridDim.x - 1) / gridDim.x;
    const long long s0 = min(p.n, seg * blockIdx.x), s1 = min(p.n, s0 + seg);
    uint32_t* s_max = s_hist;     // reuse
    uint32_t mx = 0;
    for (long long i = s0 + threadIdx.x; i < s1; i += ST) mx = max(mx, key32_at(p, i));
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t m = 0;
      for (int w = 0; w < ST / 32; ++w) m = max(m, s_max[w]);
      p.seg_max[blockIdx.x] = m;
    }
    grid_barrier(p.barrier, epoch);
    uint32_t run = 0;
    for (int b = 0; b < (int)blockIdx.x; ++b) run = max(run, (uint32_t)__ldcg(p.seg_max + b));
    // inside the segment: chunks of ST elements, block-wide exclusive max-scan per chunk
    for (long long c0 = s0; c0 < s1; c0 += ST) {
      long long i = c0 + threadIdx.x;
      uint32_t v = i < s1 ? key32_at(p, i) : 0u;
      uint32_t incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((threadIdx.x & 31) >= o) incl = max(incl, t); }
      uint32_t excl = __shfl_up_sync(0xffffffffu, incl, 1);
      if ((threadIdx.x & 31) == 0) excl = 0;
      __syncthreads();
      if ((threadIdx.x & 31) == 31) s_max[threadIdx.x >> 5] = incl;
      __syncthreads();
      uint32_t before = run, chunk = 0;
      for (int w = 0; w < ST / 32; ++w) { uint32_t t = s_max[w]; if (w < (int)(threadIdx.x >> 5)) before = max(before, t); chunk = max(chunk, t); }
      before = max(max(before, excl), floor);
      if (i < s1 && v > before) {
        unsigned pos = atomicAdd(p.n_cand, 1u);
        if (pos < KMAX) p.cand[pos] = make_key(p, i);
      }
      run = max(run, chunk);
    }
    grid_barrier(p.barrier, epoch);
    if (blockIdx.x == 0) {
      const int cnt = (int)min((unsigned)KMAX, (unsigned)__ldcg(p.n_cand));
      int m = 1; while (m < cnt) m <<= 1;
      for (int t = threadIdx.x; t < m; t += ST) s_keys[t] = t < cnt ? __ldcg(p.cand + t) : 0ull;
      __syncthreads();
      bitonic_desc(s_keys, m);      // descending score == descending index along a chain
      const int keep = min(cnt, p.k);
      // generation order = ascending: reverse; if the chain is longer than the capacity keep its tail (the best)
      for (int t = threadIdx.x; t < keep; t += ST) write_record(p, keep - 1 - t, s_keys[t]);
      if (threadIdx.x == 0) {
        *p.n_out = (int)__ldcg(p.n_cand);
        if (p.hdr) { pgp_hyp r{}; r.index = p.n; r.count = (uint32_t)keep; r.score = __ldcg(p.n_cand) > (unsigned)p.k ? 1.f : 0.f; *p.hdr = r; }   // score = 1: chain overflowed the capacity
      }
    }
  }
}

int bits_for(unsigned long long v) { int b = 1; while (b < 64 && (v >> b)) ++b; return b; }

int run_select(pgp_ctx* ctx, const LastBatch& b, int k, int64_t index_base, pgp_hyp* out_host, int mode, int* n_out, pgp_hyp* out_dev = nullptr,
               pgp_hyp* hdr_dev = nullptr) {
  if (n_out) *n_out = 0;
  if (b.n <= 0 || k <= 0) return PGP_OK;
  if (k > KMAX) return pgp_fail(ctx, PGP_E_INVALID, "k = %d exceeds %d", k, KMAX);
  if (b.n > (1ll << 40)) return pgp_fail(ctx, PGP_E_INVALID, "batch too large for selection");
  const Model& m = ctx->models[b.obj];
  const bool binary_weight = (b.mode == PGP_LCP_WEIGHTED) && ctx->scene.priors_binary;
  SelParams p{};
  p.counts = b.counts; p.scores = b.scores; p.T = b.T; p.n = b.n; p.nv = m.nv;
  p.k = k; p.index_base = index_base; p.mode = mode;
  p.ibits = bits_for((unsigned long long)(b.n - 1));
  if (b.mode == PGP_LCP_COUNT) { p.key32 = b.counts; p.kbits = bits_for((unsigned long long)m.nv); }
  else {
    if (!b.scores) return pgp_fail(ctx, PGP_E_NO_SCORES, "weighted selection needs the score array");
    p.key32 = reinterpret_cast<const uint32_t*>(b.scores); p.kbits = 32; p.float_keys = true;
  }
  (void)binary_weight;
  if (p.ibits + p.kbits > 63) return pgp_fail(ctx, PGP_E_INVALID, "batch too large for a 64-bit selection key");
  const size_t off_hist = 2048, off_bar = off_hist + (size_t)MAX_PASSES * BINS * 4, off_ncand = off_bar + 64, off_nout = off_ncand + 64,
               off_cand = off_nout + 64, off_seg = off_cand + (size_t)KMAX * 8, off_out = off_seg + 8 * 1024, total = off_out + (size_t)KMAX * sizeof(pgp_hyp);
  static_assert(2048 + (size_t)MAX_PASSES * BINS * 4 + 3 * 64 + (size_t)KMAX * 8 + 8 * 1024 + (size_t)KMAX * sizeof(pgp_hyp) <= PGP_WORK_BYTES, "K4 scratch exceeds pgp_ctx::work");
  if (total > ctx->work.cap) return pgp_fail(ctx, PGP_E_NOMEM, "selection scratch (%zu bytes) exceeds the work buffer", total);
  char* w = ctx->work.as<char>();
  p.hist = reinterpret_cast<uint32_t*>(w + off_hist);
  p.barrier = reinterpret_cast<unsigned*>(w + off_bar);
  p.n_cand = reinterpret_cast<unsigned*>(w + off_ncand);
  p.n_out = reinterpret_cast<int*>(w + off_nout);
  p.cand = reinterpret_cast<unsigned long long*>(w + off_cand);
  p.seg_max = reinterpret_cast<unsigned long long*>(w + off_seg);
  p.out = out_dev ? out_dev : reinterpret_cast<pgp_hyp*>(w + off_out);
  p.hdr = hdr_dev;
  PGP_CUDA(ctx, cudaMemsetAsync(w + off_hist, 0, off_cand - off_hist, ctx->stream));
  int grid = (int)std::min<long long>(ctx->sm_count, (b.n + ST - 1) / ST);
  if (grid > 1024) grid = 1024;
  void* args[] = {(void*)&p};
  PGP_CUDA(ctx, cudaLaunchCooperativeKernel((const void*)k4_select_kernel, dim3(grid), dim3(ST), args, 0, ctx->stream));
  ctx->launches++;
  PGP_CUDA(ctx, cudaGetLastError());
  if (out_dev) return PGP_OK;      // asynchronous: the records stay on the device (e.g. an NCCL send buffer)
  int n_found = 0;
  PGP_CUDA(ctx, cudaMemcpyAsync(&n_found, p.n_out, 4, cudaMemcpyDeviceToHost, ctx->stream));
  PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  int n_copy = std::min(n_found, k);
  if (n_copy > 0) PGP_CUDA(ctx, cudaMemcpy(out_host, p.out, (size_t)n_copy * sizeof(pgp_hyp), cudaMemcpyDeviceToHost));
  *n_out = n_found;
  return PGP_OK;
}

}  // namespace

int k4_topk(pgp_ctx* ctx, const LastBatch& b, int k, int64_t index_base, pgp_hyp* out_host, int* n_out) {
  return run_select(ctx, b, k, index_base, out_host, 0, n_out);
}
int k4_topk_dev(pgp_ctx* ctx, const LastBatch& b, int k, int64_t index_base, pgp_hyp* out_dev) {
  return run_select(ctx, b, k, index_base, nullptr, 0, nullptr, out_dev);
}
int k4_chain(pgp_ctx* ctx, const LastBatch& b, int64_t index_base, pgp_hyp* out_host, int cap, int* n_out) {
  return run_select(ctx, b, cap, index_base, out_host, 1, n_out);
}
// asynchronous: header record + k records into device memory (the send buffer of the multi-GPU exchange); mode 0 = top-k, 1 = chain
int k4_select_dev(pgp_ctx* ctx, const LastBatch& b, int k, int64_t index_base, int mode, pgp_hyp* hdr_dev, pgp_hyp* out_dev) {
  return run_select(ctx, b, k, index_base, nullptr, mode, nullptr, out_dev, hdr_dev);
}
