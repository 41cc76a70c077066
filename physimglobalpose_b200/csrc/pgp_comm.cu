// Multi-GPU layer of the C ABI (SURVEY.md 8(b)/(e)): hypotheses -- or, for generated requests, bases -- shard across the GPUs of one
// box, the scene grid and the models are replicated, and the ONLY exchange on the path is the all-gather of the per-GPU selection
// records (header + k x 64 bytes per GPU) after K4, followed by a deterministic merge whose result does not depend on the number
// of GPUs.  The reference has no counterpart (one thread: S4/algorithms/match4pcsBase.cc:1855-1877 per base, :1888-1901 per
// hypothesis, PPE/src/data_layer/SceneCfg.cpp:379-390 per object); the contract kept is that the merged top-k / improving chain
// equal what the serial scan over the concatenated hypothesis list returns.
//
// Two process models:
//   * one process per GPU (torchrun, MPI ...): pgp_comm_unique_id on rank 0, the 128 bytes travel by any host channel,
//     pgp_comm_init on every rank (ncclCommInitRank);
//   * one process, n devices: pgp_group_create (ncclCommInitAll), one worker thread per device for the calls that synchronise.
// NCCL is loaded with dlopen("libnccl.so.2") on first use, so libpgp.so has no link-time dependency on it and single-GPU users need
// no NCCL at all (inside a torch process the already-loaded bundled NCCL is the one that answers).
//
// The exchange never sits on the scoring stream: K4 writes header + records into a slot's send buffer on the context's stream, an
// event hands over to the context's exchange stream, which runs ncclAllGather and the device->host copy of the gathered records
// into the slot's pinned buffer; pgp_topk_end waits on the slot's event and merges on the host.  Eight slots per context let the
// caller keep several steps in flight (pgp_topk_begin of step i+1 does not wait for step i's collective).
#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <thread>
#include <vector>

#include "pgp_internal.cuh"

namespace {

struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
};

NcclApi& nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (!api.handle) { api.error = std::string("dlopen(libnccl.so.2) failed: ") + (dlerror() ? dlerror() : "?"); return; }
    auto sym = [&](const char* name) -> void* {
      void* p = dlsym(api.handle, name);
      if (!p && api.error.empty()) api.error = std::string("NCCL symbol missing: ") + name;
      return p;
    };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  });
  return api;
}

#define PGP_NCCL(ctx, expr)                                                                                  \
  do {                                                                                                       \
    ncclResult_t r__ = (expr);                                                                               \
    if (r__ != ncclSuccess)                                                                                  \
      return pgp_fail(ctx, PGP_E_COMM, "%s:%d %s: %s", __FILE__, __LINE__, #expr, nccl_api().GetErrorString(r__)); \
  } while (0)

constexpr int NSLOT = 8;

struct Slot {
  DevBuf send, recv;            // (k + 1) records;  world x (k + 1) records
  pgp_hyp* host = nullptr;      // pinned, world x (k + 1) records
  size_t host_cap = 0;
  cudaEvent_t ev_sel = nullptr, ev_done = nullptr;
  int k = 0, kind = 0, mode = 0, obj = -1;
  bool auto_base = false, busy = false;
};

struct Comm {
  ncclComm_t nccl = nullptr;
  int rank = 0, world = 1;
  cudaStream_t stream = nullptr;
  Slot slot[NSLOT];
  DevBuf cnt_dev;               // pgp_comm_sync_generated: world x int64
  long long* cnt_host = nullptr;
};

Comm* comm_of(pgp_ctx* ctx) {
  if (!ctx->comm) {
    Comm* c = new Comm();
    // Default stream priority.  Measured (tools/gpu_round2_g.sh, gpu_round2_i.sh): giving the exchange stream the highest priority
    // does not shorten a scoring step (c2 at N = 4: 0.5637 vs 0.5628 ms) and makes a request made of many small launches slower and
    // erratic (c3 at N = 2: 159 / 112 ms per step against 82 ms) -- PGP_EXCHANGE_PRIORITY=1 turns it on for experiments.
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    const char* pe = getenv("PGP_EXCHANGE_PRIORITY");
    if (cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, (pe && atoi(pe) == 1) ? hi : lo) != cudaSuccess) { delete c; return nullptr; }
    ctx->comm = c;
  }
  return static_cast<Comm*>(ctx->comm);
}

int slot_prepare(pgp_ctx* ctx, Comm* c, Slot& s, int k) {
  const size_t rec = (size_t)(k + 1) * sizeof(pgp_hyp);
  PGP_CUDA(ctx, s.send.reserve(rec));
  PGP_CUDA(ctx, s.recv.reserve(rec * c->world));
  if (s.host_cap < rec * c->world) {
    if (s.host) cudaFreeHost(s.host);
    s.host = nullptr; s.host_cap = 0;
    PGP_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&s.host), rec * c->world));
    s.host_cap = rec * c->world;
  }
  if (!s.ev_sel) PGP_CUDA(ctx, cudaEventCreateWithFlags(&s.ev_sel, cudaEventDisableTiming));
  if (!s.ev_done) PGP_CUDA(ctx, cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
  s.k = k;
  return PGP_OK;
}

// stage 1 (context stream): K4 writes header + records into the slot's send buffer; the exchange stream waits for it
int stage_select(pgp_ctx* ctx, Comm* c, Slot& s, int obj, int k, int64_t index_base, int kind) {
  int rc = slot_prepare(ctx, c, s, k);
  if (rc) return rc;
  s.kind = kind; s.obj = obj; s.mode = ctx->last.mode;
  s.auto_base = index_base == PGP_INDEX_AUTO;
  pgp_hyp* send = s.send.as<pgp_hyp>();
  if (ctx->last.obj == obj && ctx->last.n > 0) {
    rc = k4_select_dev(ctx, ctx->last, k, s.auto_base ? 0 : index_base, kind, send, send + 1);
    if (rc) return rc;
  } else {
    PGP_CUDA(ctx, cudaMemsetAsync(send, 0, sizeof(pgp_hyp), ctx->stream));     // empty shard: header {batch size 0, 0 records}
  }
  PGP_CUDA(ctx, cudaEventRecord(s.ev_sel, ctx->stream));
  PGP_CUDA(ctx, cudaStreamWaitEvent(c->stream, s.ev_sel, 0));
  return PGP_OK;
}
// stage 2 (exchange stream): the collective.  Single-process groups wrap this stage of all devices in one ncclGroup.
int stage_gather(pgp_ctx* ctx, Comm* c, Slot& s) {
  if (c->world > 1)
    PGP_NCCL(ctx, nccl_api().AllGather(s.send.p, s.recv.p, (size_t)(s.k + 1) * sizeof(pgp_hyp), ncclChar, c->nccl, c->stream));
  return PGP_OK;
}
// stage 3 (exchange stream): gathered records -> pinned host buffer
int stage_download(pgp_ctx* ctx, Comm* c, Slot& s) {
  const size_t bytes = (size_t)(s.k + 1) * sizeof(pgp_hyp) * c->world;
  PGP_CUDA(ctx, cudaMemcpyAsync(s.host, c->world > 1 ? s.recv.p : s.send.p, bytes, cudaMemcpyDeviceToHost, c->stream));
  PGP_CUDA(ctx, cudaEventRecord(s.ev_done, c->stream));
  s.busy = true;
  return PGP_OK;
}

// waits for the slot's exchange and merges (pgp_exchange_merge below)
int slot_finish(pgp_ctx* ctx, Comm* c, Slot& s, pgp_hyp* out, int cap) {
  PGP_CUDA(ctx, cudaEventSynchronize(s.ev_done));
  s.busy = false;
  const int m = pgp_exchange_merge(s.host, c->world, s.k, s.kind, s.mode, s.auto_base ? 1 : 0, out, cap);
  if (m == PGP_E_CAPACITY) return pgp_fail(ctx, PGP_E_CAPACITY, "improving chain: a rank's local chain exceeds %d elements or the merged chain the capacity %d", s.k, cap);
  if (m < 0) return pgp_fail(ctx, m, "pgp_exchange_merge failed");
  return m;
}

int find_free_slot(Comm* c) {
  for (int i = 0; i < NSLOT; ++i) if (!c->slot[i].busy) return i;
  return -1;
}

int check_batch(pgp_ctx* ctx, Comm* c, int obj, int k) {
  if (k <= 0 || k > K4_MAX_K) return pgp_fail(ctx, PGP_E_INVALID, "k = %d outside 1..%d", k, K4_MAX_K);
  if (obj < 0 || obj >= PGP_MAX_OBJECTS) return pgp_fail(ctx, PGP_E_INVALID, "object slot %d out of range", obj);
  if (c->world == 1 && (ctx->last.obj != obj || ctx->last.n <= 0)) return pgp_fail(ctx, PGP_E_NO_SCORES, "no scored batch for object %d", obj);
  return PGP_OK;
}

int select_begin(pgp_ctx* ctx, int obj, int k, int64_t index_base, int kind) {
  Comm* c = comm_of(ctx);
  if (!c) return pgp_fail(ctx, PGP_E_CUDA, "cannot create the exchange stream");
  int rc = check_batch(ctx, c, obj, k);
  if (rc) return rc;
  const int t = find_free_slot(c);
  if (t < 0) return pgp_fail(ctx, PGP_E_INVALID, "all %d selection slots are in flight: call pgp_topk_end first", NSLOT);
  Slot& s = c->slot[t];
  if ((rc = stage_select(ctx, c, s, obj, k, index_base, kind))) return rc;
  if ((rc = stage_gather(ctx, c, s))) return rc;
  if ((rc = stage_download(ctx, c, s))) return rc;
  return t;
}

}  // namespace

bool pgp_comm_active(const pgp_ctx* ctx) { return ctx->comm && static_cast<const Comm*>(ctx->comm)->world > 1; }

void pgp_comm_release(pgp_ctx* ctx) {
  if (!ctx->comm) return;
  Comm* c = static_cast<Comm*>(ctx->comm);
  cudaStreamSynchronize(c->stream);
  if (c->nccl) nccl_api().CommDestroy(c->nccl);
  for (Slot& s : c->slot) {
    s.send.release(); s.recv.release();
    if (s.host) cudaFreeHost(s.host);
    if (s.ev_sel) cudaEventDestroy(s.ev_sel);
    if (s.ev_done) cudaEventDestroy(s.ev_done);
  }
  c->cnt_dev.release();
  if (c->cnt_host) cudaFreeHost(c->cnt_host);
  cudaStreamDestroy(c->stream);
  delete c;
  ctx->comm = nullptr;
}

extern "C" {

// Deterministic merge of the gathered wire blocks, on the host; the same bytes arrive on every rank, so every rank computes the
// same answer.  Wire format: per rank (k + 1) records -- a header {index = the rank's batch size, count = valid records,
// score != 0: the rank's chain overflowed k} followed by k records.
//   kind 0, top-k:  (score desc, global index asc) over the union                  == pgp_topk on the concatenated batch
//   kind 1, chain:  ranks in order, a record survives iff it beats everything before it == the strictly improving scan of
//           match4pcsBase.cc:1888-1901 over the concatenated batch (an element of the global chain beats every earlier element
//           of its own shard too, so it is in that shard's local chain; the local chains are all that has to travel).
//           COUNT mode compares the integer counts (what Verify's fraction is made of), WEIGHTED mode the fp32 scores, exactly
//           as K4 does locally.
// auto_base: the records carry shard-local indices; rank r's are offset by the batch sizes of the ranks before it.
int pgp_exchange_merge(const pgp_hyp* wire, int world, int k, int kind, int mode, int auto_base, pgp_hyp* out, int cap) {
  if (!wire || !out || world < 1 || k < 1 || cap < 0) return PGP_E_INVALID;
  const int stride = k + 1;
  std::vector<pgp_hyp> v;
  v.reserve((size_t)world * k);
  int64_t offset = 0;
  bool overflow = false;
  for (int r = 0; r < world; ++r) {
    const pgp_hyp& h = wire[(size_t)r * stride];
    const int n_valid = (int)std::min<int64_t>(h.count, k);
    if (h.score != 0.f) overflow = true;
    for (int i = 0; i < n_valid; ++i) {
      pgp_hyp rec = wire[(size_t)r * stride + 1 + i];
      if (rec.index < 0) continue;
      if (auto_base) rec.index += offset;
      v.push_back(rec);
    }
    offset += h.index;
  }
  int m = 0;
  if (kind == 0) {
    std::sort(v.begin(), v.end(), [](const pgp_hyp& a, const pgp_hyp& b) { return a.score != b.score ? a.score > b.score : a.index < b.index; });
    m = std::min<int>({cap, k, (int)v.size()});
    for (int i = 0; i < m; ++i) out[i] = v[i];
  } else {
    if (overflow) return PGP_E_CAPACITY;
    uint32_t best_c = 0; float best_s = 0.f;
    for (const pgp_hyp& r : v) {
      const bool better = mode == PGP_LCP_COUNT ? r.count > best_c : r.score > best_s;
      if (!better) continue;
      if (m >= cap) return PGP_E_CAPACITY;
      out[m++] = r; best_c = r.count; best_s = r.score;
    }
  }
  return m;
}

int pgp_comm_unique_id(void* id128) {
  if (!id128) return PGP_E_INVALID;
  NcclApi& api = nccl_api();
  if (!api.error.empty()) return pgp_fail(nullptr, PGP_E_COMM, "%s", api.error.c_str());
  static_assert(sizeof(ncclUniqueId) == PGP_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  ncclResult_t r = api.GetUniqueId(&id);
  if (r != ncclSuccess) return pgp_fail(nullptr, PGP_E_COMM, "ncclGetUniqueId: %s", api.GetErrorString(r));
  memcpy(id128, &id, sizeof(id));
  return PGP_OK;
}

int pgp_comm_init(pgp_ctx* ctx, const void* id128, int rank, int world) {
  if (!ctx) return PGP_E_INVALID;
  cudaSetDevice(ctx->device);
  if (world < 1 || rank < 0 || rank >= world || (world > 1 && !id128)) return pgp_fail(ctx, PGP_E_INVALID, "pgp_comm_init: bad rank %d / world %d", rank, world);
  Comm* c = comm_of(ctx);
  if (!c) return pgp_fail(ctx, PGP_E_CUDA, "cannot create the exchange stream");
  if (c->nccl) return pgp_fail(ctx, PGP_E_INVALID, "pgp_comm_init: the context already has a communicator");
  for (Slot& s : c->slot) if (s.busy) return pgp_fail(ctx, PGP_E_INVALID, "pgp_comm_init with selections in flight");
  if (world > 1) {
    NcclApi& api = nccl_api();
    if (!api.error.empty()) return pgp_fail(ctx, PGP_E_COMM, "%s", api.error.c_str());
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    PGP_NCCL(ctx, api.CommInitRank(&c->nccl, world, id, rank));
  }
  c->rank = rank; c->world = world;
  return PGP_OK;
}

int pgp_comm_init_all(pgp_ctx** ctxs, int n) {
  if (!ctxs || n < 1) return PGP_E_INVALID;
  for (int i = 0; i < n; ++i) if (!ctxs[i]) return PGP_E_INVALID;
  std::vector<Comm*> cs(n);
  std::vector<int> devs(n);
  for (int i = 0; i < n; ++i) {
    cudaSetDevice(ctxs[i]->device);
    cs[i] = comm_of(ctxs[i]);
    if (!cs[i]) return pgp_fail(ctxs[i], PGP_E_CUDA, "cannot create the exchange stream");
    if (cs[i]->nccl) return pgp_fail(ctxs[i], PGP_E_INVALID, "pgp_comm_init_all: context %d already has a communicator", i);
    devs[i] = ctxs[i]->device;
  }
  if (n > 1) {
    NcclApi& api = nccl_api();
    if (!api.error.empty()) return pgp_fail(ctxs[0], PGP_E_COMM, "%s", api.error.c_str());
    std::vector<ncclComm_t> comms(n);
    PGP_NCCL(ctxs[0], api.CommInitAll(comms.data(), n, devs.data()));
    for (int i = 0; i < n; ++i) cs[i]->nccl = comms[i];
  }
  for (int i = 0; i < n; ++i) { cs[i]->rank = i; cs[i]->world = n; }
  return PGP_OK;
}

int pgp_comm_rank(const pgp_ctx* ctx) { return ctx && ctx->comm ? static_cast<const Comm*>(ctx->comm)->rank : 0; }
int pgp_comm_world(const pgp_ctx* ctx) { return ctx && ctx->comm ? static_cast<const Comm*>(ctx->comm)->world : 1; }

int pgp_comm_destroy(pgp_ctx* ctx) {
  if (!ctx) return PGP_E_INVALID;
  cudaSetDevice(ctx->device);
  pgp_comm_release(ctx);
  return PGP_OK;
}

int pgp_topk_begin(pgp_ctx* ctx, int obj, int k, int64_t index_base) {
  if (!ctx) return PGP_E_INVALID;
  cudaSetDevice(ctx->device);
  return select_begin(ctx, obj, k, index_base, 0);
}

int pgp_topk_end(pgp_ctx* ctx, int ticket, pgp_hyp* out_host) {
  if (!ctx) return PGP_E_INVALID;
  cudaSetDevice(ctx->device);
  Comm* c = static_cast<Comm*>(ctx->comm);
  if (!c || ticket < 0 || ticket >= NSLOT || !c->slot[ticket].busy) return pgp_fail(ctx, PGP_E_INVALID, "pgp_topk_end: ticket %d is not in flight", ticket);
  if (!out_host) return pgp_fail(ctx, PGP_E_INVALID, "null output");
  Slot& s = c->slot[ticket];
  return slot_finish(ctx, c, s, out_host, s.k);
}

// Makes the context's stream wait for the ticket's exchange (measurement hook: an event recorded on the stream afterwards marks
// the point where the gathered records are on the host).
int pgp_topk_stream_wait(pgp_ctx* ctx, int ticket) {
  if (!ctx) return PGP_E_INVALID;
  cudaSetDevice(ctx->device);
  Comm* c = static_cast<Comm*>(ctx->comm);
  if (!c || ticket < 0 || ticket >= NSLOT || !c->slot[ticket].busy) return pgp_fail(ctx, PGP_E_INVALID, "pgp_topk_stream_wait: ticket %d is not in flight", ticket);
  PGP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, c->slot[ticket].ev_done, 0));
  return PGP_OK;
}

// Collective improving chain (hypothesisSet of Perform_N_steps, match4pcsBase.cc:1888-1914) over all ranks' batches in rank order.
int pgp_comm_improving_chain(pgp_ctx* ctx, int obj, int64_t index_base, pgp_hyp* out_host, int cap) {
  if (!ctx) return PGP_E_INVALID;
  cudaSetDevice(ctx->device);
  if (cap <= 0 || !out_host) return pgp_fail(ctx, PGP_E_INVALID, "bad capacity / output");
  const int t = select_begin(ctx, obj, PGP_CHAIN_EXCHANGE_CAP, index_base, 1);
  if (t < 0) return t;
  Comm* c = static_cast<Comm*>(ctx->comm);
  return slot_finish(ctx, c, c->slot[t], out_host, cap);
}

// The cut a global hypothesis cap makes in a request whose bases are sharded: ranks in order, the first ones keep everything, the
// one that crosses max_hyp is truncated, the rest keep nothing -- exactly the prefix of the concatenated list that the single-GPU
// generator keeps (it stops appending at max_hyp).  Pure host arithmetic (tests/test_sharding_gloo.py exercises it without a GPU).
int pgp_generated_cap_split(const int64_t* counts, int world, int64_t max_hyp, int rank, int64_t* keep, int64_t* index_base, int64_t* n_total) {
  if (!counts || world < 1 || rank < 0 || rank >= world) return PGP_E_INVALID;
  int64_t before = 0, total = 0;
  for (int r = 0; r < world; ++r) { if (counts[r] < 0) return PGP_E_INVALID; if (r < rank) before += counts[r]; total += counts[r]; }
  int64_t k = counts[rank];
  if (max_hyp > 0) {
    k = std::max<int64_t>(0, std::min<int64_t>(k, max_hyp - before));
    total = std::min(total, max_hyp);
    before = std::min(before, max_hyp);
  }
  if (keep) *keep = k;
  if (index_base) *index_base = before;
  if (n_total) *n_total = total;
  return PGP_OK;
}

// Bases sharded across ranks (pgp_generate_pcs_range): the per-rank hypothesis counts are exchanged, the global cap max_hyp is
// applied in rank order -- the same cut the single-GPU generator makes -- and every rank learns the global index of its first
// hypothesis.  The one other exchange on the path (8 bytes per rank).
int pgp_comm_sync_generated(pgp_ctx* ctx, int obj, int64_t max_hyp, int64_t* index_base_out, int64_t* n_total_out) {
  if (!ctx) return PGP_E_INVALID;
  cudaSetDevice(ctx->device);
  if (obj < 0 || obj >= PGP_MAX_OBJECTS || !ctx->models[obj].ready) return pgp_fail(ctx, PGP_E_NO_MODEL, "no model in slot %d", obj);
  Comm* c = comm_of(ctx);
  if (!c) return pgp_fail(ctx, PGP_E_CUDA, "cannot create the exchange stream");
  Model& m = ctx->models[obj];
  std::vector<long long> cnt(c->world, 0);
  cnt[c->rank] = m.n_gen;
  if (c->world > 1) {
    PGP_CUDA(ctx, c->cnt_dev.reserve((size_t)(c->world + 1) * 8));
    if (!c->cnt_host) PGP_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&c->cnt_host), 8 * 64));
    if (c->world > 63) return pgp_fail(ctx, PGP_E_INVALID, "more than 63 ranks");
    long long* d = c->cnt_dev.as<long long>();
    c->cnt_host[63] = m.n_gen;
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    PGP_CUDA(ctx, cudaMemcpyAsync(d + c->world, c->cnt_host + 63, 8, cudaMemcpyHostToDevice, c->stream));
    PGP_NCCL(ctx, nccl_api().AllGather(d + c->world, d, 8, ncclChar, c->nccl, c->stream));
    PGP_CUDA(ctx, cudaMemcpyAsync(c->cnt_host, d, (size_t)c->world * 8, cudaMemcpyDeviceToHost, c->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(c->stream));
    for (int r = 0; r < c->world; ++r) cnt[r] = c->cnt_host[r];
  }
  int64_t keep = 0, before = 0, total = 0;
  std::vector<int64_t> cnt64(cnt.begin(), cnt.end());
  pgp_generated_cap_split(cnt64.data(), c->world, max_hyp, c->rank, &keep, &before, &total);
  if (keep != m.n_gen) { m.n_gen = keep; m.gen_scored = false; }
  m.gen_index_base = before;
  if (index_base_out) *index_base_out = before;
  if (n_total_out) *n_total_out = total;
  return PGP_OK;
}

}  // extern "C"

// ================================================================================================================================
// One process, n devices.
struct pgp_group {
  std::vector<pgp_ctx*> ctx;
  std::vector<int64_t> shard_lo;      // pgp_group_score_lcp: first hypothesis of device i (size n + 1)
  std::string err;
};

namespace {

int group_fail(pgp_group* g, int code, const std::string& text) { if (g) g->err = text; return code; }

// runs fn(i, ctx_i) for every device on its own thread (the per-device calls synchronise their stream) and returns the first error
template <class F>
int group_run(pgp_group* g, F fn) {
  const int n = (int)g->ctx.size();
  std::vector<int> rc(n, 0);
  if (n == 1) rc[0] = fn(0, g->ctx[0]);
  else {
    std::vector<std::thread> th;
    th.reserve(n);
    for (int i = 0; i < n; ++i) th.emplace_back([&, i] { cudaSetDevice(g->ctx[i]->device); rc[i] = fn(i, g->ctx[i]); });
    for (auto& t : th) t.join();
  }
  for (int i = 0; i < n; ++i)
    if (rc[i] < 0) return group_fail(g, rc[i], "device " + std::to_string(g->ctx[i]->device) + ": " + g->ctx[i]->err);
  return PGP_OK;
}

// K4 on every device -> ONE grouped ncclAllGather -> downloads -> merge (device 0's copy; every device receives the same bytes)
int group_select(pgp_group* g, int obj, int k, int kind, const std::vector<int64_t>& index_base, pgp_hyp* out, int cap) {
  const int n = (int)g->ctx.size();
  std::vector<int> ticket(n, -1);
  for (int i = 0; i < n; ++i) {
    pgp_ctx* ctx = g->ctx[i];
    cudaSetDevice(ctx->device);
    Comm* c = comm_of(ctx);
    if (!c) return group_fail(g, PGP_E_CUDA, "cannot create the exchange stream");
    int rc = check_batch(ctx, c, obj, k);
    if (rc) return group_fail(g, rc, ctx->err);
    ticket[i] = find_free_slot(c);
    if (ticket[i] < 0) return group_fail(g, PGP_E_INVALID, "no free selection slot");
    if ((rc = stage_select(ctx, c, c->slot[ticket[i]], obj, k, index_base[i], kind))) return group_fail(g, rc, ctx->err);
  }
  if (n > 1) {
    NcclApi& api = nccl_api();
    ncclResult_t r = api.GroupStart();
    if (r != ncclSuccess) return group_fail(g, PGP_E_COMM, api.GetErrorString(r));
    for (int i = 0; i < n; ++i) {
      cudaSetDevice(g->ctx[i]->device);
      Comm* c = static_cast<Comm*>(g->ctx[i]->comm);
      int rc = stage_gather(g->ctx[i], c, c->slot[ticket[i]]);
      if (rc) { api.GroupEnd(); return group_fail(g, rc, g->ctx[i]->err); }
    }
    r = api.GroupEnd();
    if (r != ncclSuccess) return group_fail(g, PGP_E_COMM, api.GetErrorString(r));
  }
  for (int i = 0; i < n; ++i) {
    cudaSetDevice(g->ctx[i]->device);
    Comm* c = static_cast<Comm*>(g->ctx[i]->comm);
    int rc = stage_download(g->ctx[i], c, c->slot[ticket[i]]);
    if (rc) return group_fail(g, rc, g->ctx[i]->err);
  }
  int m = 0;
  for (int i = n - 1; i >= 0; --i) {            // every slot is waited for and released; device 0's result is returned
    cudaSetDevice(g->ctx[i]->device);
    Comm* c = static_cast<Comm*>(g->ctx[i]->comm);
    std::vector<pgp_hyp> tmp((size_t)std::max(cap, k));
    m = slot_finish(g->ctx[i], c, c->slot[ticket[i]], i == 0 ? out : tmp.data(), cap);
    if (m < 0) return group_fail(g, m, g->ctx[i]->err);
  }
  return m;
}

}  // namespace

extern "C" {

pgp_group* pgp_group_create(int n_devices, const int* device_ids) {
  if (n_devices < 1 || n_devices > 64) { pgp_fail(nullptr, PGP_E_INVALID, "pgp_group_create: %d devices", n_devices); return nullptr; }
  pgp_group* g = new pgp_group();
  for (int i = 0; i < n_devices; ++i) {
    pgp_ctx* c = pgp_create(device_ids ? device_ids[i] : i);
    if (!c) { for (pgp_ctx* p : g->ctx) pgp_destroy(p); delete g; return nullptr; }
    g->ctx.push_back(c);
  }
  if (pgp_comm_init_all(g->ctx.data(), n_devices) != PGP_OK) {
    pgp_fail(nullptr, PGP_E_COMM, "%s", g->ctx[0]->err.c_str());
    for (pgp_ctx* p : g->ctx) pgp_destroy(p);
    delete g;
    return nullptr;
  }
  return g;
}

void pgp_group_destroy(pgp_group* g) {
  if (!g) return;
  for (pgp_ctx* p : g->ctx) pgp_destroy(p);
  delete g;
}

int pgp_group_size(const pgp_group* g) { return g ? (int)g->ctx.size() : 0; }
pgp_ctx* pgp_group_ctx(pgp_group* g, int i) { return g && i >= 0 && i < (int)g->ctx.size() ? g->ctx[i] : nullptr; }
const char* pgp_group_last_error(const pgp_group* g) { return g ? g->err.c_str() : pgp_last_error(nullptr); }

int pgp_group_set_scene(pgp_group* g, const float* xyz, const float* nrm, int n, float delta) {
  if (!g) return PGP_E_INVALID;
  return group_run(g, [&](int, pgp_ctx* c) { return pgp_set_scene(c, xyz, nrm, n, delta); });
}
int pgp_group_set_scene_prior_image(pgp_group* g, const uint16_t* img, int rows, int cols, const float* K9) {
  if (!g) return PGP_E_INVALID;
  return group_run(g, [&](int, pgp_ctx* c) { return pgp_set_scene_prior_image(c, img, rows, cols, K9); });
}
int pgp_group_set_scene_priors(pgp_group* g, const float* prior) {
  if (!g) return PGP_E_INVALID;
  return group_run(g, [&](int, pgp_ctx* c) { return pgp_set_scene_priors(c, prior); });
}
int pgp_group_set_model(pgp_group* g, int obj, const float* sx, const float* sn, int nq, const float* vx, const float* vn, int nv) {
  if (!g) return PGP_E_INVALID;
  return group_run(g, [&](int, pgp_ctx* c) { return pgp_set_model(c, obj, sx, sn, nq, vx, vn, nv); });
}
int pgp_group_set_ppf_map(pgp_group* g, int obj, const int32_t* keys4, const int64_t* offsets, const int32_t* pairs, int64_t n_keys) {
  if (!g) return PGP_E_INVALID;
  return group_run(g, [&](int, pgp_ctx* c) { return pgp_set_ppf_map(c, obj, keys4, offsets, pairs, n_keys); });
}
int pgp_group_build_ppf_map(pgp_group* g, int obj) {
  if (!g) return PGP_E_INVALID;
  return group_run(g, [&](int, pgp_ctx* c) { return pgp_build_ppf_map(c, obj); });
}

// Bases [i B / n, (i+1) B / n) on device i (each device generates AND later scores its own hypotheses: no transform traffic),
// then the global cap in device order, exactly where pgp_generate_pcs on one device would stop.
int pgp_group_generate_pcs(pgp_group* g, int obj, const pgp_pcs_opts* opts, uint64_t seed, int64_t max_hyp, int64_t* n_hyp) {
  if (!g || !n_hyp || max_hyp <= 0) return PGP_E_INVALID;
  pgp_pcs_opts o;
  if (opts) o = *opts; else pgp_pcs_default_opts(&o);
  const int n = (int)g->ctx.size(), B = std::max(1, o.n_bases);
  std::vector<int64_t> cnt(n, 0);
  int rc = group_run(g, [&](int i, pgp_ctx* c) {
    const int lo = (int)((int64_t)B * i / n), hi = (int)((int64_t)B * (i + 1) / n);
    return pgp_generate_pcs_range(c, obj, &o, seed, lo, hi, max_hyp, &cnt[i]);
  });
  if (rc) return rc;
  int64_t before = 0;
  for (int i = 0; i < n; ++i) {
    Model& m = g->ctx[i]->models[obj];
    const int64_t keep = std::max<int64_t>(0, std::min<int64_t>(cnt[i], max_hyp - before));
    m.n_gen = keep;
    m.gen_index_base = before;
    before += keep;
  }
  *n_hyp = before;
  return PGP_OK;
}

int pgp_group_score_generated(pgp_group* g, int obj, int mode) {
  if (!g) return PGP_E_INVALID;
  for (pgp_ctx* c : g->ctx) {                       // asynchronous per device: no threads needed
    if (c->models[obj].n_gen <= 0) { c->last = LastBatch(); continue; }
    int rc = pgp_score_generated(c, obj, mode);
    if (rc) return group_fail(g, rc, c->err);
  }
  g->shard_lo.assign(g->ctx.size() + 1, -1);        // the shards are the generated ranges
  return PGP_OK;
}

// Hypotheses [lo_i, hi_i) on device i; T_host and the outputs should be pinned so that the n uploads / downloads overlap.
int pgp_group_score_lcp(pgp_group* g, int obj, const float* T_host, int64_t n_hyp, int mode, uint32_t* counts_host, float* scores_host) {
  if (!g || n_hyp < 0 || (n_hyp > 0 && !T_host)) return PGP_E_INVALID;
  const int n = (int)g->ctx.size();
  g->shard_lo.assign(n + 1, 0);
  for (int i = 0; i <= n; ++i) g->shard_lo[i] = n_hyp * i / n;
  for (int i = 0; i < n; ++i) {
    const int64_t lo = g->shard_lo[i], cnt = g->shard_lo[i + 1] - lo;
    int rc = pgp_score_lcp_begin(g->ctx[i], obj, T_host + 12 * lo, cnt, mode, counts_host ? counts_host + lo : nullptr, scores_host ? scores_host + lo : nullptr);
    if (rc) return group_fail(g, rc, g->ctx[i]->err);
  }
  for (int i = 0; i < n; ++i) {
    int rc = pgp_score_lcp_end(g->ctx[i]);
    if (rc < 0) return group_fail(g, rc, g->ctx[i]->err);
    if ((rc = pgp_synchronize(g->ctx[i]))) return group_fail(g, rc, g->ctx[i]->err);
  }
  return PGP_OK;
}

static std::vector<int64_t> group_index_bases(pgp_group* g, int obj) {
  const int n = (int)g->ctx.size();
  std::vector<int64_t> base(n, PGP_INDEX_AUTO);
  for (int i = 0; i < n; ++i) {
    if ((int)g->shard_lo.size() == n + 1 && g->shard_lo[i] >= 0) base[i] = g->shard_lo[i];
    else if (g->ctx[i]->models[obj].gen_index_base >= 0) base[i] = g->ctx[i]->models[obj].gen_index_base;
  }
  return base;
}

int pgp_group_topk(pgp_group* g, int obj, int k, pgp_hyp* out_host) {
  if (!g || !out_host) return PGP_E_INVALID;
  return group_select(g, obj, k, 0, group_index_bases(g, obj), out_host, k);
}

int pgp_group_improving_chain(pgp_group* g, int obj, pgp_hyp* out_host, int cap) {
  if (!g || !out_host || cap <= 0) return PGP_E_INVALID;
  return group_select(g, obj, PGP_CHAIN_EXCHANGE_CAP, 1, group_index_bases(g, obj), out_host, cap);
}

}  // extern "C"
