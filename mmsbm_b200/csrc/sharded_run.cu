// ONE set of S runs sharded over the GPUs of a box (one process per GPU): the multi-GPU form of
// the loop src/mmsbm.py:243-250 for a fit that is too slow (or too large) for one GPU.
//
// Sharding ("owner computes" on both sides, SURVEY.md section 8e.3 taken one step further):
//   rank g owns a contiguous USER range and a contiguous ITEM range, both balanced by rating
//   count.  It holds a CSR over its users built from ALL their ratings and a CSC over its items
//   built from ALL theirs, so n_theta of its users and n_eta of its items are complete local sums:
//   no partial theta / eta sums ever cross the NVLink, and no item-side work is replicated.
//   What a pass gathers are rows of the OTHER side for arbitrary ids, so every rank keeps full
//   gather tables (eta for the by-user pass, theta for the by-item pass, in the run-interleaved
//   layouts of segment_pass.cuh) in an EXCHANGE BUFFER that its peers map through CUDA IPC.
//
// One iteration on a rank (main stream `st`, copy stream `cs`):
//   prep_p, W_u = theta_own x Pw, W_i = eta_own x Pw                      local rows only
//   by-user pass over own users (gathers tables[cur].eta)      -> g_u -> theta_own'
//   interleave theta_own' into own tables[nxt].theta; cs: push that slice into every peer's
//     buffer with the COPY ENGINES (cudaMemcpy2DAsync over NVLink) -- overlaps the by-item pass
//   by-item pass over own items (gathers tables[cur].theta)    -> g_i -> eta_own'
//   interleave eta_own' into tables[nxt].eta; cs: push
//   n_pr partial over own items (or users), then ONE small ncclAllReduce of n_pr [S][K][L][R]
//     after the rank's pushes have completed: it is the only collective of the iteration and
//     doubles as the barrier that tells every rank all slices have landed (and that nobody
//     still reads the tables that the next iteration overwrites); normalise pr.
// The SMs never move parameter rows: slices travel by DMA while the segment pass computes.
// Sums have a fixed order for a fixed world size; vs one GPU only the n_pr order differs.
#include <dlfcn.h>
#include <nccl.h>

#include <chrono>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "em_internal.cuh"

namespace mmsbm {

// ---- NCCL through dlopen (the library torch.distributed already loaded) --------------------
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

#define MMSBM_NCCL(expr)                                                                   \
  do {                                                                                     \
    ncclResult_t r__ = (expr);                                                             \
    if (r__ != ncclSuccess) {                                                              \
      set_error("%s failed: %s", #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "?"); \
      return 1000 + (int)r__;                                                              \
    }                                                                                      \
  } while (0)

static int nccl_ready() {
  MMSBM_REQUIRE(g_nccl.handle, MMSBM_EINVAL, "NCCL is not loaded: call mmsbm_nccl_load first");
  return 0;
}

// ---- layout of the exchange buffer ------------------------------------------------------------
// Two halves (the tables an iteration reads, the tables it fills for the next one); each half:
//   eta  tables of the by-user pass:  hexa [S/6][I][6][ldl] | pairs [S/2][I][2][ldl] | plain [S][I][ldl]
//   theta tables of the by-item pass:                         pairs [S/2][U][2][ldk] | plain [S][U][ldk]
// Every table is addressed as on one GPU (segment_pass.cuh); only the run groups the pass
// really uses (plan_runs) are filled and exchanged.  256 bytes of scratch close the buffer.
struct Table { size_t off; int gs, group0, groups, ld, n_all; };     // off: bytes inside a half
struct GridLayout {
  Table eta[3], theta[2];
  size_t half_bytes, total_bytes;
};

static GridLayout grid_layout(int U, int I, int K, int L, int R, int S) {
  const int ldk = row_stride(K), ldl = row_stride(L);
  const RunPlan pu = plan_runs(ldl, R, S, true), pi = plan_runs(ldk, R, S, false);
  GridLayout g{};
  size_t off = 0;
  auto put = [&](Table& t, int gs, int group0, int groups, int ld, int n_all, int addr_groups) {
    t = Table{off, gs, group0, groups, ld, n_all};
    off += align_up((size_t)addr_groups * gs * n_all * ld * 8);
  };
  put(g.eta[0], 6, 0, pu.hexas, ldl, I, pu.hexas);
  put(g.eta[1], 2, pu.pair_group0, pu.pairs, ldl, I, pu.pairs ? S / 2 : 0);
  put(g.eta[2], 1, pu.single_from, S - pu.single_from, ldl, I, S > pu.single_from ? S : 0);
  put(g.theta[0], 2, pi.pair_group0, pi.pairs, ldk, U, pi.pairs ? S / 2 : 0);
  put(g.theta[1], 1, pi.single_from, S - pi.single_from, ldk, U, S > pi.single_from ? S : 0);
  g.half_bytes = off;
  g.total_bytes = 2 * off + 256;
  return g;
}

// the tables of half `half` of the own buffer as the target of row_n_kernel's second store
static RowPublish row_publish(const void* base, const GridLayout& g, const Table* tabs, int n_tabs, int half,
                              int n_all, int row0) {
  RowPublish p{};
  for (int k = 0; k < n_tabs && k < 3; ++k) {
    const Table& t = tabs[k];
    if (t.groups == 0) continue;
    p.dst[k] = reinterpret_cast<double*>(const_cast<char*>(static_cast<const char*>(base)) +
                                         (size_t)half * g.half_bytes + t.off);
    p.gs[k] = t.gs; p.group0[k] = t.group0; p.groups[k] = t.groups;
  }
  p.n_all = n_all; p.row0 = row0;
  return p;
}

static const double* table_ptr(const void* base, const GridLayout& g, int half, const Table& t) {
  if (t.groups == 0) return nullptr;
  return reinterpret_cast<const double*>(static_cast<const char*>(base) + (size_t)half * g.half_bytes + t.off);
}

// Streams and events of the exchange: one COPY stream per peer (the pushes to different peers run
// on different copy engines at the same time; on one stream they would queue up behind each other
// and a 30 MB push made of 21 strided copies would be latency-bound), one SIDE stream for NCCL.
struct Exchange {
  int peers = 0;
  cudaStream_t side = nullptr;
  cudaStream_t aux = nullptr;                   // high priority: epilogue of pass 1 beside pass 2
  cudaEvent_t p_ready = nullptr, w2_ready = nullptr, pass1_done = nullptr, aux_done = nullptr;
  cudaStream_t cp[16] = {nullptr};
  cudaEvent_t ready = nullptr;                  // main -> copy streams: the slice is in the own tables
  cudaEvent_t done[16] = {nullptr};             // copy stream p -> side: its copies have been issued and finished
  cudaEvent_t partial = nullptr, pr_done = nullptr;      // main -> side, side -> main: n_pr all-reduce
  // side -> main: [0][.] theta tables, [1][.] eta tables complete everywhere; two events per table,
  // used by alternate iterations (a pass waits for the PREVIOUS iteration's barrier while this
  // iteration's one is already being recorded)
  cudaEvent_t arrived[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  int open(int world) {
    peers = world - 1;
    if (peers <= 0) return 0;
    MMSBM_REQUIRE(peers <= 16, MMSBM_ERANGE, "sharded runs support up to 17 ranks");
    MMSBM_CUDA(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
    {
      int lo = 0, hi = 0;                       // (numerically lowest = highest priority)
      MMSBM_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
      MMSBM_CUDA(cudaStreamCreateWithPriority(&aux, cudaStreamNonBlocking, hi));
    }
    for (int p = 0; p < peers; ++p) {
      MMSBM_CUDA(cudaStreamCreateWithFlags(&cp[p], cudaStreamNonBlocking));
      MMSBM_CUDA(cudaEventCreateWithFlags(&done[p], cudaEventDisableTiming));
    }
    cudaEvent_t* evs[] = {&ready, &partial, &pr_done, &arrived[0][0], &arrived[0][1], &arrived[1][0], &arrived[1][1],
                          &p_ready, &w2_ready, &pass1_done, &aux_done};
    for (cudaEvent_t* e : evs) MMSBM_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    return 0;
  }
  ~Exchange() {                                 // queued work finishes first: handles are released lazily
    cudaEvent_t evs[] = {ready, partial, pr_done, arrived[0][0], arrived[0][1], arrived[1][0], arrived[1][1],
                         p_ready, w2_ready, pass1_done, aux_done};
    for (cudaEvent_t e : evs) if (e) cudaEventDestroy(e);
    for (int p = 0; p < peers; ++p) {
      if (done[p]) cudaEventDestroy(done[p]);
      if (cp[p]) cudaStreamDestroy(cp[p]);
    }
    if (side) cudaStreamDestroy(side);
    if (aux) cudaStreamDestroy(aux);
  }
};

// own rows [lo, lo + n_own) of one parameter (plain [S][n_own][ld]) -> the tables of half `half`:
// interleave into the own buffer on `st`, then DMA the slice into every peer's buffer, one copy
// stream per peer (barrier_on_side makes the side stream wait for them)
static int publish_side(const mmsbm_shard_t& sh, const GridLayout& g, const Table* tabs, int n_tabs,
                        const double* own_rows, int n_own, int lo, int half, cudaStream_t st,
                        const Exchange& ex) {
  char* mine = static_cast<char*>(sh.exchange_dev[sh.rank]);
  for (int k = 0; k < n_tabs && own_rows; ++k) {             // own_rows == NULL: row_n_kernel wrote the slice already
    const Table& t = tabs[k];
    if (t.groups == 0) continue;
    double* dst = reinterpret_cast<double*>(mine + (size_t)half * g.half_bytes + t.off);
    int rc = launch_interleave(own_rows, dst, n_own, t.n_all, lo, t.ld, t.group0, t.groups, t.gs, st);
    if (rc) return rc;
  }
  if (sh.world == 1) return 0;
  MMSBM_CUDA(cudaEventRecord(ex.ready, st));
  for (int d = 1; d < sh.world; ++d) {
    const int peer = (sh.rank + d) % sh.world;               // copy stream d-1 serves peer rank+d
    cudaStream_t cs = ex.cp[d - 1];
    char* theirs = static_cast<char*>(sh.exchange_dev[peer]);
    MMSBM_CUDA(cudaStreamWaitEvent(cs, ex.ready, 0));
    for (int k = 0; k < n_tabs; ++k) {
      const Table& t = tabs[k];
      if (t.groups == 0) continue;
      const size_t row_bytes = (size_t)t.gs * t.ld * 8;
      const size_t pitch = (size_t)t.n_all * row_bytes;
      const size_t o = (size_t)half * g.half_bytes + t.off + ((size_t)t.group0 * t.n_all + lo) * row_bytes;
      MMSBM_CUDA(cudaMemcpy2DAsync(theirs + o, pitch, mine + o, pitch, (size_t)n_own * row_bytes,
                                   (size_t)t.groups, cudaMemcpyDeviceToDevice, cs));
    }
    MMSBM_CUDA(cudaEventRecord(ex.done[d - 1], cs));
  }
  return 0;
}

// on the side stream, after this rank's pushes: a one-element all-reduce = "every rank's slices of
// this table have landed everywhere, and every rank is past the pass that produced them"
static int barrier_on_side(const mmsbm_shard_t& sh, const GridLayout& g, const Exchange& ex, cudaEvent_t signal) {
  for (int p = 0; p < ex.peers; ++p) MMSBM_CUDA(cudaStreamWaitEvent(ex.side, ex.done[p], 0));
  double* scratch = reinterpret_cast<double*>(static_cast<char*>(sh.exchange_dev[sh.rank]) + 2 * g.half_bytes);
  MMSBM_NCCL(g_nccl.AllReduce(scratch, scratch, 1, ncclFloat64, ncclSum, static_cast<ncclComm_t>(sh.nccl_comm), ex.side));
  MMSBM_CUDA(cudaEventRecord(signal, ex.side));
  return 0;
}

static int check_shard(const mmsbm_shard_t* sh, const char* who) {
  MMSBM_REQUIRE(sh, MMSBM_EINVAL, "%s: null shard", who);
  MMSBM_REQUIRE(sh->n_users > 0 && sh->n_items > 0 && sh->n_levels > 0 && sh->K > 0 && sh->L > 0 &&
                    sh->n_runs > 0 && sh->n_users_own > 0 && sh->n_items_own > 0 && sh->n_ratings_u >= 0 &&
                    sh->n_ratings_i >= 0, MMSBM_EINVAL, "%s: bad size", who);
  MMSBM_REQUIRE(sh->user_lo >= 0 && sh->user_lo + sh->n_users_own <= sh->n_users && sh->item_lo >= 0 &&
                    sh->item_lo + sh->n_items_own <= sh->n_items, MMSBM_EINVAL, "%s: own range outside the ids", who);
  MMSBM_REQUIRE(sh->world >= 1 && sh->rank >= 0 && sh->rank < sh->world && sh->exchange_dev, MMSBM_EINVAL,
                "%s: bad rank / world / exchange", who);
  for (int r = 0; r < sh->world; ++r)
    MMSBM_REQUIRE(sh->exchange_dev[r], MMSBM_EINVAL, "%s: exchange pointer of rank %d is null", who, r);
  MMSBM_REQUIRE(sh->world == 1 || sh->nccl_comm, MMSBM_EINVAL, "%s: world > 1 needs an NCCL communicator", who);
  MMSBM_REQUIRE(sh->K <= 32 && sh->L <= 32 && sh->n_levels <= 31, MMSBM_ERANGE,
                "%s: sharded runs support K, L <= 32 and R <= 31", who);
  return 0;
}

struct ShardDims {
  int ldk, ldl, rnb_u, rnb_i;
  bool emit_items;
  int64_t pmax_u, pmax_i, lmax_u, lmax_i, smax_u, smax_i;
  size_t p_elems, wg_u, wg_i, partial, slots_u, slots_i, ctr;
};

static ShardDims shard_dims(const mmsbm_shard_t& s) {
  ShardDims d;
  const int S = s.n_runs, R = s.n_levels;
  d.ldk = row_stride(s.K); d.ldl = row_stride(s.L);
  d.rnb_u = R * d.ldl; d.rnb_i = R * d.ldk;
  d.emit_items = s.n_items <= s.n_users;
  d.pmax_u = (int64_t)s.n_users_own + s.n_ratings_u / MMSBM_PIECE_LEN + 1;      // = graph_build.cu
  d.pmax_i = (int64_t)s.n_items_own + s.n_ratings_i / MMSBM_PIECE_LEN + 1;
  d.lmax_u = s.n_ratings_u / MMSBM_PIECE_LEN + 1; d.lmax_i = s.n_ratings_i / MMSBM_PIECE_LEN + 1;
  d.smax_u = 2 * (s.n_ratings_u / MMSBM_PIECE_LEN) + 1; d.smax_i = 2 * (s.n_ratings_i / MMSBM_PIECE_LEN) + 1;
  d.p_elems = (size_t)S * d.ldk * d.ldl * R;
  d.wg_u = (size_t)S * s.n_users_own * d.rnb_u;
  d.wg_i = (size_t)S * s.n_items_own * d.rnb_i;
  const size_t pi = (size_t)s.L * R * d.ldk, pu = (size_t)s.K * R * d.ldl;   // either side may emit n_pr
  d.partial = (size_t)S * kPrSlabs * (pi > pu ? pi : pu);
  d.slots_u = (size_t)S * d.smax_u * d.rnb_u;
  d.slots_i = (size_t)S * d.smax_i * d.rnb_i;
  d.ctr = 2 * ((size_t)S + 8);
  return d;
}

}  // namespace mmsbm

using namespace mmsbm;

// ---- NCCL plumbing -----------------------------------------------------------------------------
extern "C" int mmsbm_nccl_load(const char* path) {
  if (g_nccl.handle) return 0;
  void* h = dlopen((path && *path) ? path : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  MMSBM_REQUIRE(h, MMSBM_ENODEV, "cannot load NCCL (%s): %s", (path && *path) ? path : "libnccl.so.2", dlerror());
  NcclApi api;
  api.handle = h;
  api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
  api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
  api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(h, "ncclAllReduce"));
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
  MMSBM_REQUIRE(api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.GetErrorString,
                MMSBM_ENODEV, "NCCL library lacks a required symbol");
  g_nccl = api;
  return 0;
}

extern "C" int mmsbm_nccl_unique_id(unsigned char* id128) {
  int rc = nccl_ready();
  if (rc) return rc;
  MMSBM_REQUIRE(id128, MMSBM_EINVAL, "mmsbm_nccl_unique_id: null output");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  MMSBM_NCCL(g_nccl.GetUniqueId(&id));
  memcpy(id128, &id, 128);
  return 0;
}

extern "C" int mmsbm_nccl_comm_init(const unsigned char* id128, int32_t rank, int32_t world, void** comm) {
  int rc = nccl_ready();
  if (rc) return rc;
  MMSBM_REQUIRE(id128 && comm && world >= 1 && rank >= 0 && rank < world, MMSBM_EINVAL,
                "mmsbm_nccl_comm_init: bad argument");
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  ncclComm_t c = nullptr;
  MMSBM_NCCL(g_nccl.CommInitRank(&c, world, id, rank));
  *comm = c;
  return 0;
}

extern "C" int mmsbm_nccl_comm_destroy(void* comm) {
  if (!comm || !g_nccl.handle) return 0;
  MMSBM_NCCL(g_nccl.CommDestroy(static_cast<ncclComm_t>(comm)));
  return 0;
}

// ---- peer-mappable device memory (CUDA IPC) -----------------------------------------------------
extern "C" int mmsbm_ipc_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64) {
  MMSBM_REQUIRE(dev_ptr && handle64 && bytes > 0, MMSBM_EINVAL, "mmsbm_ipc_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  void* p = nullptr;
  MMSBM_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    set_error("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    return (int)e;
  }
  memcpy(handle64, &h, 64);
  *dev_ptr = p;
  return 0;
}
extern "C" int mmsbm_ipc_open(const unsigned char* handle64, void** dev_ptr) {
  MMSBM_REQUIRE(dev_ptr && handle64, MMSBM_EINVAL, "mmsbm_ipc_open: bad argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  MMSBM_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
extern "C" int mmsbm_ipc_close(void* dev_ptr) {
  if (dev_ptr) MMSBM_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return 0;
}
extern "C" int mmsbm_ipc_free(void* dev_ptr) {
  if (dev_ptr) MMSBM_CUDA(cudaFree(dev_ptr));
  return 0;
}

// ---- sizes ------------------------------------------------------------------------------------------
extern "C" int mmsbm_shard_exchange_bytes(int32_t U, int32_t I, int32_t K, int32_t L, int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && U > 0 && I > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_shard_exchange_bytes: bad argument");
  // the layout follows the run plan, which depends on the number of rating levels through shared
  // memory: the buffer is sized for the largest layout over every supported level count
  size_t most = 0;
  for (int R = 1; R <= 31; ++R) {
    const size_t b = grid_layout(U, I, K, L, R, S).total_bytes;
    if (b > most) most = b;
  }
  *bytes = most;
  return 0;
}

extern "C" int mmsbm_shard_workspace_bytes(const mmsbm_shard_t* sh, size_t* bytes) {
  int rc = check_shard(sh, "mmsbm_shard_workspace_bytes");
  if (rc) return rc;
  MMSBM_REQUIRE(bytes, MMSBM_EINVAL, "mmsbm_shard_workspace_bytes: null output");
  const ShardDims d = shard_dims(*sh);
  *bytes = 4 * align_up(d.p_elems * 8) + align_up(d.wg_u * 8) + align_up(d.wg_i * 8) + align_up(d.partial * 8) +
           align_up(d.slots_u * 8) + align_up(d.slots_i * 8) + align_up(d.ctr * 4) + 256;
  return 0;
}

// The tables of half `half` <- this rank's rows of theta and eta, on every rank; returns after the
// NCCL barrier has been enqueued on `stream` (every rank must call it).
extern "C" int mmsbm_shard_publish(const mmsbm_shard_t* sh, const double* theta_own, const double* eta_own,
                                   int32_t half, void* stream) {
  int rc = check_shard(sh, "mmsbm_shard_publish");
  if (rc) return rc;
  MMSBM_REQUIRE(theta_own && eta_own && (half == 0 || half == 1), MMSBM_EINVAL, "mmsbm_shard_publish: bad argument");
  if (sh->world > 1 && (rc = nccl_ready())) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const GridLayout g = grid_layout(sh->n_users, sh->n_items, sh->K, sh->L, sh->n_levels, sh->n_runs);
  Exchange ex;
  if ((rc = ex.open(sh->world))) return rc;
  if (sh->world > 1) {                          // the side stream starts behind everything queued on `st`
    MMSBM_CUDA(cudaEventRecord(ex.partial, st));
    MMSBM_CUDA(cudaStreamWaitEvent(ex.side, ex.partial, 0));
  }
  if ((rc = publish_side(*sh, g, g.theta, 2, theta_own, sh->n_users_own, sh->user_lo, half, st, ex))) return rc;
  if ((rc = publish_side(*sh, g, g.eta, 3, eta_own, sh->n_items_own, sh->item_lo, half, st, ex))) return rc;
  if (sh->world > 1) {
    // (one barrier covers both tables: the copy streams run their theta and eta copies in order)
    if ((rc = barrier_on_side(*sh, g, ex, ex.arrived[0][0]))) return rc;
    MMSBM_CUDA(cudaStreamWaitEvent(st, ex.arrived[0][0], 0));
  }
  return 0;
}

// `iterations` EM steps of the sharded loop.  (theta, eta)_a/_b: this rank's OWN rows, plain layout
// [S][n_users_own][ldk] / [S][n_items_own][ldl]; pr_a/_b: [S][K][L][R], replicated.  The tables of half
// `half` must hold the parameters of the _a buffers on every rank (mmsbm_shard_publish).  The result is
// in _a (tables in `half`) when iterations is even, else in _b (tables in half ^ 1).
//
// Schedule of one iteration with peers (main stream st, side stream for NCCL, one copy stream per peer):
//   st:   P tables, W of the own users and items
//   st:   wait "tables of pass 1 arrived" | pass 1 | n of its side | interleave the new rows into the own
//         next tables | n_pr partial from the g rows of pass 1
//   copy: push the slice to every peer (overlaps pass 2)      side: all-reduce n_pr (overlaps pass 2),
//                                                                   then, once the pushes are done, the
//                                                                   arrival barrier of that table
//   st:   wait "tables of pass 2 arrived" | pass 2 | n | interleave      copy: push      side: barrier
//   st:   wait n_pr | normalise pr
// Passes ALTERNATE their order from one iteration to the next (by-user, by-item | by-item, by-user | ...):
// the table a first pass gathers was pushed during the previous iteration's second pass, and the one a
// second pass gathers was pushed at the very end of the previous iteration and has the whole first pass to
// arrive, so no push and no barrier is waited for.  n_pr always comes from the side with fewer segments;
// in the iterations where that side is pass 1 its all-reduce hides behind pass 2.  With world == 1 nothing
// of this applies: fixed order, n_pr normalised in place -- bit for bit what mmsbm_em_run computes.
//
// prof (optional, 8 floats): mean device ms per iteration of {whole iteration, wait for n_pr at its end,
// P tables + W, pass 1, n + publish + pr partial, (wait +) pass 2, n + publish} and the HOST ms it took to issue
// an iteration; measuring
// synchronises every iteration (which serialises the overlap: stage times, not a throughput figure).
extern "C" int mmsbm_em_run_sharded(const mmsbm_shard_t* shp, int32_t iterations, double* theta_a, double* eta_a,
                                    double* pr_a, double* theta_b, double* eta_b, double* pr_b, int32_t half,
                                    void* ws, size_t ws_bytes, void* stream, float* prof) {
  int rc = check_shard(shp, "mmsbm_em_run_sharded");
  if (rc) return rc;
  const mmsbm_shard_t& sh = *shp;
  MMSBM_REQUIRE(iterations >= 0 && theta_a && eta_a && pr_a && theta_b && eta_b && pr_b && ws &&
                    (half == 0 || half == 1), MMSBM_EINVAL, "mmsbm_em_run_sharded: bad argument");
  MMSBM_REQUIRE(sh.useg_dev && sh.udeg_dev && sh.usched_dev && sh.iseg_dev && sh.ideg_dev && sh.isched_dev &&
                    (sh.n_ratings_u == 0 || sh.uadj_dev) && (sh.n_ratings_i == 0 || sh.iadj_dev), MMSBM_EINVAL,
                "mmsbm_em_run_sharded: null index pointer");
  const bool peers = sh.world > 1;
  if (peers && (rc = nccl_ready())) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int S = sh.n_runs, R = sh.n_levels, K = sh.K, L = sh.L;
  const int Uo = sh.n_users_own, Io = sh.n_items_own;
  const ShardDims d = shard_dims(sh);
  const GridLayout g = grid_layout(sh.n_users, sh.n_items, K, L, R, S);
  Arena arena(ws, ws_bytes);
  double* pw_u = arena.take<double>(d.p_elems);
  double* pn_u = arena.take<double>(d.p_elems);
  double* pw_i = arena.take<double>(d.p_elems);
  double* pn_i = arena.take<double>(d.p_elems);
  double* wg_u = arena.take<double>(d.wg_u);
  double* wg_i = arena.take<double>(d.wg_i);
  double* partial = arena.take<double>(d.partial);
  double* slots_u = arena.take<double>(d.slots_u);
  double* slots_i = arena.take<double>(d.slots_i);
  int32_t* counters = arena.take<int32_t>(d.ctr);
  MMSBM_REQUIRE(pw_u && pn_u && pw_i && pn_i && wg_u && wg_i && partial && slots_u && slots_i && counters,
                MMSBM_ENOMEM, "mmsbm_em_run_sharded: workspace too small (%zu)", ws_bytes);

  Exchange ex;
  if ((rc = ex.open(sh.world))) return rc;
  constexpr int kProf = 7;
  cudaEvent_t ev[kProf] = {nullptr};
  struct Cleanup {
    cudaEvent_t* ev;
    ~Cleanup() {
      for (int k = 0; k < kProf; ++k) if (ev[k]) cudaEventDestroy(ev[k]);
      set_reserved_ctas(0);
    }
  } cleanup{ev};
  if (prof) for (int k = 0; k < kProf; ++k) MMSBM_CUDA(cudaEventCreate(&ev[k]));
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define MMSBM_MARK(k) do { if (prof) MMSBM_CUDA(cudaEventRecord(ev[k], st)); } while (0)

  const int64_t n_big = sh.n_ratings_u > sh.n_ratings_i ? sh.n_ratings_u : sh.n_ratings_i;
  // launch-wide piece queues from 1M ratings on a rank (one GPU: from 4M): with a rank's share of the
  // pieces a warp gets only a few, and claiming them dynamically evens the tails out (measured on one
  // rank's share of ML-20M / 8: 0.907 -> 0.897 ms per iteration)
  const bool dyn = env_int("MMSBM_DYN", n_big >= ((int64_t)1 << 20) ? 1 : 0) != 0;
  const bool alternate = peers;
  const bool overlap = peers;                   // aux stream beside the main one
  // persistent CTAs of the passes leave a few slots free so that the NCCL kernels of the side stream
  // can start while a pass runs
  if (peers) set_reserved_ctas(4);
  const void* mine = sh.exchange_dev[sh.rank];
  if (peers) {                                  // the side stream starts behind everything queued on `st`
    MMSBM_CUDA(cudaEventRecord(ex.partial, st));
    MMSBM_CUDA(cudaStreamWaitEvent(ex.side, ex.partial, 0));
  }
  bool have_arrival[2] = {false, false};        // an arrival barrier of this call is pending for [theta, eta]

  for (int it = 0; it < iterations; ++it) {
    const bool fwd = (it & 1) == 0;
    const int cur = half ^ (it & 1), nxt = cur ^ 1;
    const double* th = fwd ? theta_a : theta_b; const double* et = fwd ? eta_a : eta_b;
    const double* pr = fwd ? pr_a : pr_b;
    double* th_n = fwd ? theta_b : theta_a; double* et_n = fwd ? eta_b : eta_a; double* pr_n = fwd ? pr_b : pr_a;
    const bool users_first = !alternate || (it & 1) == 0;
    // n_pr comes from the g rows of the side with fewer segments (accumulating over 480k users instead of
    // 17.7k items costs more than an exposed all-reduce); when that side is pass 1 its all-reduce hides
    // behind pass 2
    const bool emit_items = d.emit_items;
    const bool emit_after_pass1 = peers && (emit_items != users_first);

    // what follows a pass (n contraction, interleave into the next tables, push, n_pr partial) runs on `fs`:
    // the main stream, or -- after pass 1, with peers -- the AUX stream, so that it overlaps pass 2
    auto pass_users = [&]() -> int {            // gathers eta rows of ALL items, new theta rows of the own users
      if (have_arrival[1]) MMSBM_CUDA(cudaStreamWaitEvent(st, ex.arrived[1][(it + 1) & 1], 0));
      SegArgs a{sh.useg_dev, sh.uadj_dev, sh.usched_dev, table_ptr(mine, g, cur, g.eta[2]), wg_u, slots_u, d.pmax_u,
                d.lmax_u, d.smax_u, Uo, sh.n_items, d.ldl, R, 0, 0, 0, dyn ? counters : nullptr};
      return launch_segment_pass_and_fixup(a, table_ptr(mine, g, cur, g.eta[1]), table_ptr(mine, g, cur, g.eta[0]),
                                           sh.n_ratings_u, S, st);
    };
    // (row_n_kernel stores the new rows twice: plain into the own buffer and, interleaved, into the own
    //  slice of the next gather tables -- no separate interleave pass)
    auto finish_users = [&](cudaStream_t fs) -> int {
      const RowPublish pub = row_publish(mine, g, g.theta, 2, nxt, sh.n_users, sh.user_lo);
      int r = launch_n(wg_u, pn_u, th, sh.udeg_dev, th_n, Uo, d.ldk, d.rnb_u, 1, S, fs, &pub);
      if (r) return r;
      return publish_side(sh, g, g.theta, 2, nullptr, Uo, sh.user_lo, nxt, fs, ex);
    };
    auto pass_items = [&]() -> int {            // gathers theta rows of ALL users, new eta rows of the own items
      if (have_arrival[0]) MMSBM_CUDA(cudaStreamWaitEvent(st, ex.arrived[0][(it + 1) & 1], 0));
      SegArgs a{sh.iseg_dev, sh.iadj_dev, sh.isched_dev, table_ptr(mine, g, cur, g.theta[1]), wg_i, slots_i, d.pmax_i,
                d.lmax_i, d.smax_i, Io, sh.n_users, d.ldk, R, 0, 0, 0, dyn ? counters + d.ctr / 2 : nullptr};
      return launch_segment_pass_and_fixup(a, table_ptr(mine, g, cur, g.theta[0]), nullptr, sh.n_ratings_i, S, st);
    };
    auto finish_items = [&](cudaStream_t fs) -> int {
      const RowPublish pub = row_publish(mine, g, g.eta, 3, nxt, sh.n_items, sh.item_lo);
      int r = launch_n(wg_i, pn_i, et, sh.ideg_dev, et_n, Io, d.ldl, d.rnb_i, 1, S, fs, &pub);
      if (r) return r;
      return publish_side(sh, g, g.eta, 3, nullptr, Io, sh.item_lo, nxt, fs, ex);
    };
    auto reduce_pr = [&](cudaStream_t fs) -> int {   // partial n_pr on fs, its sum over the ranks on the side stream
      int r = launch_pr(emit_items ? et : th, emit_items ? wg_i : wg_u, partial, pr, pr_n, emit_items ? Io : Uo,
                        emit_items ? L : K, emit_items ? d.ldl : d.ldk, emit_items ? d.ldk : d.ldl, K, L, R, S,
                        emit_items, !peers, fs);
      if (r || !peers) return r;
      MMSBM_CUDA(cudaEventRecord(ex.partial, fs));
      MMSBM_CUDA(cudaStreamWaitEvent(ex.side, ex.partial, 0));
      MMSBM_NCCL(g_nccl.AllReduce(pr_n, pr_n, (size_t)S * K * L * R, ncclFloat64, ncclSum,
                                  static_cast<ncclComm_t>(sh.nccl_comm), ex.side));
      MMSBM_CUDA(cudaEventRecord(ex.pr_done, ex.side));
      return 0;
    };
    auto after_publish = [&](int which) -> int {   // side stream: arrival barrier of table `which`
      if (!peers) return 0;
      return barrier_on_side(sh, g, ex, ex.arrived[which][it & 1]);
    };
    cudaStream_t aux = overlap ? ex.aux : st;

    const auto host_t0 = std::chrono::steady_clock::now();
    MMSBM_MARK(0);
    if (dyn) MMSBM_CUDA(cudaMemsetAsync(counters, 0, d.ctr * 4, st));
    if ((rc = launch_prep_p(pr, K, L, R, d.ldk, d.ldl, S, pw_u, pn_u, pw_i, pn_i, st))) return rc;
    if (overlap) {                              // W of pass 2's side on the aux stream, beside pass 1
      MMSBM_CUDA(cudaEventRecord(ex.p_ready, st));
      MMSBM_CUDA(cudaStreamWaitEvent(aux, ex.p_ready, 0));
    }
    if (users_first) {
      if ((rc = launch_w(th, pw_u, wg_u, Uo, d.ldk, d.rnb_u, S, st))) return rc;
      if ((rc = launch_w(et, pw_i, wg_i, Io, d.ldl, d.rnb_i, S, aux))) return rc;
    } else {
      if ((rc = launch_w(et, pw_i, wg_i, Io, d.ldl, d.rnb_i, S, st))) return rc;
      if ((rc = launch_w(th, pw_u, wg_u, Uo, d.ldk, d.rnb_u, S, aux))) return rc;
    }
    if (overlap) MMSBM_CUDA(cudaEventRecord(ex.w2_ready, aux));
    MMSBM_MARK(1);
    // ---- pass 1; its epilogue goes to the aux stream ----
    if ((rc = users_first ? pass_users() : pass_items())) return rc;
    MMSBM_MARK(2);
    if (overlap) {
      MMSBM_CUDA(cudaEventRecord(ex.pass1_done, st));
      MMSBM_CUDA(cudaStreamWaitEvent(aux, ex.pass1_done, 0));
    }
    if ((rc = users_first ? finish_users(aux) : finish_items(aux))) return rc;
    if (emit_after_pass1 && (rc = reduce_pr(aux))) return rc;
    if ((rc = after_publish(users_first ? 0 : 1))) return rc;
    if (overlap) MMSBM_CUDA(cudaEventRecord(ex.aux_done, aux));
    MMSBM_MARK(3);
    // ---- pass 2 ----
    if (overlap) MMSBM_CUDA(cudaStreamWaitEvent(st, ex.w2_ready, 0));
    if ((rc = users_first ? pass_items() : pass_users())) return rc;
    MMSBM_MARK(4);
    if (!emit_after_pass1) {                    // n_pr from pass 2's side: beside its n contraction, on the aux stream
      if (overlap) {
        MMSBM_CUDA(cudaEventRecord(ex.pass1_done, st));
        MMSBM_CUDA(cudaStreamWaitEvent(aux, ex.pass1_done, 0));
      }
      if ((rc = reduce_pr(aux))) return rc;
      if (overlap) MMSBM_CUDA(cudaEventRecord(ex.aux_done, aux));
    }
    if ((rc = users_first ? finish_items(st) : finish_users(st))) return rc;
    if ((rc = after_publish(users_first ? 1 : 0))) return rc;
    MMSBM_MARK(5);
    if (overlap) MMSBM_CUDA(cudaStreamWaitEvent(st, ex.aux_done, 0));
    if (peers) {
      MMSBM_CUDA(cudaStreamWaitEvent(st, ex.pr_done, 0));
      if ((rc = launch_finalize_pr(pr_n, S * K * L, R, st))) return rc;
      have_arrival[0] = have_arrival[1] = true;  // from now on every pass waits for the previous iteration's barrier
    }
    MMSBM_MARK(6);
    if (prof) {
      acc[7] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count();
      MMSBM_CUDA(cudaEventSynchronize(ev[6]));
      float t = 0.f;
      cudaEventElapsedTime(&t, ev[0], ev[6]); acc[0] += t;
      cudaEventElapsedTime(&t, ev[5], ev[6]); acc[1] += t;
      for (int k = 0; k < 5; ++k) { cudaEventElapsedTime(&t, ev[k], ev[k + 1]); acc[2 + k] += t; }
    }
  }
#undef MMSBM_MARK
  if (peers && iterations > 0) {                // drain: every table complete everywhere before the call returns its stream
    MMSBM_CUDA(cudaStreamWaitEvent(st, ex.arrived[0][(iterations - 1) & 1], 0));
    MMSBM_CUDA(cudaStreamWaitEvent(st, ex.arrived[1][(iterations - 1) & 1], 0));
  }
  if (prof) for (int k = 0; k < 8; ++k) prof[k] = iterations > 0 ? (float)(acc[k] / iterations) : 0.f;
  return 0;
}
