// tlc_api.cu -- host orchestration and the C-ABI of libtlc_b200.so (include/tlc_b200.h).
//
// A call processes its targets in CHUNKS.  The counting pass of kernel 1 gives every target's vicinity size; the host
// orders the live targets (shared-memory class, size: largest first), packs as many as fit the HBM arena, and
// runs the stage kernels over the chunk.  Two routes (chosen per call, same results bit for bit):
//   materialised : 1 fill -> 1b filtration -> 2v vertex order -> 3v sweep -> [1c edge list -> 2 sort -> 3 union-find
//                  (descending sweep, Pos/Neg lists, targets 3v handed back)] -> [3b loops] -> 4 image
//   graph-row    : (light counting pass) -> 1b filtration on the graph's own CSR rows -> 2v -> 3v -> 4 image
//                  -- ascending-sweep-only calls on vicinities that are dense in the graph; no adjacency in HBM
// Per-target segments of every array are addressed through exclusive offsets uploaded per chunk; the image kernel
// scatters rows to their final position, so results keep the caller's target order.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#include "tlc_common.cuh"

namespace tlc {
static std::atomic_llong g_launches{0};
int64_t launch_count() { return g_launches.load(); }
void count_launch() { g_launches.fetch_add(1); }
}  // namespace tlc

using namespace tlc;

static thread_local std::string g_err;
static int fail(int rc, const std::string& msg) {
  g_err = msg;
  return rc;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(TLC_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_) + " @" + __FILE__ + ":" + \
                                  std::to_string(__LINE__));                                       \
  } while (0)

// device or pinned host memory owned by one object: freed by its destructor on every exit path (the CK macro returns
// early), by tlc_graph's destructor for the graph's buffers
template <cudaError_t (*Alloc)(void**, size_t), cudaError_t (*Free)(void*)>
struct Owned {
  void* p = nullptr;
  size_t bytes = 0;
  Owned() = default;
  Owned(Owned&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
  Owned& operator=(Owned&& o) noexcept {
    if (this != &o) { release(); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; }
    return *this;
  }
  ~Owned() { release(); }
  void release() { if (p) Free(p); p = nullptr; bytes = 0; }
  // grow-only; a larger block is allocated after the old one is freed, so the two never coexist
  cudaError_t reserve(size_t n) {
    if (p && n <= bytes) return cudaSuccess;
    release();
    const cudaError_t e = Alloc(&p, n ? n : 16);
    if (e == cudaSuccess) bytes = n; else p = nullptr;
    return e;
  }
  template <typename T_> T_* as() const { return static_cast<T_*>(p); }
};
using DevBuf = Owned<cudaMalloc, cudaFree>;
using PinBuf = Owned<cudaMallocHost, cudaFreeHost>;

static constexpr size_t ALIGN = 256;
static size_t align_up(size_t x) { return (x + ALIGN - 1) / ALIGN * ALIGN; }

// bytes of arena per vertex / edge / pair slot (see carve())
static constexpr size_t BV = 4 * 6 + 8 * 3 + 8 * 3 + 4 * 6;           // vert vcls vs0 vs1 vs2 neg | fval d1 d2 | v64a v64b v64c | vord vrank bfirst astart adeg aminw
static constexpr size_t BE = 4 * 4 + 8 + 4 * 4 + 8 * 2 + 1;           // elo ehi pos arank | ew | ord_asc ord_desc sp0 sp1 | sk0 sk1 | isneg
static constexpr size_t BA = 4 + 8;                                   // anb | aw, per adjacency slot
static constexpr size_t BP = 1 + 4 * 2 + 8 * 2;                       // pkind | pbv pdv | pbirth pdeath
static constexpr size_t BT = 8 * 4 + 4 * 11 + 2 + 4;                  // tidx voff eoff aoff | tn tm tlu tlv tnp tnpos tnneg tncls tnb tminv tmaxv | tstatus tfb | bfirst terminator

// what the tlc_last_* functions report about the last call
struct CallStats {
  double stage_ms[10] = {0};
  int chunks = 0;
  int64_t live = 0, sum_n = 0, sum_m = 0;                    // targets with status <= TRIVIAL, their vertices / edges
  int64_t handed_back = 0, general = 0, rowcheck = 0, blocks = 0;  // sweep counters of kernels 2v / 3v
  int64_t direct = 0, table = 0;  // targets that took the graph-row route, those of them filtered from the tables
  int64_t two_root = 0;            // ... and those kernel 1t ran with both roots in the same passes
  double bytes = 0;               // compulsory bytes (SURVEY.md 8d)
  double small_ms[3] = {0, 0, 0};
  int64_t small_rows[4] = {0, 0, 0, 0};  // rows finished by kernel S's class A / B / C, rows handed to the staged pipeline
  CallStats& operator+=(const CallStats& o) {
    for (int i = 0; i < 10; i++) stage_ms[i] += o.stage_ms[i];
    for (int i = 0; i < 3; i++) small_ms[i] += o.small_ms[i];
    for (int i = 0; i < 4; i++) small_rows[i] += o.small_rows[i];
    chunks += o.chunks; live += o.live; sum_n += o.sum_n; sum_m += o.sum_m; handed_back += o.handed_back;
    general += o.general; rowcheck += o.rowcheck; blocks += o.blocks; direct += o.direct; table += o.table;
    two_root += o.two_root;
    bytes += o.bytes;
    return *this;
  }
};

// grow b to `need` bytes keeping its first `used` bytes (DevBuf::reserve frees before it allocates and loses them)
static cudaError_t grow_keep(DevBuf& b, size_t used, size_t need, cudaStream_t st) {
  if (b.p && need <= b.bytes) return cudaSuccess;
  DevBuf nb;
  cudaError_t e = nb.reserve(need);
  if (e == cudaSuccess && used) e = cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) b = std::move(nb);
  return e;
}

// a pair array set owned by the graph: capacity in pairs, grow-only
struct PairBufs {
  DevBuf kind, bv, dv, birth, death;
  int64_t cap = 0;
  DiagArea view() const {
    return DiagArea{kind.as<uint8_t>(), bv.as<int32_t>(), dv.as<int32_t>(), birth.as<double>(), death.as<double>()};
  }
  // room for `need` pairs; the first `used` pairs are kept
  cudaError_t grow(int64_t used, int64_t need, cudaStream_t st) {
    if (need <= cap && kind.p) return cudaSuccess;
    const int64_t n = std::max<int64_t>(need, cap + cap / 2);
    cudaError_t e = cudaSuccess;
    DevBuf* bufs[5] = {&kind, &bv, &dv, &birth, &death};
    const size_t sz[5] = {1, 4, 4, 8, 8};
    for (int i = 0; i < 5 && e == cudaSuccess; i++) e = grow_keep(*bufs[i], (size_t)used * sz[i], (size_t)n * sz[i] + 16, st);
    if (e == cudaSuccess) cap = n;
    return e;
  }
};

// the pairs of a tlc_vicinity_diagrams call while it runs.  Every target's diagram is one contiguous segment of the
// staging: kernel S writes its rows into `small` at offsets fixed before it runs, the staged pipeline's chunks are
// exported into `staged` (staging offsets >= small_total); np / soff record count and offset per target of the call.
struct DiagCollect {
  bool on = false;
  DevBuf np, soff, poff;  // [E] int32, [E] int64, [E + 1] int64 (host entry point: the final offsets)
  PairBufs small, staged, out;  // out: the host entry point's gathered arrays before they are copied back
  int64_t small_total = 0, staged_used = 0;
  DevBuf chunk;  // per chunk: staging offset and call row of each target
};

// the outputs of a tlc_vicinity_batch_dev call while it runs: voff / eoff hold the final offsets before the first chunk,
// every chunk's targets are exported into the arrays at those offsets
struct BatchCollect {
  bool on = false;
  tlc_vicinity_batch out{};
  uint8_t* status = nullptr;
  int64_t total_v = 0, total_e = 0;
};

struct tlc_graph {
  int device = 0;
  GraphView gv{};  // views of rowptr / col / kappa / rec
  DevBuf rowptr, col, kappa, rec;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  // the filtration launches of a chunk's sub-ranges are independent: they run on side streams, forked from / joined to
  // the call's stream with events, so that the tail wave of one sub-range is filled by CTAs of the next
  cudaStream_t side[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr};
  DevBuf arena;
  size_t arena_req = 0;
  // vicinity scratch (depends on hop)
  DevBuf bitmaps, queue;
  // ball cache (valid for vic_hop)
  DevBuf ball_cache, ball_acc, ball_state, ball_list;
  int vic_grid = 0, vic_hop = -1;
  DevBuf work_counter;
  ChunkView detail_chunk{};  // the chunk of the last tlc_vicinity_detail call (still carved in the arena)
  DevBuf gminw;  // [N] float: smallest kappa + 1 of each node's row, rounded down (graph-row route's settling margin)
  // density probe of the graph-row route (per hop / mode): decision and calls since it was taken
  int probe_hop = -1, probe_mode = -1, probe_age = 0;
  bool probe_direct = false;
  // per-call device buffers
  DevBuf d_n, d_m, d_ds, d_st, d_bytes;
  int64_t call_cap = 0;
  // device staging of the host-buffer entry point (tlc_vicinity_pi): targets in, image rows + status out
  DevBuf io_t, io_pi, io_st;
  int64_t io_cap_t = 0, io_cap_pi = 0;
  PinBuf h_pin;  // host staging
  CallStats last;
  // kernel S (fused small-vicinity path): deferral lists, counters + statistics, their pinned host mirror
  DevBuf sm_list_b, sm_list_c, sm_list_big, sm_list_b2;
  cudaStream_t small_stream2 = nullptr;  // ... class C beside class B
  cudaEvent_t ev_small_c = nullptr;
  cudaStream_t small_stream = nullptr;   // classes B / C of kernel S run here while the staged pipeline takes the big targets
  cudaEvent_t ev_small_a = nullptr, ev_small_bc = nullptr;
  DevBuf sm_sub;    // [cap][2] targets handed on to the staged pipeline
  DevBuf sm_idx;    // [cap] their rows
  DevBuf sm_pi;     // [cap][r2] staged results of those rows, scattered back
  DevBuf sm_pi32, sm_st;
  int64_t sm_cap = 0, sm_sub_cap = 0;
  DevBuf sm_dev;    // [int counters[2] | pad | SmallStats]
  PinBuf sm_host;   // pinned mirror
  int small_skip = 0;              // calls left for which the small path is not tried (it handled too few rows)
  int small_hop = -1, small_mode = -1;
  double hks_time = 0.1;   // diffusion time of TLC_F_FILT_HKS (data_utils_NC.py: hks_time = 0.1)
  // kernel 1t: per-root shortest-path tables over the roots' k-hop balls (valid for sssp_plain and sssp_hop), scratch of
  // the build kernel
  SsspTables sssp{};  // views of the sssp_* buffers, null until they exist
  DevBuf sssp_D, sssp_P, sssp_QW, sssp_state, sssp_list, sssp_count, sssp_pw;
  int sssp_plain = -1, sssp_hop = -1;
  bool sssp_tried = false, sssp_all = false;
  double sssp_build_ms = 0;   // device time of the (one-time) table build
  // multi-GPU exchange by peer stores: this rank's table, the mapped tables of all ranks, exchange epoch
  DevBuf peer_own;
  int64_t peer_rows = 0;
  int peer_r2 = 0;
  PeerTables peers{};
  std::vector<void*> peer_opened;   // tables mapped with cudaIpcOpenMemHandle
  unsigned int peer_epoch = 0;
  DevBuf peer_ticket;
  DevBuf px_pi32, px_pi, px_st;     // [cap][r2] staging of the shard's rows
  int64_t px_cap = 0;
  std::vector<cudaEvent_t> ev_pool;  // stage-timing events, reused from call to call
  int sm_count = 0;
  DiagCollect dg;
  BatchCollect vb;

  ~tlc_graph() {
    for (void* q : peer_opened) cudaIpcCloseMemHandle(q);
    for (cudaStream_t s : {own_stream, side[0], side[1], side[2], small_stream, small_stream2})
      if (s) cudaStreamDestroy(s);
    for (cudaEvent_t e : {ev_fork, ev_join[0], ev_join[1], ev_join[2], ev_small_a, ev_small_bc, ev_small_c})
      if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ev_pool) cudaEventDestroy(e);
  }
};

static int ensure_call_buffers(tlc_graph* g, int64_t E) {
  if (E <= g->call_cap) return TLC_OK;
  const size_t cap = (size_t)(E + E / 8 + 1024);
  CK(g->d_n.reserve(cap * 4));
  CK(g->d_m.reserve(cap * 4));
  CK(g->d_ds.reserve(cap * 4));
  CK(g->d_st.reserve(cap));
  CK(g->d_bytes.reserve(cap * 8));
  g->call_cap = (int64_t)cap;
  return TLC_OK;
}

static int ensure_io_buffers(tlc_graph* g, int64_t E, int r2) {
  const int64_t cap = E + E / 8 + 1024;
  if (E > g->io_cap_t) {
    CK(g->io_t.reserve((size_t)cap * 8));
    CK(g->io_st.reserve((size_t)cap));
    g->io_cap_t = cap;
  }
  if (E * r2 > g->io_cap_pi) {
    CK(g->io_pi.reserve((size_t)cap * r2 * 8));
    g->io_cap_pi = cap * r2;
  }
  return TLC_OK;
}

// the configured arena size: tlc_graph_create's arena_bytes, else TLC_ARENA_GB, default 24 GiB
static size_t arena_limit(const tlc_graph* g) {
  if (g->arena_req) return g->arena_req;
  const char* env = getenv("TLC_ARENA_GB");
  return (size_t)((env ? atof(env) : 24.0) * (double)(1ull << 30));
}

// grow-only arena: at least `need_min` (one chunk must fit), preferably `need_all` (the whole call in one chunk), never
// more than arena_limit() or 85 % of free memory
static int ensure_arena(tlc_graph* g, size_t need_min, size_t need_all) {
  const size_t limit = arena_limit(g);
  // large enough for a chunk; grow only if the call would otherwise be split and there is headroom left
  if (g->arena.p && g->arena.bytes >= need_min && g->arena.bytes >= std::min(need_all, limit)) return TLC_OK;
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  const size_t had = g->arena.bytes;
  free_b += had;
  g->arena.release();  // (also when free memory is short and the new arena ends up smaller)
  size_t want = std::max(std::min(limit, need_all + need_all / 2), need_min);  // (no 24 GiB for a handful of small vicinities; 50 % headroom: calls of similar size do not reallocate)
  // a floor and geometric growth: the handful of large vicinities kernel S leaves to the staged pipeline differs a lot
  // from call to call, and every reallocation is a device-wide synchronisation (measured: 10 - 60 ms per call)
  want = std::max(want, std::min(limit, std::max<size_t>(2 * had, (size_t)256 << 20)));
  const size_t cap = (size_t)((double)free_b * 0.85);
  if (want > cap) want = cap;
  if (want < need_min)
    return fail(TLC_E_NOMEM, "one vicinity needs " + std::to_string(need_min) + " arena bytes, only " +
                                 std::to_string(cap) + " available");
  CK(g->arena.reserve(want));
  return TLC_OK;
}

static VicinityScratch make_vs(const tlc_graph* g) {
  return VicinityScratch{g->bitmaps.as<uint32_t>(), g->queue.as<int32_t>(), g->vic_grid, g->ball_cache.as<uint32_t>(),
                         g->ball_acc.as<unsigned long long>(), g->ball_state.as<int32_t>(), g->ball_list.as<int32_t>(),
                         g->work_counter.as<int>() + 2};
}

static int ensure_vicinity_scratch(tlc_graph* g, const Params& p) {
  if (g->vic_hop == p.hop && g->vic_grid > 0) return TLC_OK;
  for (DevBuf* b : {&g->bitmaps, &g->queue, &g->ball_cache, &g->ball_acc, &g->ball_state, &g->ball_list}) b->release();
  {
    // one bitmap row per node, if that is affordable (TLC_BALL_CACHE_GB, default 16; 0 disables)
    const char* env = getenv("TLC_BALL_CACHE_GB");
    const double gb = env ? atof(env) : 16.0;
    const size_t Wc = ((size_t)g->gv.N + 31) / 32;
    const size_t need = (size_t)g->gv.N * Wc * sizeof(uint32_t);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    if (gb > 0 && (double)need <= gb * (double)(1ull << 30) && need <= free_b / 4) {
      CK(g->ball_cache.reserve(std::max<size_t>(need, 16)));
      CK(g->ball_acc.reserve((size_t)g->gv.N * 2 * sizeof(unsigned long long)));
      CK(g->ball_state.reserve((size_t)g->gv.N * sizeof(int32_t)));
      CK(g->ball_list.reserve((size_t)g->gv.N * sizeof(int32_t)));
      CK(cudaMemset(g->ball_state.p, 0, (size_t)g->gv.N * sizeof(int32_t)));
    }
  }
  size_t W = 0;
  bool smem = false;
  g->vic_grid = vicinity_grid(g->device, g->gv, p, &W, &smem);
  if (!smem) CK(g->bitmaps.reserve((size_t)g->vic_grid * 2 * W * sizeof(uint32_t)));
  if (p.hop > 2) CK(g->queue.reserve((size_t)g->vic_grid * 2 * (size_t)g->gv.N * sizeof(int32_t)));
  g->vic_hop = p.hop;
  return TLC_OK;
}

// the opening of every entry point that expands vicinities
static int prepare_call(tlc_graph* g, const Params& p, int64_t E) {
  int rc = ensure_call_buffers(g, E);
  return rc ? rc : ensure_vicinity_scratch(g, p);
}

// kernel 1t's tables: three [N][N] arrays (D, P, {Q, W}), allocated once when the graph is small enough (N <= 16384: the
// build kernel keeps a root's whole distance / parent vector and ball in shared memory) and 28 N^2 bytes fit
// TLC_SSSP_CACHE_GB (default 8, 0 disables).  Their rows depend on the summation rule (path sums) and the hop (the ball
// each row is restricted to): a call with another of either marks every row for rebuilding.
static int ensure_sssp_tables(tlc_graph* g, const Params& p) {
  const int plain = (p.flags & TLC_F_SUM_PLAIN) ? 1 : 0;
  if (!g->sssp_tried) {
    g->sssp_tried = true;
    const char* env = getenv("TLC_SSSP_CACHE_GB");
    const double gb = env ? atof(env) : 8.0;
    const size_t N = (size_t)g->gv.N;
    const size_t need = N * N * (8 + 4 + 16);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    if (gb > 0 && N <= 16384 && (double)need <= gb * (double)(1ull << 30) && need <= free_b / 3 &&
        sssp_build_smem((int)N) <= 227 * 1024) {
      CK(g->sssp_D.reserve(N * N * 8));
      CK(g->sssp_P.reserve(N * N * 4));
      CK(g->sssp_QW.reserve(N * N * 16));
      CK(g->sssp_state.reserve(N * 4));
      CK(g->sssp_list.reserve(N * 4));
      CK(g->sssp_count.reserve(64));
      CK(g->sssp_pw.reserve((size_t)g->sm_count * N * 8));
      CK(cudaMemset(g->sssp_state.p, 0, N * 4));
      g->sssp = SsspTables{g->sssp_D.as<double>(), g->sssp_P.as<int32_t>(), g->sssp_QW.as<double2>(),
                           g->sssp_state.as<int32_t>(), g->sssp_list.as<int32_t>(), g->sssp_count.as<int>()};
      g->sssp_plain = plain;
      g->sssp_hop = p.hop;
    }
  }
  if (g->sssp.D && (g->sssp_plain != plain || g->sssp_hop != p.hop)) {
    CK(cudaMemsetAsync(g->sssp.state, 0, (size_t)g->gv.N * 4, g->stream));
    g->sssp_plain = plain;
    g->sssp_hop = p.hop;
    g->sssp_all = false;
  }
  return TLC_OK;
}

// carve the arena for a chunk with T targets, Nv vertices, Ne edges (pairs = Nv + Ne + T)
static size_t chunk_bytes(int64_t T, int64_t Nv, int64_t Ne, int64_t Na, int64_t Wd = 0) {
  const int64_t Np = Nv + Ne + T;
  // every array individually aligned: 16 vertex arrays, 13 edge arrays, 5 pair arrays, 16 target arrays;
  // Wd > 0 (graph-row route): bitmap + word prefix of every target
  return (size_t)(Nv * BV + Ne * BE + Na * BA + Np * BP + (T + 1) * BT + T * Wd * 8) + ALIGN * 60;
}

template <typename T_>
static T_* take(char*& cur, int64_t count) {
  T_* p = reinterpret_cast<T_*>(cur);
  cur += align_up((size_t)count * sizeof(T_));
  return p;
}

static ChunkView carve(char* arena, int64_t T, int64_t Nv, int64_t Ne, int64_t Na, const int32_t* d_targets,
                       int64_t Wd = 0) {
  ChunkView c{};
  char* cur = arena;
  const int64_t Np = Nv + Ne + T;
  c.T = (int32_t)T;
  c.tgt = d_targets;
  c.tidx = take<int64_t>(cur, T);
  c.voff = take<int64_t>(cur, T + 1);
  c.eoff = take<int64_t>(cur, T + 1);
  c.aoff = take<int64_t>(cur, T + 1);
  c.tn = take<int32_t>(cur, T); c.tm = take<int32_t>(cur, T); c.tlu = take<int32_t>(cur, T); c.tlv = take<int32_t>(cur, T);
  c.tnp = take<int32_t>(cur, T); c.tnpos = take<int32_t>(cur, T); c.tnneg = take<int32_t>(cur, T); c.tncls = take<int32_t>(cur, T);
  c.tnb = take<int32_t>(cur, T); c.tminv = take<int32_t>(cur, T); c.tmaxv = take<int32_t>(cur, T);
  c.tstatus = take<uint8_t>(cur, T);
  c.tfb = take<uint8_t>(cur, T);
  c.vord = take<int32_t>(cur, Nv); c.vrank = take<int32_t>(cur, Nv);
  c.bfirst = take<int32_t>(cur, Nv + T);
  c.astart = take<int32_t>(cur, Nv); c.adeg = take<int32_t>(cur, Nv); c.aminw = take<float>(cur, Nv);
  c.anb = take<uint32_t>(cur, Na); c.aw = take<double>(cur, Na);
  c.vert = take<int32_t>(cur, Nv); c.vcls = take<int32_t>(cur, Nv); c.vs0 = take<int32_t>(cur, Nv);
  c.vs1 = take<int32_t>(cur, Nv); c.vs2 = take<int32_t>(cur, Nv); c.neg = take<int32_t>(cur, Nv);
  c.fval = take<double>(cur, Nv); c.d1 = take<double>(cur, Nv); c.d2 = take<double>(cur, Nv);
  c.v64a = take<unsigned long long>(cur, Nv); c.v64b = take<unsigned long long>(cur, Nv);
  c.v64c = take<unsigned long long>(cur, Nv);
  c.elo = take<int32_t>(cur, Ne); c.ehi = take<int32_t>(cur, Ne); c.pos = take<int32_t>(cur, Ne);
  c.arank = take<int32_t>(cur, Ne);
  c.ew = take<double>(cur, Ne);
  c.ord_asc = take<uint32_t>(cur, Ne); c.ord_desc = take<uint32_t>(cur, Ne);
  c.sp0 = take<uint32_t>(cur, Ne); c.sp1 = take<uint32_t>(cur, Ne);
  c.sk0 = take<unsigned long long>(cur, Ne); c.sk1 = take<unsigned long long>(cur, Ne);
  c.isneg = take<uint8_t>(cur, Ne);
  c.pkind = take<uint8_t>(cur, Np);
  c.pbv = take<int32_t>(cur, Np); c.pdv = take<int32_t>(cur, Np);
  c.pbirth = take<double>(cur, Np); c.pdeath = take<double>(cur, Np);
  c.dbm = Wd > 0 ? take<uint32_t>(cur, T * 2 * Wd) : nullptr;
  c.W = (int32_t)Wd;
  return c;
}

static int block_for(int64_t m_max) {
  if (m_max >= 32768) return 512;
  if (m_max >= 4096) return 256;
  if (m_max >= 512) return 128;
  if (m_max >= 96) return 64;
  return 32;
}
static int size_class(int64_t m) { return block_for(m); }
// kernel 1b keeps 9 - 11 bytes of state per vertex in shared memory: 0 = does not fit at all (state in the arena),
// 1 = fits only in the lean layout, 2 = fits (thresholds a little under the kernel's own limits, which also hold bitmaps)
static int smem_class(int64_t n) { return n > 22000 ? 0 : (n > 16000 ? 1 : 2); }

struct StageTimer {
  // per-stage CUDA events (TLC_STAGE_TIMING=1).  The events come from a pool owned by the graph and are reused from call
  // to call: no cudaEventCreate / cudaEventDestroy inside a timed call once the pool has grown to a call's needs.
  bool on;
  cudaStream_t st;
  std::vector<cudaEvent_t>* pool;
  size_t used, first;  // next free pool slot; first slot of the marks not collected yet
  std::vector<int> stage;
  StageTimer(cudaStream_t s, std::vector<cudaEvent_t>* pool_, size_t start) : st(s), pool(pool_), used(start), first(start) {
    const char* env = getenv("TLC_STAGE_TIMING");
    on = env && atoi(env) != 0;
  }
  cudaEvent_t take() {
    if (used == pool->size()) { cudaEvent_t e; cudaEventCreate(&e); pool->push_back(e); }
    return (*pool)[used++];
  }
  void mark(int stage_id) {  // marks the START of stage_id (or the end marker with id -1)
    if (!on) return;
    cudaEventRecord(take(), st);
    stage.push_back(stage_id);
  }
  void collect(double* ms8) {  // ms8: per-stage accumulators (10 slots); call after the stream is synchronised
    if (!on) return;
    for (size_t i = 0; i + 1 < stage.size(); i++) {
      if (stage[i] < 0) continue;
      float ms = 0;
      cudaEventElapsedTime(&ms, (*pool)[first + i], (*pool)[first + i + 1]);
      ms8[stage[i]] += ms;
    }
    first = used;
    stage.clear();
  }
};

// run the stage kernels over one carved chunk (offsets already uploaded)
// kernels whose shared-memory footprint follows the vicinity size are launched per SUB-RANGE of the chunk's
// (size-sorted) targets, each with the capacity of its own largest vicinity: smaller vicinities get more
// resident CTAs per SM
struct SubRange { int t0, cnt; int64_t n_min, n_max; };

// launch(range, stream) for every sub-range; sub-ranges 1 - 3 run on the side streams, forked from / joined to `st`
template <typename F_>
static void for_subranges(const tlc_graph* g, const std::vector<SubRange>& subs, cudaStream_t st, F_ launch) {
  const bool fork = subs.size() > 1 && g->ev_fork != nullptr;
  if (fork) cudaEventRecord(g->ev_fork, st);
  for (size_t i = 0; i < subs.size(); i++) {
    cudaStream_t s = st;
    if (fork && i > 0 && i <= 3) { s = g->side[i - 1]; cudaStreamWaitEvent(s, g->ev_fork, 0); }
    launch(subs[i], s);
    if (s != st) { cudaEventRecord(g->ev_join[i - 1], s); cudaStreamWaitEvent(st, g->ev_join[i - 1], 0); }
  }
}

// kernel 1t filters a graph-row sub-range when the call has the tables and the sub-range's largest vicinity fits its
// shared memory
static bool takes_table(const tlc_graph* g, bool use_table, const SubRange& r) {
  return use_table && filtration_table_smem(g->gv.N, r.n_max) <= 226 * 1024;
}

// the filtration of a chunk: a structural one or HKS over the whole chunk, else kernel 1t / 1b per sub-range; returns
// the number of targets whose filtration came from kernel 1t's tables
static int64_t run_filtration(tlc_graph* g, const Params& p, const ChunkView& c, int64_t n_max, int block,
                              const std::vector<SubRange>& subs, bool use_table) {
  cudaStream_t st = g->stream;
  VicinityScratch vs = make_vs(g);
  int64_t from_table = 0;
  if (p.flags & TLC_F_FILT_HKS) launch_hks_filtration(p, c, g->hks_time, n_max, st);
  else if (p.flags & (TLC_F_FILT_DEGREE | TLC_F_FILT_CENTRALITY | TLC_F_FILT_CLUSTERING)) launch_degree_filtration(p, c, st);
  else {
    for_subranges(g, subs, st, [&](const SubRange& r, cudaStream_t s) {
      if (c.dbm && takes_table(g, use_table, r)) {
        launch_filtration_table(g->gv, p, c, vs, g->sssp, g->d_n.as<int32_t>(), r.t0, r.cnt, block, r.n_min, r.n_max, s);
        from_table += r.cnt;
      } else if (c.dbm) launch_filtration_direct(g->gv, p, c, vs, g->gminw.as<float>(), r.t0, r.cnt, block, r.n_max, s);
      else launch_filtration(p, c, r.t0, r.cnt, block, r.n_max, s);
    });
  }
  return from_table;
}

// returns the number of targets whose filtration came from kernel 1t's tables
static int64_t run_stages(tlc_graph* g, const Params& p, const ChunkView& c, int64_t n_max, int64_t m_max,
                          const std::vector<SubRange>& subs, double* d_pi, float* d_pi32, uint8_t* d_status,
                          bool want_lists, StageTimer& tm, bool use_table) {
  cudaStream_t st = g->stream;
  const int block = block_for(m_max);
  VicinityScratch vs = make_vs(g);
  tm.mark(1);
  if (!c.dbm) launch_vicinity_fill(g->gv, p, c, vs, g->work_counter.as<int>(), st);
  tm.mark(2);
  const int64_t from_table = run_filtration(g, p, c, n_max, block, subs, use_table);
  // ascending sweep: vertex-ordered kernels 2v + 3v; targets they hand back (tfb) and, when the descending
  // sweep is wanted (diagram output, Pos/Neg lists for the loops), the edge-sorted kernels 2 + 3.  The image
  // only needs PD_up and [min,max]: PD_down and [max,min] have death <= birth, i.e. weight 0 (SURVEY.md F6).
  const bool ext = (p.flags & TLC_F_EXTENDED) != 0;
  const bool want_desc = (ext || want_lists) && !(p.flags & TLC_F_ASC_ONLY);
  // keep-zero calls (PDGNN generators) that sort the edges anyway for the descending sweep: the vertex-ordered sweep has
  // no trivial blocks there (every merge emits a pair), so the ascending sweep rides on the edge-sorted kernels too
  const bool edge_sorted = (p.flags & TLC_F_EDGE_SORTED) != 0 || ((p.flags & TLC_F_KEEP_ZERO) != 0 && want_desc);
  tm.mark(3);
  if (edge_sorted) {
    cudaMemsetAsync(c.tfb, 1, (size_t)c.T, st);
  } else {
    // per sub-range like kernel 1b: 2v's block table and 3v's parents in shared memory are sized by the sub-range's
    // largest vicinity
    for_subranges(g, subs, st, [&](const SubRange& r, cudaStream_t s) { launch_vorder(p, c, r.t0, r.cnt, block, r.n_max, s); });
    tm.mark(4);
    for_subranges(g, subs, st, [&](const SubRange& r, cudaStream_t s) { launch_sweep(p, c, r.t0, r.cnt, r.n_max, s); });
  }
  tm.mark(5);
  if (!c.dbm) {  // (graph-row route: no adjacency to derive edges from; a chunk with handed-back targets is redone)
    // the edge-sorted kernels work on the canonical (lo, hi) edge list, derived from the adjacency where needed
    launch_edgelist(p, c, block, want_desc ? 0 : 1, st);
    // kernel 3b ranks loop edges by their position in the ascending order, so `extended` needs ord_asc of every target
    launch_sort(p, c, block, want_desc ? 3 : 1, want_desc ? 0 : 1, st);
  }
  tm.mark(6);
  const int64_t uf_ints = 2 * n_max * 4 <= 96 * 1024 ? 2 * n_max : 0;
  if (!c.dbm) launch_union_find(p, c, block, (int)uf_ints, want_desc ? 1 : 0, want_desc ? 3 : 1, 1, st);
  tm.mark(7);
  if (ext) {
    const int64_t lp_ints = 3 * n_max * 4 <= 200 * 1024 ? 3 * n_max : 0;
    launch_loops(p, c, std::min(block, 128), (int)lp_ints, n_max, st);
  }
  tm.mark(8);
  launch_pimg(p, c, d_pi, d_pi32, d_status, std::max(32, std::min(block, 256)), st);
  tm.mark(-1);
  return from_table;
}

// vicinity batch call (materialised route): kernel 1's fill, the filtration when values are wanted (not with a bad
// descriptor: no target reaches it), kernel 1c's edge list of every target, then kernel 10's export of the chunk into the
// call's arrays at their final offsets
static void run_structure(tlc_graph* g, const Params& p, const ChunkView& c, int64_t n_max, int64_t m_max,
                          const std::vector<SubRange>& subs, bool bad_desc, StageTimer& tm) {
  cudaStream_t st = g->stream;
  const int block = block_for(m_max);
  const tlc_vicinity_batch& o = g->vb.out;
  tm.mark(1);
  launch_vicinity_fill(g->gv, p, c, make_vs(g), g->work_counter.as<int>(), st);
  tm.mark(2);
  if (o.fval && !bad_desc) run_filtration(g, p, c, n_max, block, subs, false);
  tm.mark(5);
  launch_edgelist(p, c, block, 0, st);
  tm.mark(-1);
  launch_vicinity_export(c, o.voff, o.eoff, o.vert, o.ea, o.eb, o.fval, g->vb.status, bad_desc ? 1 : 0, st);
}

static int check_params(const tlc_params* p) {
  if (!p) return fail(TLC_E_INVALID, "params is NULL");
  if (p->resolution < 1 || p->resolution > 16) return fail(TLC_E_INVALID, "resolution must be in 1..16");
  if (p->hop < 0) return fail(TLC_E_INVALID, "hop must be >= 0");
  if (p->mode < TLC_MODE_EDGE || p->mode > TLC_MODE_EDGE_REMOVEINTER) return fail(TLC_E_INVALID, "bad mode");
  if ((p->flags & TLC_F_ASC_ONLY) && (p->flags & TLC_F_EXTENDED))
    return fail(TLC_E_INVALID, "TLC_F_ASC_ONLY excludes TLC_F_EXTENDED (the loops need the Pos/Neg lists)");
  return TLC_OK;
}

static Params to_params(const tlc_params* up) {
  return Params{up->hop, up->mode, up->descriptor, up->resolution, up->flags, up->img_mask};
}

// targets whose image row was really computed (riccidist2dgm.py:354)
static int64_t count_computed(const uint8_t* h_st, int64_t E) {
  int64_t cnt = 0;
  for (int64_t i = 0; i < E; i++) cnt += h_st[i] <= TLC_ST_TRIVIAL;
  return cnt;
}

// the route of a staged call.  The graph-row route (no adjacency in HBM) serves calls that need the ascending sweep only;
// it reads D_S graph-row entries per root where the materialised route reads the 2m induced ones, so it is taken where the
// vicinities are dense in the graph.  use_table: kernel 1t's per-root tables (built here once) filter its targets.
static int choose_route(tlc_graph* g, const Params& p, const int32_t* d_targets, int64_t E, const VicinityScratch& vs,
                        bool direct_ok, bool* direct, bool* use_table) {
  cudaStream_t st = g->stream;
  *direct = direct_ok && (p.flags & TLC_F_DIRECT);
  *use_table = false;
  if (direct_ok && !*direct) {
    // density probe: the full counting pass on a strided sample of the call's targets (measured on B200: one route
    // per call beats mixing; Computers-shaped 2-hop: D_S / 2m = 1.4, PubMed / collab: > 2).  The verdict is kept
    // for the next calls with the same hop and mode and refreshed every 32 calls.
    if (g->probe_hop == p.hop && g->probe_mode == p.mode && g->probe_age < 32) {
      *direct = g->probe_direct;
      g->probe_age++;
    } else {
      double direct_ratio = 2.0;
      if (const char* env = getenv("TLC_DIRECT_RATIO")) direct_ratio = atof(env);
      const int64_t S = std::min<int64_t>(E, std::max<int64_t>(64, E / 64));
      const int64_t stride = E / S;
      DevBuf sample_buf;
      CK(sample_buf.reserve((size_t)S * 8));
      int32_t* d_sample = sample_buf.as<int32_t>();
      CK(cudaMemcpy2DAsync(d_sample, 8, d_targets, (size_t)stride * 8, 8, (size_t)S, cudaMemcpyDeviceToDevice, st));
      launch_vicinity_sizes(g->gv, p, d_sample, S, g->d_n.as<int32_t>(), g->d_m.as<int32_t>(), g->d_ds.as<int32_t>(),
                            g->d_st.as<uint8_t>(), g->d_bytes.as<double>(), vs, g->work_counter.as<int>(), st);
      std::vector<int32_t> sm((size_t)S), sds((size_t)S);
      std::vector<uint8_t> sst((size_t)S);
      CK(cudaMemcpyAsync(sm.data(), g->d_m.p, (size_t)S * 4, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(sds.data(), g->d_ds.p, (size_t)S * 4, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(sst.data(), g->d_st.p, (size_t)S, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      double a = 0, b = 0;
      for (int64_t i = 0; i < S; i++) if (sst[(size_t)i] == TLC_ST_OK) { a += sds[(size_t)i]; b += 2.0 * sm[(size_t)i]; }
      *direct = b > 0 && a <= direct_ratio * b;
      g->probe_hop = p.hop; g->probe_mode = p.mode; g->probe_age = 0; g->probe_direct = *direct;
    }
  }
  // Kernel 1t's proof needs S to be a subset of each root's ball (the graph of the root's table row): true for EDGE
  // (ball(u) & ball(v)) and NODE (ball(u)), not for FORCED, UNION or REMOVEINTER, which must never reach the tables.
  const bool table_mode = p.mode == TLC_MODE_EDGE || p.mode == TLC_MODE_NODE;
  if (*direct && table_mode && !(p.flags & TLC_F_NO_TABLE) && !getenv("TLC_NO_TABLE")) {
    int rc = ensure_sssp_tables(g, p);
    if (rc) return rc;
    if (g->sssp.D) {
      *use_table = true;
      if (!g->sssp_all) {
        // the rows of ALL roots, once per graph (summation rule and hop): a full pass over a dataset touches every node
        // anyway, and a handful of late rows would cost a whole single-CTA shortest-path run in the middle of a step.
        // Every row needs its root's ball for this hop: prepare_call has already reset the ball cache on a hop change.
        cudaEvent_t b0 = nullptr, b1 = nullptr;
        cudaEventCreate(&b0); cudaEventCreate(&b1);
        cudaEventRecord(b0, st);
        launch_ball_cache(g->gv, p, nullptr, 0, vs, st);
        launch_sssp_build(g->gv, p, nullptr, 0, g->sssp, vs.ball_cache, g->gminw.as<float>(), g->sssp_pw.as<double>(),
                          g->sm_count, st);
        cudaEventRecord(b1, st);
        CK(cudaStreamSynchronize(st));
        float ms = 0;
        cudaEventElapsedTime(&ms, b0, b1);
        g->sssp_build_ms = ms;
        cudaEventDestroy(b0); cudaEventDestroy(b1);
        g->sssp_all = true;
      }
    }
  }
  return TLC_OK;
}

// the call's pinned host staging: the counting pass's results, the per-chunk offsets ([E + 2] each) and edge counts
struct HostStage {
  int32_t *n, *m, *ds;
  uint8_t* st;
  double* bytes;
  int64_t *tidx, *voff, *eoff, *aoff;
  int32_t* tm;
};

// the order in which the live targets are packed into chunks, and an arena that holds at least one target's chunk,
// preferably the whole call's.  Wc: bitmap words per target (graph-row route).
static int plan_call(tlc_graph* g, const HostStage& h, int64_t E, bool light, int64_t Wc, const tlc_detail* detail,
                     std::vector<int64_t>& order) {
  order.reserve(E);
  if (detail) {
    for (int64_t i = 0; i < E; i++) order.push_back(i);
  } else {
    // one 64-bit key per live target, then a plain sort: [shared-memory class | size, largest first | row]
    // (a comparator-based stable sort of the index vector cost ~1 ms per 8 k targets: a third of a PubMed-shaped step).
    // Ahead of everything the few vicinities too large for kernel 1b's shared-memory state (heavy-tailed graphs): they
    // get sub-ranges of their own (split_subranges) instead of dragging a whole size group onto the arena path.
    std::vector<uint64_t> keys;
    keys.reserve(E);
    for (int64_t i = 0; i < E; i++) {
      // (the vicinity batch call exports the structure of every vicinity that has vertices, whatever its status)
      if (h.st[i] != TLC_ST_OK && !(g->vb.on && h.n[i] > 0)) continue;
      const uint64_t cls = (uint64_t)smem_class(h.n[i]);
      const uint64_t msz = (uint64_t)std::min<int64_t>(h.m[i], (1 << 28) - 1);
      keys.push_back((cls << 61) | ((((uint64_t)1 << 28) - 1 - msz) << 32) | (uint64_t)i);
    }
    std::sort(keys.begin(), keys.end());
    for (uint64_t k : keys) order.push_back((int64_t)(k & 0xffffffffull));
  }
  int64_t need_one = 0, Nv = 0, Ne = 0, Na = 0;
  for (int64_t i : order) {
    need_one = std::max<int64_t>(need_one, (int64_t)chunk_bytes(1, h.n[i], light ? 0 : h.m[i], light ? 0 : h.ds[i], Wc));
    Nv += h.n[i];
    if (!light) { Ne += h.m[i]; Na += h.ds[i]; }
  }
  const size_t whole = chunk_bytes((int64_t)order.size(), Nv, Ne, Na, Wc);
  if (detail) {  // one chunk
    need_one = (int64_t)whole;
    if (Nv > detail->cap_v || Ne > detail->cap_e || Nv + Ne + E > detail->cap_p)
      return fail(TLC_E_CAPACITY, "detail capacity too small: need v=" + std::to_string(Nv) + " e=" +
                                      std::to_string(Ne) + " p=" + std::to_string(Nv + Ne + E));
  }
  return ensure_arena(g, (size_t)need_one, std::max((size_t)need_one, whole));
}

struct Packed { size_t end; int64_t T, Nv, Ne, Na, n_max, m_max; };  // targets order[pos, end) of one chunk

// greedy pack of the targets from order[pos]: same size class, fits the arena.  Their offsets go to the pinned staging at
// the same positions: the region [pos, end) is one no earlier chunk's upload reads.
static Packed pack_chunk(const tlc_graph* g, const std::vector<int64_t>& order, size_t pos, const HostStage& h, bool light,
                         int64_t Wc, bool detail) {
  const int64_t max_T = 1 << 16;
  Packed k{pos, 0, 0, 0, 0, 0, 0};
  int cls0 = size_class(h.m[order[pos]]);
  size_t& q = k.end;
  while (q < order.size() && k.T < max_T) {
    const int64_t i = order[q];
    if (!detail && size_class(h.m[i]) != cls0) {
      // a new size class starts its own chunk (own CTA width) only if it can fill the GPU about twice;
      // a handful of smaller targets ride along in the current chunk instead of paying a tail of their own
      const int cls1 = size_class(h.m[i]);
      size_t q2 = q;
      while (q2 < order.size() && q2 - q < (size_t)(2 * g->sm_count) && size_class(h.m[order[q2]]) == cls1) q2++;
      if (q2 - q >= (size_t)(2 * g->sm_count)) break;
      cls0 = cls1;
    }
    const int64_t mi = light ? 0 : h.m[i], di = light ? 0 : h.ds[i];  // (graph-row batch call: no edge / adjacency arrays)
    if (chunk_bytes(k.T + 1, k.Nv + h.n[i], k.Ne + mi, k.Na + di, Wc) > g->arena.bytes) break;
    h.tidx[q] = i; h.voff[q] = k.Nv; h.eoff[q] = k.Ne; h.aoff[q] = k.Na; h.tm[q] = h.m[i];
    k.Nv += h.n[i]; k.Ne += mi; k.Na += di;
    k.n_max = std::max<int64_t>(k.n_max, h.n[i]); k.m_max = std::max<int64_t>(k.m_max, h.m[i]);
    k.T++; q++;
  }
  return k;
}

// the sub-ranges of the chunk order[pos, pos + T): the shared-memory classes first (a chunk is sorted by them), then the
// rest in 1, 2 or 4 equal parts, as many as fill the GPU twice each
static std::vector<SubRange> split_subranges(const tlc_graph* g, const std::vector<int64_t>& order, size_t pos, int64_t T,
                                             const int32_t* h_n) {
  std::vector<SubRange> subs;
  const int groups = T >= 4 * 2 * g->sm_count ? 4 : (T >= 2 * 2 * g->sm_count ? 2 : 1);
  int64_t first = 0;
  for (int cls = 0; cls < 2; cls++) {
    int64_t b = first;
    while (b < T && smem_class(h_n[order[pos + b]]) == cls) b++;
    if (b > first) {
      int64_t n0 = INT64_MAX, nm = 0;
      for (int64_t k = first; k < b; k++) { n0 = std::min<int64_t>(n0, h_n[order[pos + k]]); nm = std::max<int64_t>(nm, h_n[order[pos + k]]); }
      subs.push_back(SubRange{(int)first, (int)(b - first), n0, nm});
      first = b;
    }
  }
  const int64_t rest = T - first;
  for (int gi = 0; gi < groups && rest > 0; gi++) {
    const int64_t a = first + rest * gi / groups, b = first + rest * (gi + 1) / groups;
    if (b <= a) continue;
    int64_t n0 = INT64_MAX, nm = 0;
    for (int64_t k = a; k < b; k++) { n0 = std::min<int64_t>(n0, h_n[order[pos + k]]); nm = std::max<int64_t>(nm, h_n[order[pos + k]]); }
    subs.push_back(SubRange{(int)a, (int)(b - a), n0, nm});
  }
  return subs;
}

// every intermediate of the detail call's single chunk, copied back (input order == chunk order)
static int copy_detail(tlc_detail* detail, const ChunkView& c, const Packed& k, const int64_t* voff, const int64_t* eoff,
                       const Params& p) {
  const int64_t T = k.T, Nv = k.Nv, Ne = k.Ne;
#define D2H(dst, src, count, type) \
  if (detail->dst) CK(cudaMemcpy(detail->dst, src, (size_t)(count) * sizeof(type), cudaMemcpyDeviceToHost))
  D2H(n, c.tn, T, int32_t); D2H(m, c.tm, T, int32_t); D2H(lu, c.tlu, T, int32_t); D2H(lv, c.tlv, T, int32_t);
  D2H(npairs, c.tnp, T, int32_t); D2H(npos, c.tnpos, T, int32_t); D2H(nneg, c.tnneg, T, int32_t);
  D2H(vert, c.vert, Nv, int32_t); D2H(fval, c.fval, Nv, double); D2H(neg, c.neg, Nv, int32_t);
  if (!(p.flags & TLC_F_ASC_ONLY)) {
    D2H(elo, c.elo, Ne, int32_t); D2H(ehi, c.ehi, Ne, int32_t); D2H(ew, c.ew, Ne, double);
    D2H(ord_asc, c.ord_asc, Ne, int32_t); D2H(ord_desc, c.ord_desc, Ne, int32_t); D2H(pos, c.pos, Ne, int32_t);
  }
  D2H(pbv, c.pbv, Nv + Ne + T, int32_t); D2H(pdv, c.pdv, Nv + Ne + T, int32_t);
  D2H(pbirth, c.pbirth, Nv + Ne + T, double); D2H(pdeath, c.pdeath, Nv + Ne + T, double);
#undef D2H
  if (detail->pkind) {
    std::vector<uint8_t> k8((size_t)(Nv + Ne + T));
    CK(cudaMemcpy(k8.data(), c.pkind, k8.size(), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < k8.size(); i++) detail->pkind[i] = k8[i];
  }
  for (int64_t t = 0; t <= T; t++) {
    const int64_t vo = t < T ? voff[t] : Nv, eo = t < T ? eoff[t] : Ne;
    if (detail->voff) detail->voff[t] = vo;
    if (detail->eoff) detail->eoff[t] = eo;
    if (detail->poff) detail->poff[t] = vo + eo + t;
  }
  return TLC_OK;
}

static int run_staged(tlc_graph* g, const int32_t* d_targets, int64_t E, const tlc_params* up, double* d_pi,
                      float* d_pi32, uint8_t* d_status, int64_t* cnt_compute, tlc_detail* detail, CallStats& s,
                      size_t ev_base, const int64_t* drow = nullptr);

// diagram call: the pairs of a finished chunk into the staging area.  tidx: the chunk's rows of this (sub-)call, drow:
// their rows in the diagram call (NULL: the same); skip[t] != 0: target t is redone by a later sub-call, not exported.
static int export_chunk(tlc_graph* g, const ChunkView& c, int64_t T, const int64_t* tidx, const int64_t* drow,
                        const std::vector<uint8_t>& skip) {
  DiagCollect& d = g->dg;
  cudaStream_t st = g->stream;
  std::vector<int32_t> tnp((size_t)T);
  std::vector<uint8_t> tst((size_t)T);
  CK(cudaMemcpyAsync(tnp.data(), c.tnp, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(tst.data(), c.tstatus, (size_t)T, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  std::vector<int64_t> h((size_t)T * 2);  // [T] staging offsets | [T] rows of the diagram call
  int64_t sum = 0;
  for (int64_t t = 0; t < T; t++) {
    const bool redone = !skip.empty() && skip[(size_t)t];
    h[(size_t)t] = d.small_total + d.staged_used + sum;
    h[(size_t)(T + t)] = redone ? -1 : (drow ? drow[tidx[t]] : tidx[t]);
    if (!redone) sum += diag_pairs(tst[(size_t)t], tnp[(size_t)t]);
  }
  CK(d.staged.grow(d.staged_used, d.staged_used + sum, st));
  CK(d.chunk.reserve((size_t)T * 16));
  CK(cudaMemcpyAsync(d.chunk.p, h.data(), (size_t)T * 16, cudaMemcpyHostToDevice, st));
  launch_export_pairs(c, d.chunk.as<int64_t>(), d.chunk.as<int64_t>() + T, d.staged.view(), d.small_total,
                      d.np.as<int32_t>(), d.soff.as<int64_t>(), g->sm_count, st);
  CK(cudaStreamSynchronize(st));
  d.staged_used += sum;
  return TLC_OK;
}

// the targets kernel 3v handed back on a graph-row batch call, as their own call on the materialised route; rows scattered
// back.  The targets are counted already: of the redo's statistics only its chunks and stage times are added to s.
static int redo_handed_back(tlc_graph* g, const int32_t* d_targets, int64_t E, const std::vector<int64_t>& redo,
                            const tlc_params* up, double* d_pi, float* d_pi32, uint8_t* d_status, size_t ev_base,
                            CallStats& s, const int64_t* drow) {
  cudaStream_t st = g->stream;
  const int r2 = up->resolution * up->resolution;
  const int64_t k = (int64_t)redo.size();
  // (all copies on the call's stream -- a non-blocking stream is not ordered with the legacy stream a plain cudaMemcpy uses --
  // and synchronised before the host vectors are touched or go away; the device buffers free themselves on every exit path)
  std::vector<int32_t> h_all((size_t)E * 2), h_sub((size_t)k * 2);
  CK(cudaMemcpyAsync(h_all.data(), d_targets, (size_t)E * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int64_t i = 0; i < k; i++) { h_sub[2 * i] = h_all[2 * redo[i]]; h_sub[2 * i + 1] = h_all[2 * redo[i] + 1]; }
  DevBuf b_sub, b_idx, b_pi, b_pi32, b_st;
  CK(b_sub.reserve((size_t)k * 8));
  CK(b_idx.reserve((size_t)k * 8));
  CK(b_pi.reserve((size_t)k * r2 * 8));
  CK(b_pi32.reserve((size_t)k * r2 * 4));
  CK(b_st.reserve((size_t)k));
  CK(cudaMemcpyAsync(b_sub.p, h_sub.data(), (size_t)k * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(b_idx.p, redo.data(), (size_t)k * 8, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  tlc_params up2 = *up;
  up2.flags = (up2.flags | TLC_F_NO_DIRECT) & ~TLC_F_DIRECT;
  std::vector<int64_t> rows((size_t)k);  // diagram call: the redone targets' rows in it
  for (int64_t i = 0; i < k; i++) rows[(size_t)i] = drow ? drow[redo[i]] : redo[i];
  CallStats sub;
  const int rc = run_staged(g, b_sub.as<int32_t>(), k, &up2, b_pi.as<double>(), b_pi32.as<float>(), b_st.as<uint8_t>(),
                            nullptr, nullptr, sub, ev_base, rows.data());
  if (rc) return rc;
  launch_scatter_rows(b_pi.as<double>(), d_pi32 ? b_pi32.as<float>() : nullptr, d_status ? b_st.as<uint8_t>() : nullptr,
                      b_idx.as<int64_t>(), k, r2, d_pi, d_pi32, d_status, g->sm_count, st);
  cudaStreamSynchronize(st);
  s.chunks += sub.chunks;
  for (int i = 0; i < 10; i++) s.stage_ms[i] += sub.stage_ms[i];
  return TLC_OK;
}

// the STAGED pipeline over device-resident targets; the call's statistics go to s.  detail != NULL: single chunk in input
// order, every intermediate copied back to host.  ev_base: the first of the graph's stage-timing events this call may use
// (a nested call's live behind its caller's).
static int run_staged(tlc_graph* g, const int32_t* d_targets, int64_t E, const tlc_params* up, double* d_pi,
                      float* d_pi32, uint8_t* d_status, int64_t* cnt_compute, tlc_detail* detail, CallStats& s,
                      size_t ev_base, const int64_t* drow) {
  s = CallStats();
  if (E < 0 || E >= ((int64_t)1 << 32)) return fail(TLC_E_INVALID, "E must be in [0, 2^32)");
  CK(cudaSetDevice(g->device));
  const Params p = to_params(up);
  const int r2 = p.resolution * p.resolution;
  cudaStream_t st = g->stream;
  int* fb_counters = g->work_counter.as<int>() + 4;  // handed back, general, rowcheck, blocks | kernel 1t two-root targets
  CK(cudaMemsetAsync(fb_counters, 0, 5 * sizeof(int), st));
  if (cnt_compute) *cnt_compute = 0;
  if (E == 0) return TLC_OK;
  const bool bad_desc = p.descriptor < 0 || p.descriptor > 2;
  int rc;
  if ((rc = prepare_call(g, p, E))) return rc;
  StageTimer tm(st, &g->ev_pool, ev_base);
  cudaEvent_t ev_total0 = nullptr, ev_total1 = nullptr;
  if (tm.on) { ev_total0 = tm.take(); ev_total1 = tm.take(); tm.first = tm.used; cudaEventRecord(ev_total0, st); }
  int32_t *d_n = g->d_n.as<int32_t>(), *d_m = g->d_m.as<int32_t>(), *d_ds = g->d_ds.as<int32_t>();
  uint8_t* d_st = g->d_st.as<uint8_t>();
  double* d_bytes = g->d_bytes.as<double>();

  // ---- route, one per call ----
  const int64_t Wd = ((int64_t)g->gv.N + 31) / 32;
  // (pair output -- detail or diagram call -- wants PD_down and [max,min] unless TLC_F_ASC_ONLY)
  const bool want_pairs = detail != nullptr || g->dg.on;
  const bool want_desc_call = ((p.flags & TLC_F_EXTENDED) != 0 || want_pairs) && !(p.flags & TLC_F_ASC_ONLY);
  const bool direct_ok = g->ball_cache.p != nullptr && g->gminw.p != nullptr && !want_desc_call && !bad_desc && !g->vb.on &&
                         p.mode <= TLC_MODE_NODE && !(p.flags & TLC_F_FILT_ANY_STRUCT) &&
                         !(p.flags & (TLC_F_NO_DIRECT | TLC_F_EDGE_SORTED)) && (size_t)Wd * 8 <= 64 * 1024;
  VicinityScratch vs = make_vs(g);
  tm.mark(0);
  launch_ball_cache(g->gv, p, d_targets, E, vs, st);
  bool direct = false, use_table = false;
  if ((rc = choose_route(g, p, d_targets, E, vs, direct_ok, &direct, &use_table))) return rc;
  if (detail) direct = direct_ok && (p.flags & TLC_F_DIRECT);  // (the probe's verdict serves the batch calls only)
  // the batch call on the graph-row route skips counting the induced edges (kernel 1b counts them as it reads the rows)
  const bool light = direct && detail == nullptr;
  const int64_t Wc = direct ? Wd : 0;

  // ---- kernel 1, counting pass ----
  if (light) launch_vicinity_light(g->gv, p, d_targets, E, d_n, d_m, d_ds, d_st, d_bytes, vs, g->sm_count, st);
  else launch_vicinity_sizes(g->gv, p, d_targets, E, d_n, d_m, d_ds, d_st, d_bytes, vs, g->work_counter.as<int>(), st);
  tm.mark(-1);
  const size_t pin_need = align_up((size_t)E * 8) + (size_t)E * 9 + ALIGN;
  const size_t pin_need2 = align_up((size_t)E * 4);  // h.ds
  CK(g->h_pin.reserve(align_up(pin_need) + pin_need2 + (size_t)(E + 2) * 8 * 4 + (size_t)(E + 2) * 4 + ALIGN));
  char* pin = g->h_pin.as<char>();
  HostStage h;
  h.n = reinterpret_cast<int32_t*>(pin);
  h.m = h.n + E;
  h.bytes = reinterpret_cast<double*>(pin + align_up((size_t)E * 8));
  h.st = reinterpret_cast<uint8_t*>(h.bytes + E);
  h.ds = reinterpret_cast<int32_t*>(pin + align_up(pin_need));
  h.tidx = reinterpret_cast<int64_t*>(pin + align_up(pin_need) + pin_need2);
  h.voff = h.tidx + (E + 2);
  h.eoff = h.voff + (E + 2);
  h.aoff = h.eoff + (E + 2);
  h.tm = reinterpret_cast<int32_t*>(h.aoff + (E + 2));
  CK(cudaMemcpyAsync(h.n, d_n, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h.m, d_m, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h.ds, d_ds, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h.st, d_st, (size_t)E, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h.bytes, d_bytes, (size_t)E * 8, cudaMemcpyDeviceToHost, st));
  // rows of targets that never reach the image kernel stay zero (riccidist2dgm.py:363)
  if (d_pi) CK(cudaMemsetAsync(d_pi, 0, (size_t)E * r2 * sizeof(double), st));
  if (d_pi32) CK(cudaMemsetAsync(d_pi32, 0, (size_t)E * r2 * sizeof(float), st));
  CK(cudaStreamSynchronize(st));
  if (bad_desc) {  // KeyError in perturb_filter_function for every target that got that far (accelerated_PD.py:13)
    for (int64_t i = 0; i < E; i++) if (h.st[i] == TLC_ST_OK) h.st[i] = TLC_ST_BAD_DESCRIPTOR;
    if (d_status) CK(cudaMemcpyAsync(d_status, h.st, (size_t)E, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    if (!g->vb.on) return TLC_OK;  // (the vicinity batch call still exports the structure)
  } else if (d_status) {
    CK(cudaMemcpyAsync(d_status, d_st, (size_t)E, cudaMemcpyDeviceToDevice, st));
  }
  if (g->vb.on) {  // the final offsets (kernel 7's scan of n and m) and totals; too small a capacity ends the call here
    BatchCollect& b = g->vb;
    launch_scan_counts(d_n, E, b.out.voff, st);
    launch_scan_counts(d_m, E, b.out.eoff, st);
    b.total_v = 0; b.total_e = 0;
    for (int64_t i = 0; i < E; i++) { b.total_v += h.n[i]; b.total_e += h.m[i]; }
    CK(cudaStreamSynchronize(st));
    if (b.total_v > b.out.cap_v || b.total_e > b.out.cap_e)
      return fail(TLC_E_CAPACITY, "the vicinities hold " + std::to_string(b.total_v) + " vertices and " +
                                      std::to_string(b.total_e) + " edges, cap_v is " + std::to_string(b.out.cap_v) +
                                      " and cap_e is " + std::to_string(b.out.cap_e));
    if ((b.out.ea || b.out.eb) && b.total_v >= ((int64_t)1 << 31))
      return fail(TLC_E_INVALID, "the vicinities hold " + std::to_string(b.total_v) + " vertices: int32 batch ids need < 2^31");
  }
  for (int64_t i = 0; i < E; i++)
    if (h.st[i] == TLC_ST_OK) { s.bytes += h.bytes[i]; s.live++; s.sum_n += h.n[i]; if (!light) s.sum_m += h.m[i]; }

  std::vector<int64_t> order;
  if ((rc = plan_call(g, h, E, light, Wc, detail, order))) return rc;
  std::vector<int64_t> redo;  // graph-row batch call: rows of the targets kernel 3v handed back
  for (size_t pos = 0; pos < order.size();) {
    const Packed k = pack_chunk(g, order, pos, h, light, Wc, detail != nullptr);
    if (k.T == 0) return fail(TLC_E_NOMEM, "a vicinity does not fit the arena");
    ChunkView c = carve(g->arena.as<char>(), k.T, k.Nv, k.Ne, k.Na, d_targets, Wc);
    c.fb_counter = fb_counters;
    c.gcol = g->gv.col;
    c.gkappa = g->gv.kappa;
    // offsets: [pos, pos+T) plus the terminating total.  voff/eoff need T+1 entries; the terminator is
    // copied from k (synchronised below) so that the next chunk's slot `end` is not clobbered.
    CK(cudaMemcpyAsync((void*)c.tidx, h.tidx + pos, (size_t)k.T * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync((void*)c.voff, h.voff + pos, (size_t)k.T * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync((void*)c.eoff, h.eoff + pos, (size_t)k.T * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync((void*)c.aoff, h.aoff + pos, (size_t)k.T * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync((void*)(c.voff + k.T), &k.Nv, 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync((void*)(c.eoff + k.T), &k.Ne, 8, cudaMemcpyHostToDevice, st));
    const std::vector<SubRange> subs = split_subranges(g, order, pos, k.T, h.n);
    std::vector<uint8_t> fbv;  // graph-row batch call: targets kernel 3v handed back (redone below)
    if (g->vb.on) {
      run_structure(g, p, c, k.n_max, k.m_max, subs, bad_desc, tm);
    } else if (direct) {
      c.count_m = light ? 1 : 0;
      // tm: counted by kernel 1b (batch call) or known from the full counting pass (detail call)
      if (!light) CK(cudaMemcpyAsync((void*)c.tm, h.tm + pos, (size_t)k.T * 4, cudaMemcpyHostToDevice, st));
      int fb0 = 0, fb1[5] = {0, 0, 0, 0, 0};
      CK(cudaMemcpyAsync(&fb0, fb_counters, sizeof(int), cudaMemcpyDeviceToHost, st));
      s.table += run_stages(g, p, c, k.n_max, k.m_max, subs, d_pi, d_pi32, d_status, want_pairs, tm, use_table);
      CK(cudaMemcpyAsync(fb1, fb_counters, 5 * sizeof(int), cudaMemcpyDeviceToHost, st));
      if (light) CK(cudaMemcpyAsync(h.tm + pos, c.tm, (size_t)k.T * 4, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      s.direct += k.T;
      s.two_root = fb1[4];  // (a running count over the call's chunks; a redo of handed-back targets below resets the counter)
      if (light) {  // the exact edge counts: totals and the 16 m term of the compulsory bytes (SURVEY.md 8d)
        for (int64_t t = 0; t < k.T; t++) { s.sum_m += h.tm[pos + t]; s.bytes += 16.0 * (double)h.tm[pos + t]; }
      }
      if (fb1[0] != fb0) {
        // kernel 3v handed targets back: their edge-sorted sweep needs the adjacency
        if (light) {  // no adjacency space was reserved: those targets are redone on the materialised route below
          fbv.resize((size_t)k.T);
          CK(cudaMemcpyAsync(fbv.data(), c.tfb, (size_t)k.T, cudaMemcpyDeviceToHost, st));
          CK(cudaStreamSynchronize(st));
          for (const SubRange& r : subs)
            for (int64_t t = r.t0; t < r.t0 + r.cnt; t++) {
              if (!fbv[(size_t)t]) continue;
              redo.push_back(h.tidx[pos + t]);
              s.direct--;
              if (takes_table(g, use_table, r)) s.table--;
            }
        } else {
          // the chunk is redone on the materialised route (its space is reserved), image rows and statuses are rewritten
          c.dbm = nullptr;
          c.W = 0;
          s.direct -= k.T;
          run_stages(g, p, c, k.n_max, k.m_max, subs, d_pi, d_pi32, d_status, want_pairs, tm, use_table);
        }
      }
    } else {
      run_stages(g, p, c, k.n_max, k.m_max, subs, d_pi, d_pi32, d_status, want_pairs, tm, use_table);
    }
    s.chunks++;
    CK(cudaStreamSynchronize(st));
    if (g->dg.on && (rc = export_chunk(g, c, k.T, h.tidx + pos, drow, fbv))) return rc;
    if (detail) {
      g->detail_chunk = c;
      if ((rc = copy_detail(detail, c, k, h.voff + pos, h.eoff + pos, p))) return rc;
    }
    pos = k.end;
  }
  if (!redo.empty()) {
    tm.collect(s.stage_ms);
    if ((rc = redo_handed_back(g, d_targets, E, redo, up, d_pi, d_pi32, d_status, tm.used, s, drow))) return rc;
  }
  if (tm.on) {
    cudaEventRecord(ev_total1, st);
    cudaStreamSynchronize(st);
    float ms = 0;
    cudaEventElapsedTime(&ms, ev_total0, ev_total1);
    s.stage_ms[9] = ms;
    tm.collect(s.stage_ms);
  }
  if ((cnt_compute || (detail && detail->status)) && d_status) {
    CK(cudaMemcpyAsync(h.st, d_status, (size_t)E, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (cnt_compute) *cnt_compute = count_computed(h.st, E);
    if (detail && detail->status) memcpy(detail->status, h.st, (size_t)E);
  }
  {
    int fb[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(fb, fb_counters, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    s.handed_back = fb[0]; s.general = fb[1]; s.rowcheck = fb[2]; s.blocks = fb[3];
  }
  CK(cudaGetLastError());
  return TLC_OK;
}

static int ensure_small_buffers(tlc_graph* g, int64_t E) {
  if (!g->sm_dev.p) {
    CK(g->sm_dev.reserve(256));
    CK(g->sm_host.reserve(256));
    CK(cudaEventCreateWithFlags(&g->ev_small_a, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&g->ev_small_bc, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&g->ev_small_c, cudaEventDisableTiming));
    if (!getenv("TLC_NO_SIDE_STREAMS")) {
      CK(cudaStreamCreateWithFlags(&g->small_stream, cudaStreamNonBlocking));
      CK(cudaStreamCreateWithFlags(&g->small_stream2, cudaStreamNonBlocking));
    }
  }
  if (E <= g->sm_cap) return TLC_OK;
  const size_t cap = (size_t)(E + E / 8 + 1024);
  for (DevBuf* b : {&g->sm_list_b, &g->sm_list_c, &g->sm_list_big, &g->sm_list_b2}) CK(b->reserve(cap * 4));
  g->sm_cap = (int64_t)cap;
  return TLC_OK;
}

static int ensure_small_sub(tlc_graph* g, int64_t k, int r2) {
  if (k <= g->sm_sub_cap) return TLC_OK;
  const size_t cap = (size_t)(k + k / 4 + 256);
  CK(g->sm_sub.reserve(cap * 8));
  CK(g->sm_idx.reserve(cap * 8));
  CK(g->sm_pi.reserve(cap * r2 * 8));
  CK(g->sm_pi32.reserve(cap * r2 * 4));
  CK(g->sm_st.reserve(cap));
  g->sm_sub_cap = (int64_t)cap;
  return TLC_OK;
}

static constexpr size_t SM_STATS_OFF = 32;  // SmallStats behind the eight list counters in sm_dev / sm_host

// which calls kernel S (k0_small.cu) can take: the batch call with a Ricci-distance filtration and a 5 x 5 image on a
// graph whose ball cache exists; the route-forcing diagnostic flags keep their meaning (they name staged kernels)
static bool small_applicable(const tlc_graph* g, const tlc_params* up, int64_t E, const tlc_detail* detail) {
  if (detail || E <= 0 || E >= ((int64_t)1 << 31)) return false;
  if (up->resolution != 5 || up->descriptor < 0 || up->descriptor > 2) return false;
  if (up->flags & (TLC_F_FILT_ANY_STRUCT | TLC_F_EDGE_SORTED | TLC_F_DIRECT | TLC_F_NO_DIRECT | TLC_F_NO_SMALL |
                   (g->dg.on ? 0u : TLC_F_ASC_ONLY))) return false;  // (the diagram call: kernel S skips the descending sweep)
  if (getenv("TLC_NO_SMALL")) return false;
  return true;
}

// the staged pipeline over a device-side list of rows, results scattered back into the caller's tables; its statistics
// are added to s
static int run_staged_list(tlc_graph* g, const int32_t* d_targets, const int32_t* d_list, int64_t k, const tlc_params* up,
                           double* d_pi, float* d_pi32, uint8_t* d_status, size_t ev_base, CallStats& s) {
  const int r2 = up->resolution * up->resolution;
  cudaStream_t st = g->stream;
  int rc;
  if ((rc = ensure_small_sub(g, k, r2))) return rc;
  int32_t* sub = g->sm_sub.as<int32_t>();
  int64_t* idx = g->sm_idx.as<int64_t>();
  double* pi = g->sm_pi.as<double>();
  float* pi32 = g->sm_pi32.as<float>();
  uint8_t* sst = g->sm_st.as<uint8_t>();
  launch_gather_targets(d_targets, d_list, k, sub, idx, st);
  std::vector<int64_t> rows;  // diagram call: the sub-list's rows in it
  if (g->dg.on) {
    rows.resize((size_t)k);
    CK(cudaMemcpyAsync(rows.data(), idx, (size_t)k * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  tlc_params up2 = *up;
  up2.flags |= TLC_F_NO_SMALL;
  CallStats part;
  if ((rc = run_staged(g, sub, k, &up2, pi, pi32, sst, nullptr, nullptr, part, ev_base, g->dg.on ? rows.data() : nullptr)))
    return rc;
  launch_scatter_rows(pi, d_pi32 ? pi32 : nullptr, d_status ? sst : nullptr, idx, k, r2, d_pi, d_pi32, d_status, g->sm_count, st);
  CK(cudaStreamSynchronize(st));
  s += part;
  return TLC_OK;
}

// diagram call: kernel S's staging area.  The counting pass bounds the pairs of every row kernel S can finish (<= 1024
// vertices, <= 4096 edges) by n + m + 2 (ascending sweep only: n + 2), the other rows by 0; the row's segment starts at
// the exclusive prefix of those bounds (dg.soff, which the staged export overwrites for the rows it takes)
static int small_diagram_area(tlc_graph* g, const Params& p, const int32_t* d_targets, int64_t E, const VicinityScratch& vs,
                              SmallDiag* out) {
  DiagCollect& d = g->dg;
  cudaStream_t st = g->stream;
  launch_vicinity_sizes(g->gv, p, d_targets, E, g->d_n.as<int32_t>(), g->d_m.as<int32_t>(), g->d_ds.as<int32_t>(),
                        g->d_st.as<uint8_t>(), g->d_bytes.as<double>(), vs, g->work_counter.as<int>(), st);
  std::vector<int32_t> n((size_t)E), m((size_t)E);
  CK(cudaMemcpyAsync(n.data(), g->d_n.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(m.data(), g->d_m.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const bool asc = (p.flags & TLC_F_ASC_ONLY) != 0;
  std::vector<int64_t> off((size_t)E);
  int64_t total = 0;
  for (int64_t i = 0; i < E; i++) {
    off[(size_t)i] = total;
    if (n[(size_t)i] <= 1024 && m[(size_t)i] <= 4096) total += n[(size_t)i] + (asc ? 0 : m[(size_t)i]) + 2;
  }
  CK(d.small.grow(0, total, st));
  CK(cudaMemcpyAsync(d.soff.p, off.data(), (size_t)E * 8, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  d.small_total = total;
  const DiagArea a = d.small.view();
  *out = SmallDiag{d.soff.as<int64_t>(), d.np.as<int32_t>(), a.kind, a.bv, a.dv, a.birth, a.death};
  out->graph_ids = 1;
  out->want_desc = asc ? 0 : 1;
  return TLC_OK;
}

// kernel S over the whole call, the staged pipeline over the rows it hands on.  Class A (a warp per target) sees every
// target and sorts the rest into "classes B / C" and "more than 1024 vertices: staged"; classes B and C then run on a
// stream of their own WHILE the staged pipeline takes the big targets (whose single-lane sweeps are the critical path of
// extended calls); what class C cannot take either (<= 1024 vertices but more than 4096 edges) follows at the end.
static int run_small(tlc_graph* g, const int32_t* d_targets, int64_t E, const tlc_params* up, double* d_pi, float* d_pi32,
                     uint8_t* d_status, int64_t* cnt_compute, CallStats& s, bool* fell_through) {
  *fell_through = false;
  CK(cudaSetDevice(g->device));
  const Params p = to_params(up);
  cudaStream_t st = g->stream;
  int rc;
  if ((rc = prepare_call(g, p, E))) return rc;
  if (!g->ball_cache.p) { *fell_through = true; return TLC_OK; }
  if ((rc = ensure_small_buffers(g, E))) return rc;
  if (g->small_hop != p.hop || g->small_mode != p.mode) { g->small_hop = p.hop; g->small_mode = p.mode; g->small_skip = 0; }
  if (g->small_skip > 0) { g->small_skip--; *fell_through = true; return TLC_OK; }
  StageTimer tm(st, &g->ev_pool, 0);
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evb0 = nullptr, ev1b = nullptr, evc0 = nullptr, ev2 = nullptr;
  if (tm.on) { ev0 = tm.take(); ev1 = tm.take(); evb0 = tm.take(); ev1b = tm.take(); evc0 = tm.take(); ev2 = tm.take(); }
  VicinityScratch vs = make_vs(g);
  int* counters = g->sm_dev.as<int>();
  SmallStats* d_stats = reinterpret_cast<SmallStats*>(g->sm_dev.as<char>() + SM_STATS_OFF);
  const int* h_counters = g->sm_host.as<int>();
  int32_t *list_b = g->sm_list_b.as<int32_t>(), *list_c = g->sm_list_c.as<int32_t>();
  int32_t *list_big = g->sm_list_big.as<int32_t>(), *list_b2 = g->sm_list_b2.as<int32_t>();
  launch_ball_cache(g->gv, p, d_targets, E, vs, st);
  SmallDiag dgs{};
  const SmallDiag* diag = nullptr;
  if (g->dg.on && (rc = small_diagram_area(g, p, d_targets, E, vs, &dgs))) return rc;
  if (g->dg.on) diag = &dgs;
  if (ev0) cudaEventRecord(ev0, st);
  launch_small(g->gv, p, d_targets, E, vs, d_pi, d_pi32, d_status, list_b, list_c, list_big, counters,
               nullptr, nullptr, diag, d_stats, g->sm_count, 1, st);
  if (ev1) cudaEventRecord(ev1, st);
  // the rows class A deferred, routed by their exact sizes: class B, class C and the staged pipeline then run side by side
  launch_small(g->gv, p, d_targets, E, vs, d_pi, d_pi32, d_status, list_b, list_c, list_big, counters,
               nullptr, nullptr, diag, d_stats, g->sm_count, 4, st, list_b2);
  CK(cudaEventRecord(g->ev_small_a, st));
  CK(cudaMemcpyAsync(g->sm_host.p, g->sm_dev.p, 32, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const int nB = h_counters[4], nCc = h_counters[1], nBig = h_counters[3];
  if (nBig == E) {  // nothing for kernel S: the staged pipeline takes the whole call, and the next calls do not try again
    g->small_skip = 32;
    *fell_through = true;
    return TLC_OK;
  }
  cudaStream_t sb = g->small_stream ? g->small_stream : st;
  cudaStream_t sc = g->small_stream2 ? g->small_stream2 : st;
  if (nB > 0) {
    if (sb != st) CK(cudaStreamWaitEvent(sb, g->ev_small_a, 0));
    if (evb0) cudaEventRecord(evb0, sb);
    launch_small(g->gv, p, d_targets, E, vs, d_pi, d_pi32, d_status, list_b, list_c, list_big, counters,
                 nullptr, nullptr, diag, d_stats, g->sm_count, 8, sb, list_b2);
    if (ev1b) cudaEventRecord(ev1b, sb);
    if (sb != st) CK(cudaEventRecord(g->ev_small_bc, sb));
  }
  if (nCc > 0) {
    if (sc != st) CK(cudaStreamWaitEvent(sc, g->ev_small_a, 0));
    if (evc0) cudaEventRecord(evc0, sc);
    launch_small(g->gv, p, d_targets, E, vs, d_pi, d_pi32, d_status, list_b, list_c, list_big, counters,
                 nullptr, nullptr, diag, d_stats, g->sm_count, 16, sc, list_b2);
    if (ev2) cudaEventRecord(ev2, sc);
    if (sc != st) CK(cudaEventRecord(g->ev_small_c, sc));
  }
  if (nBig > 0 && (rc = run_staged_list(g, d_targets, list_big, nBig, up, d_pi, d_pi32, d_status, tm.used, s))) return rc;
  if (nB > 0 && sb != st) CK(cudaStreamWaitEvent(st, g->ev_small_bc, 0));
  if (nCc > 0 && sc != st) CK(cudaStreamWaitEvent(st, g->ev_small_c, 0));
  CK(cudaMemcpyAsync(g->sm_host.p, g->sm_dev.p, SM_STATS_OFF + sizeof(SmallStats), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const int nC = h_counters[2];  // rows classes B / C could not take after all (listed in sm_list_b)
  const SmallStats hs = *reinterpret_cast<const SmallStats*>(g->sm_host.as<char>() + SM_STATS_OFF);
  float msA = 0, msB = 0, msC = 0;
  if (tm.on) {
    cudaEventElapsedTime(&msA, ev0, ev1);
    if (nB > 0) cudaEventElapsedTime(&msB, evb0, ev1b);
    if (nCc > 0) cudaEventElapsedTime(&msC, evc0, ev2);
  }
  if (nC > 0 && (rc = run_staged_list(g, d_targets, list_b, nC, up, d_pi, d_pi32, d_status, tm.used, s))) return rc;
  // a call whose vicinities are mostly too large: do not try again for a while (the size check alone costs a pass over
  // two ball bitmaps per target)
  if (((int64_t)nC + nBig) * 4 > E * 3) g->small_skip = 32;
  s.stage_ms[9] += msA + msB + msC;
  s.small_ms[0] = msA; s.small_ms[1] = msB; s.small_ms[2] = msC;
  s.small_rows[0] = (int64_t)hs.handled[0]; s.small_rows[1] = (int64_t)hs.handled[1]; s.small_rows[2] = (int64_t)hs.handled[2];
  s.small_rows[3] = (int64_t)nC + nBig;
  s.live += (int64_t)hs.live; s.sum_n += (int64_t)hs.sum_n; s.sum_m += (int64_t)hs.sum_m;
  s.bytes += hs.bytes;
  if (cnt_compute) {
    *cnt_compute = 0;
    if (d_status) {
      CK(g->h_pin.reserve((size_t)E + ALIGN));
      uint8_t* h_st = g->h_pin.as<uint8_t>();
      CK(cudaMemcpyAsync(h_st, d_status, (size_t)E, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      *cnt_compute = count_computed(h_st, E);
    }
  }
  CK(cudaGetLastError());
  return TLC_OK;
}

// the whole path over device-resident targets: kernel S where it applies, the staged pipeline for everything else;
// the call's statistics are published in g->last
static int run_pipeline(tlc_graph* g, const int32_t* d_targets, int64_t E, const tlc_params* up, double* d_pi,
                        float* d_pi32, uint8_t* d_status, int64_t* cnt_compute, tlc_detail* detail) {
  int rc = check_params(up);
  if (rc) return rc;
  CallStats s;
  bool fell = true;
  if (small_applicable(g, up, E, detail)) rc = run_small(g, d_targets, E, up, d_pi, d_pi32, d_status, cnt_compute, s, &fell);
  if (rc == TLC_OK && fell) rc = run_staged(g, d_targets, E, up, d_pi, d_pi32, d_status, cnt_compute, detail, s, 0);
  g->last = s;
  return rc;
}

// =================================================================================================
// C-ABI
// =================================================================================================
static int graph_upload(tlc_graph* g, int32_t N, int64_t nnz, const int32_t* rowptr, const int32_t* col, const double* kappa);

// The kernels index bitmaps / ball rows by col[] and bisect the rows: a malformed CSR would mean out-of-bounds device
// accesses, so the whole contract is checked on the host before any CUDA call (O(nnz log deg)):
//   rowptr[0] = 0, rowptr[N] = nnz, rowptr monotone; col in [0, N), strictly ascending inside a row (no duplicates), no
//   self-loops; every (x, y) has its mirror (y, x).  With curvatures (kappa != NULL): the mirror has the same curvature
//   (graph2pi.__init__ sets ricci_curv[(a,b)] = ricci_curv[(b,a)], riccidist2dgm.py:222-225), and the weight kappa + 1
//   is finite and > 0 (networkx's Dijkstra precondition; kernel 1b orders distances by their bit patterns)
static int check_csr(int32_t N, int64_t nnz, const int32_t* rowptr, const int32_t* col, const double* kappa) {
  if (rowptr[0] != 0 || rowptr[N] != nnz) return fail(TLC_E_INVALID, "rowptr[0] != 0 or rowptr[N] != nnz");
  for (int32_t x = 0; x < N; x++)
    if (rowptr[x + 1] < rowptr[x]) return fail(TLC_E_INVALID, "rowptr is not monotone at node " + std::to_string(x));
  for (int32_t x = 0; x < N; x++) {  // pass 1: every row well formed on its own (pass 2 bisects the rows)
    for (int64_t e = rowptr[x]; e < rowptr[x + 1]; e++) {
      const int32_t y = col[e];
      if (y < 0 || y >= N) return fail(TLC_E_INVALID, "col out of range in row " + std::to_string(x));
      if (y == x) return fail(TLC_E_INVALID, "self-loop at node " + std::to_string(x));
      if (e > rowptr[x] && col[e - 1] >= y) return fail(TLC_E_INVALID, "row " + std::to_string(x) + " is not strictly ascending");
      const double w = kappa ? kappa[e] + 1.0 : 1.0;
      if (!(w > 0.0) || !std::isfinite(w))
        return fail(TLC_E_INVALID, "kappa + 1 must be finite and > 0 (edge " + std::to_string(x) + "-" + std::to_string(y) + ")");
    }
  }
  for (int32_t x = 0; x < N; x++) {  // pass 2: symmetry
    for (int64_t e = rowptr[x]; e < rowptr[x + 1]; e++) {
      const int32_t y = col[e];
      const int32_t* lo = col + rowptr[y];
      const int32_t* hi = col + rowptr[y + 1];
      const int32_t* it = std::lower_bound(lo, hi, x);
      if (it == hi || *it != x) return fail(TLC_E_INVALID, "graph is not symmetric: (" + std::to_string(x) + "," + std::to_string(y) + ") has no mirror entry");
      if (kappa && kappa[it - col] != kappa[e]) return fail(TLC_E_INVALID, "curvature of (" + std::to_string(x) + "," + std::to_string(y) + ") differs from its mirror entry");
    }
  }
  return TLC_OK;
}

static int select_device(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(TLC_E_NODEVICE, "no CUDA device");
  if (device < 0 || device >= ndev) return fail(TLC_E_INVALID, "device index out of range");
  CK(cudaSetDevice(device));
  return TLC_OK;
}

extern "C" {

const char* tlc_last_error(void) { return g_err.c_str(); }
const char* tlc_version(void) { return "tlc_b200 0.1 (sm_100a)"; }
int64_t tlc_launch_count(void) { return launch_count(); }

int tlc_graph_create(int32_t N, int64_t nnz, const int32_t* rowptr, const int32_t* col, const double* kappa, int device,
                     uint64_t arena_bytes, tlc_graph** out) {
  if (!out || !rowptr || (nnz > 0 && (!col || !kappa)) || N <= 0 || nnz < 0) return fail(TLC_E_INVALID, "bad graph arguments");
  int rc = check_csr(N, nnz, rowptr, col, kappa);
  if (rc || (rc = select_device(device))) return rc;
  tlc_graph* g = new tlc_graph();
  g->device = device;
  g->arena_req = (size_t)arena_bytes;
  rc = graph_upload(g, N, nnz, rowptr, col, kappa);
  if (rc != TLC_OK) { const std::string keep = g_err; tlc_graph_destroy(g); g_err = keep; return rc; }  // nothing leaks on a failed create
  *out = g;
  return TLC_OK;
}

}  // extern "C"

// device side of tlc_graph_create: *g owns every allocation as soon as it exists, so the caller can free a partially
// built graph with tlc_graph_destroy
static int graph_upload(tlc_graph* g, int32_t N, int64_t nnz, const int32_t* rowptr, const int32_t* col, const double* kappa) {
  const int device = g->device;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  g->sm_count = prop.multiProcessorCount;
  CK(cudaStreamCreateWithFlags(&g->own_stream, cudaStreamNonBlocking));
  g->stream = g->own_stream;
  if (!getenv("TLC_NO_SIDE_STREAMS")) {
    CK(cudaEventCreateWithFlags(&g->ev_fork, cudaEventDisableTiming));
    for (int i = 0; i < 3; i++) {
      CK(cudaStreamCreateWithFlags(&g->side[i], cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&g->ev_join[i], cudaEventDisableTiming));
    }
  }
  CK(g->rowptr.reserve((size_t)(N + 1) * 4));
  CK(g->col.reserve(std::max<size_t>((size_t)nnz * 4, 16)));
  CK(g->kappa.reserve(std::max<size_t>((size_t)nnz * 8, 16)));
  g->gv = GraphView{N, nnz, g->rowptr.as<int32_t>(), g->col.as<int32_t>(), g->kappa.as<double>(), nullptr};
  CK(cudaMemcpy((void*)g->gv.rowptr, rowptr, (size_t)(N + 1) * 4, cudaMemcpyHostToDevice));
  if (nnz) {
    CK(cudaMemcpy((void*)g->gv.col, col, (size_t)nnz * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy((void*)g->gv.kappa, kappa, (size_t)nnz * 8, cudaMemcpyHostToDevice));
  }
  {
    // interleaved row records for kernel 1b's graph-row route: {id, 0, weight}; the weight is this IEEE double add
    struct Rec { uint32_t id, pad; double w; };
    static_assert(sizeof(Rec) == 16, "row record must be 16 bytes");
    std::vector<Rec> rec((size_t)nnz);
    for (int64_t e = 0; e < nnz; e++) rec[(size_t)e] = Rec{(uint32_t)col[e], 0u, kappa[e] + 1.0};
    CK(g->rec.reserve(std::max<size_t>((size_t)nnz * 16, 16)));
    g->gv.rec = g->rec.as<uint4>();
    if (nnz) CK(cudaMemcpy((void*)g->gv.rec, rec.data(), (size_t)nnz * 16, cudaMemcpyHostToDevice));
  }
  {
    // per node: smallest weight kappa + 1 of its row as a float rounded DOWN (settling margin of the graph-row route)
    std::vector<float> mw((size_t)N, 3.0e38f);
    for (int32_t x = 0; x < N; x++) {
      double lo = 3.0e38;
      for (int32_t e = rowptr[x]; e < rowptr[x + 1]; e++) lo = std::min(lo, kappa[e] + 1.0);
      float f = (float)lo;
      if ((double)f > lo) f = std::nextafterf(f, -INFINITY);
      mw[(size_t)x] = f;
    }
    CK(g->gminw.reserve((size_t)N * sizeof(float)));
    CK(cudaMemcpy(g->gminw.p, mw.data(), (size_t)N * sizeof(float), cudaMemcpyHostToDevice));
  }

  CK(g->work_counter.reserve(64));
  return TLC_OK;
}

extern "C" {

int tlc_graph_destroy(tlc_graph* g) {
  if (!g) return TLC_OK;
  cudaSetDevice(g->device);
  delete g;
  return TLC_OK;
}

int tlc_vicinity_pi_dev(tlc_graph* g, const int32_t* dev_targets, int64_t E, const tlc_params* p, double* dev_out_pi,
                        float* dev_out_pi_f32, uint8_t* dev_out_status, int64_t* cnt_compute) {
  if (!g || (E > 0 && (!dev_targets || !dev_out_pi))) return fail(TLC_E_INVALID, "NULL argument");
  uint8_t* st = dev_out_status;
  if (!st && cnt_compute && E > 0) {  // the count needs the statuses: the graph's grow-only staging, no cudaMalloc per call
    CK(cudaSetDevice(g->device));
    const int rc0 = ensure_io_buffers(g, E, 0);
    if (rc0) return rc0;
    st = g->io_st.as<uint8_t>();
  }
  return run_pipeline(g, dev_targets, E, p, dev_out_pi, dev_out_pi_f32, st, cnt_compute, nullptr);
}

int tlc_vicinity_pi(tlc_graph* g, const int32_t* targets, int64_t E, const tlc_params* p, double* out_pi,
                    uint8_t* out_status, int64_t* cnt_compute) {
  if (!g || (E > 0 && (!targets || !out_pi))) return fail(TLC_E_INVALID, "NULL argument");
  int rc = check_params(p);
  if (rc) return rc;
  if (cnt_compute) *cnt_compute = 0;
  if (E == 0) return TLC_OK;
  CK(cudaSetDevice(g->device));
  const int r2 = p->resolution * p->resolution;
  if ((rc = ensure_io_buffers(g, E, r2))) return rc;  // grow-only device staging: no cudaMalloc/cudaFree per call
  int32_t* d_t = g->io_t.as<int32_t>();
  double* d_pi = g->io_pi.as<double>();
  uint8_t* d_st = g->io_st.as<uint8_t>();
  CK(cudaMemcpyAsync(d_t, targets, (size_t)E * 8, cudaMemcpyHostToDevice, g->stream));
  // (cnt_compute is taken from the statuses that travel to the host anyway: no extra copy + synchronisation inside the pipeline)
  rc = run_pipeline(g, d_t, E, p, d_pi, nullptr, d_st, nullptr, nullptr);
  if (rc == TLC_OK) {
    uint8_t* h_st = out_status;
    if (!h_st && cnt_compute) {
      CK(g->h_pin.reserve((size_t)E + ALIGN));
      h_st = g->h_pin.as<uint8_t>();
    }
    cudaError_t e1 = cudaMemcpyAsync(out_pi, d_pi, (size_t)E * r2 * 8, cudaMemcpyDeviceToHost, g->stream);
    cudaError_t e2 = h_st ? cudaMemcpyAsync(h_st, d_st, (size_t)E, cudaMemcpyDeviceToHost, g->stream) : cudaSuccess;
    cudaError_t e3 = cudaStreamSynchronize(g->stream);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) rc = fail(TLC_E_CUDA, "copy back failed");
    else if (cnt_compute) *cnt_compute = count_computed(h_st, E);
  }
  return rc;
}

int tlc_vicinity_sizes(tlc_graph* g, const int32_t* targets, int64_t E, const tlc_params* up, int32_t* out_n,
                       int32_t* out_m, uint8_t* out_status) {
  if (!g || (E > 0 && !targets)) return fail(TLC_E_INVALID, "NULL argument");
  int rc = check_params(up);
  if (rc) return rc;
  if (E == 0) return TLC_OK;
  CK(cudaSetDevice(g->device));
  const Params p = to_params(up);
  if ((rc = prepare_call(g, p, E))) return rc;
  if ((rc = ensure_io_buffers(g, E, 0))) return rc;  // grow-only device staging: no cudaMalloc / cudaFree per call
  int32_t* d_t = g->io_t.as<int32_t>();
  CK(cudaMemcpyAsync(d_t, targets, (size_t)E * 8, cudaMemcpyHostToDevice, g->stream));
  VicinityScratch vs = make_vs(g);
  launch_ball_cache(g->gv, p, d_t, E, vs, g->stream);
  launch_vicinity_sizes(g->gv, p, d_t, E, g->d_n.as<int32_t>(), g->d_m.as<int32_t>(), g->d_ds.as<int32_t>(),
                        g->d_st.as<uint8_t>(), g->d_bytes.as<double>(), vs, g->work_counter.as<int>(), g->stream);
  if (out_n) CK(cudaMemcpyAsync(out_n, g->d_n.p, (size_t)E * 4, cudaMemcpyDeviceToHost, g->stream));
  if (out_m) CK(cudaMemcpyAsync(out_m, g->d_m.p, (size_t)E * 4, cudaMemcpyDeviceToHost, g->stream));
  if (out_status) CK(cudaMemcpyAsync(out_status, g->d_st.p, (size_t)E, cudaMemcpyDeviceToHost, g->stream));
  CK(cudaStreamSynchronize(g->stream));
  CK(cudaGetLastError());
  return TLC_OK;
}

int tlc_vicinity_detail(tlc_graph* g, const int32_t* targets, int64_t E, const tlc_params* p, tlc_detail* out) {
  if (!g || !out || (E > 0 && !targets)) return fail(TLC_E_INVALID, "NULL argument");
  int rc = check_params(p);
  if (rc) return rc;
  if (E == 0) return TLC_OK;
  CK(cudaSetDevice(g->device));
  const int r2 = p->resolution * p->resolution;
  if ((rc = ensure_io_buffers(g, E, r2))) return rc;  // grow-only device staging shared with tlc_vicinity_pi
  int32_t* d_t = g->io_t.as<int32_t>();
  double* d_pi = g->io_pi.as<double>();
  uint8_t* d_st = g->io_st.as<uint8_t>();
  CK(cudaMemcpyAsync(d_t, targets, (size_t)E * 8, cudaMemcpyHostToDevice, g->stream));
  int64_t cnt = 0;
  g->detail_chunk.T = 0;
  rc = run_pipeline(g, d_t, E, p, d_pi, nullptr, d_st, &cnt, out);
  if (rc == TLC_OK && out->pi) {
    if (cudaMemcpy(out->pi, d_pi, (size_t)E * r2 * 8, cudaMemcpyDeviceToHost) != cudaSuccess) rc = fail(TLC_E_CUDA, "copy back failed");
  }
  // the two single-kind images of the PDGNN generators: kernel 4 again over the chunk the call left in the arena
  for (int which = 0; which < 2 && rc == TLC_OK; which++) {
    double* dst = which == 0 ? out->pi_up : out->pi_one;
    if (!dst) continue;
    Params pp = to_params(p);
    pp.img_mask = 1u << (which == 0 ? TLC_K_UP : TLC_K_ONE);
    if (cudaMemsetAsync(d_pi, 0, (size_t)E * r2 * 8, g->stream) != cudaSuccess) { rc = fail(TLC_E_CUDA, "memset failed"); break; }
    if (g->detail_chunk.T == E) launch_pimg(pp, g->detail_chunk, d_pi, nullptr, nullptr, 64, g->stream);
    if (cudaMemcpyAsync(dst, d_pi, (size_t)E * r2 * 8, cudaMemcpyDeviceToHost, g->stream) != cudaSuccess ||
        cudaStreamSynchronize(g->stream) != cudaSuccess)
      rc = fail(TLC_E_CUDA, "copy back failed");
  }
  return rc;
}

int tlc_small_diagrams(tlc_graph* g, const int32_t* targets, int64_t E, const tlc_params* up, const int64_t* poff,
                       int32_t* npairs, int32_t* pkind, int32_t* pbv, int32_t* pdv, double* pbirth, double* pdeath,
                       double* out_pi, uint8_t* out_status, int32_t* out_n, int32_t* out_m) {
  if (!g || (E > 0 && (!targets || !poff))) return fail(TLC_E_INVALID, "NULL argument");
  int rc = check_params(up);
  if (rc) return rc;
  if (E == 0) return TLC_OK;
  if (E >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "E must be < 2^31");
  if (up->resolution != 5 || up->descriptor < 0 || up->descriptor > 2 ||
      (up->flags & TLC_F_FILT_ANY_STRUCT))
    return fail(TLC_E_INVALID, "kernel S serves the Ricci-distance filtrations with a 5 x 5 image");
  CK(cudaSetDevice(g->device));
  const Params p = to_params(up);
  if ((rc = prepare_call(g, p, E))) return rc;
  if (!g->ball_cache.p) return fail(TLC_E_NOMEM, "no ball cache for this graph (TLC_BALL_CACHE_GB)");
  if ((rc = ensure_small_buffers(g, E))) return rc;
  if ((rc = ensure_io_buffers(g, E, 25))) return rc;
  const int64_t P = poff[E];
  DevBuf b_poff, b_np, b_kind, b_bv, b_dv, b_birth, b_death;
  CK(b_poff.reserve((size_t)(E + 1) * 8)); CK(b_np.reserve((size_t)E * 4)); CK(b_kind.reserve((size_t)P + 16));
  CK(b_bv.reserve((size_t)P * 4 + 16)); CK(b_dv.reserve((size_t)P * 4 + 16)); CK(b_birth.reserve((size_t)P * 8 + 16)); CK(b_death.reserve((size_t)P * 8 + 16));
  cudaStream_t st = g->stream;
  int32_t* d_t = g->io_t.as<int32_t>();
  double* d_pi = g->io_pi.as<double>();
  uint8_t* d_st = g->io_st.as<uint8_t>();
  CK(cudaMemcpyAsync(d_t, targets, (size_t)E * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(b_poff.p, poff, (size_t)(E + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(b_np.p, 0, (size_t)E * 4, st));
  CK(cudaMemsetAsync(d_st, 255, (size_t)E, st));  // rows kernel S does not take keep TLC_ST_NOT_SMALL
  CK(cudaMemsetAsync(d_pi, 0, (size_t)E * 25 * 8, st));
  CK(cudaMemsetAsync(g->d_n.p, 0, (size_t)E * 4, st));
  CK(cudaMemsetAsync(g->d_m.p, 0, (size_t)E * 4, st));
  SmallDiag dg{b_poff.as<int64_t>(), b_np.as<int32_t>(), b_kind.as<uint8_t>(), b_bv.as<int32_t>(), b_dv.as<int32_t>(),
               b_birth.as<double>(), b_death.as<double>()};
  VicinityScratch vs = make_vs(g);
  launch_ball_cache(g->gv, p, d_t, E, vs, st);
  launch_small(g->gv, p, d_t, E, vs, d_pi, nullptr, d_st, g->sm_list_b.as<int32_t>(), g->sm_list_c.as<int32_t>(),
               g->sm_list_big.as<int32_t>(), g->sm_dev.as<int>(), g->d_n.as<int32_t>(), g->d_m.as<int32_t>(), &dg, nullptr,
               g->sm_count, 3, st);
  std::vector<uint8_t> k8((size_t)P + 1);
  if (npairs) CK(cudaMemcpyAsync(npairs, b_np.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  if (P > 0) {
    CK(cudaMemcpyAsync(k8.data(), b_kind.p, (size_t)P, cudaMemcpyDeviceToHost, st));
    if (pbv) CK(cudaMemcpyAsync(pbv, b_bv.p, (size_t)P * 4, cudaMemcpyDeviceToHost, st));
    if (pdv) CK(cudaMemcpyAsync(pdv, b_dv.p, (size_t)P * 4, cudaMemcpyDeviceToHost, st));
    if (pbirth) CK(cudaMemcpyAsync(pbirth, b_birth.p, (size_t)P * 8, cudaMemcpyDeviceToHost, st));
    if (pdeath) CK(cudaMemcpyAsync(pdeath, b_death.p, (size_t)P * 8, cudaMemcpyDeviceToHost, st));
  }
  if (out_pi) CK(cudaMemcpyAsync(out_pi, d_pi, (size_t)E * 25 * 8, cudaMemcpyDeviceToHost, st));
  if (out_status) CK(cudaMemcpyAsync(out_status, d_st, (size_t)E, cudaMemcpyDeviceToHost, st));
  if (out_n) CK(cudaMemcpyAsync(out_n, g->d_n.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  if (out_m) CK(cudaMemcpyAsync(out_m, g->d_m.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (pkind) for (int64_t i = 0; i < P; i++) pkind[i] = k8[(size_t)i];
  return TLC_OK;
}

}  // extern "C"

// the checks of both diagram entry points, before any CUDA call
static int check_diagram_args(tlc_graph* g, const int32_t* targets, int64_t E, const tlc_params* p, const tlc_diagrams* out) {
  if (!g) return fail(TLC_E_INVALID, "graph is NULL");
  if (!out || !out->poff) return fail(TLC_E_INVALID, "out and out->poff are required");
  if (out->cap < 0) return fail(TLC_E_INVALID, "out->cap must be >= 0");
  if (E < 0 || E >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "E must be in [0, 2^31)");
  if (E > 0 && !targets) return fail(TLC_E_INVALID, "targets is NULL");
  return check_params(p);
}

// the whole path over device-resident targets with pair collection; poff[0..E] (device) receives the final offsets,
// *total their sum.  The pairs stay in the staging until gather_diagrams.
static int run_diagrams(tlc_graph* g, const int32_t* d_targets, int64_t E, const tlc_params* p, double* d_pi,
                        uint8_t* d_status, int64_t* d_poff, int64_t* total) {
  DiagCollect& d = g->dg;
  cudaStream_t st = g->stream;
  CK(d.np.reserve((size_t)E * 4));
  CK(d.soff.reserve((size_t)E * 8));
  CK(cudaMemsetAsync(d.np.p, 0, (size_t)E * 4, st));  // targets no stage finishes have no pairs
  d.small_total = 0;
  d.staged_used = 0;
  d.on = true;
  const int rc = run_pipeline(g, d_targets, E, p, d_pi, nullptr, d_status, nullptr, nullptr);
  d.on = false;
  if (rc) return rc;
  launch_scan_counts(d.np.as<int32_t>(), E, d_poff, st);
  CK(cudaMemcpyAsync(total, d_poff + E, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  return TLC_OK;
}

static void gather_diagrams(tlc_graph* g, int64_t E, const int64_t* d_poff, const DiagArea& out) {
  const DiagCollect& d = g->dg;
  launch_gather_pairs(d.np.as<int32_t>(), d.soff.as<int64_t>(), d_poff, E, d.small.view(), d.staged.view(), d.small_total,
                      out, g->sm_count, g->stream);
}

static int capacity_error(int64_t total, int64_t cap) {
  return fail(TLC_E_CAPACITY, "the diagrams hold " + std::to_string(total) + " pairs, out->cap is " + std::to_string(cap));
}

extern "C" {

int tlc_vicinity_diagrams_dev(tlc_graph* g, const int32_t* dev_targets, int64_t E, const tlc_params* p, tlc_diagrams* out,
                              double* dev_out_pi, uint8_t* dev_out_status, int64_t* total_pairs) {
  int rc = check_diagram_args(g, dev_targets, E, p, out);
  if (rc) return rc;
  CK(cudaSetDevice(g->device));
  cudaStream_t st = g->stream;
  int64_t total = 0;
  if (E == 0) {
    CK(cudaMemsetAsync(out->poff, 0, 8, st));
    CK(cudaStreamSynchronize(st));
  } else {
    double* d_pi = dev_out_pi;
    if (!d_pi) {  // the image rows are computed anyway: the graph's grow-only staging takes them
      if ((rc = ensure_io_buffers(g, E, p->resolution * p->resolution))) return rc;
      d_pi = g->io_pi.as<double>();
    }
    if ((rc = run_diagrams(g, dev_targets, E, p, d_pi, dev_out_status, out->poff, &total))) return rc;
    if (out->npairs) CK(cudaMemcpyAsync(out->npairs, g->dg.np.p, (size_t)E * 4, cudaMemcpyDeviceToDevice, st));
    if (total <= out->cap) gather_diagrams(g, E, out->poff, DiagArea{out->kind, out->bv, out->dv, out->birth, out->death});
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
  }
  if (total_pairs) *total_pairs = total;
  return total > out->cap ? capacity_error(total, out->cap) : TLC_OK;
}

int tlc_vicinity_diagrams(tlc_graph* g, const int32_t* targets, int64_t E, const tlc_params* p, tlc_diagrams* out,
                          double* out_pi, uint8_t* out_status, int64_t* total_pairs) {
  int rc = check_diagram_args(g, targets, E, p, out);
  if (rc) return rc;
  CK(cudaSetDevice(g->device));
  cudaStream_t st = g->stream;
  int64_t total = 0;
  out->poff[0] = 0;
  if (E > 0) {
    const int r2 = p->resolution * p->resolution;
    if ((rc = ensure_io_buffers(g, E, r2))) return rc;  // grow-only device staging shared with tlc_vicinity_pi
    int32_t* d_t = g->io_t.as<int32_t>();
    double* d_pi = g->io_pi.as<double>();
    uint8_t* d_st = g->io_st.as<uint8_t>();
    DiagCollect& d = g->dg;
    CK(d.poff.reserve((size_t)(E + 1) * 8));
    CK(cudaMemcpyAsync(d_t, targets, (size_t)E * 8, cudaMemcpyHostToDevice, st));
    if ((rc = run_diagrams(g, d_t, E, p, d_pi, d_st, d.poff.as<int64_t>(), &total))) return rc;
    CK(cudaMemcpyAsync(out->poff, d.poff.p, (size_t)(E + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (out->npairs) CK(cudaMemcpyAsync(out->npairs, d.np.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
    if (out_pi) CK(cudaMemcpyAsync(out_pi, d_pi, (size_t)E * r2 * 8, cudaMemcpyDeviceToHost, st));
    if (out_status) CK(cudaMemcpyAsync(out_status, d_st, (size_t)E, cudaMemcpyDeviceToHost, st));
    if (total <= out->cap && total > 0) {
      CK(d.out.grow(0, total, st));
      const DiagArea a = d.out.view();
      gather_diagrams(g, E, d.poff.as<int64_t>(), a);
      if (out->kind) CK(cudaMemcpyAsync(out->kind, a.kind, (size_t)total, cudaMemcpyDeviceToHost, st));
      if (out->bv) CK(cudaMemcpyAsync(out->bv, a.bv, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
      if (out->dv) CK(cudaMemcpyAsync(out->dv, a.dv, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
      if (out->birth) CK(cudaMemcpyAsync(out->birth, a.birth, (size_t)total * 8, cudaMemcpyDeviceToHost, st));
      if (out->death) CK(cudaMemcpyAsync(out->death, a.death, (size_t)total * 8, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
  }
  if (total_pairs) *total_pairs = total;
  return total > out->cap ? capacity_error(total, out->cap) : TLC_OK;
}

static constexpr uint32_t VICINITY_BATCH_FLAGS = TLC_F_NORM | TLC_F_NORM_EPS | TLC_F_SUM_PLAIN | TLC_F_FILT_ANY_STRUCT;

int tlc_vicinity_batch_dev(tlc_graph* g, const int32_t* dev_targets, int64_t E, const tlc_params* p,
                           tlc_vicinity_batch* out, uint8_t* dev_status, int64_t* total_v, int64_t* total_e) {
  if (!g) return fail(TLC_E_INVALID, "graph is NULL");
  if (!out || !out->voff || !out->eoff) return fail(TLC_E_INVALID, "out, out->voff and out->eoff are required");
  if (out->cap_v < 0 || out->cap_e < 0) return fail(TLC_E_INVALID, "out->cap_v and out->cap_e must be >= 0");
  if (E < 0 || E >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "E must be in [0, 2^31)");
  if (E > 0 && !dev_targets) return fail(TLC_E_INVALID, "targets is NULL");
  if (!p) return fail(TLC_E_INVALID, "params is NULL");
  if (p->flags & ~VICINITY_BATCH_FLAGS)
    return fail(TLC_E_INVALID, "flags may only hold TLC_F_NORM, TLC_F_NORM_EPS, TLC_F_SUM_PLAIN and the TLC_F_FILT_* filtrations");
  tlc_params q = *p;  // (resolution and img_mask are ignored)
  q.resolution = 1;
  q.img_mask = 0;
  int rc = check_params(&q);
  if (rc) return rc;
  CK(cudaSetDevice(g->device));
  cudaStream_t st = g->stream;
  BatchCollect& b = g->vb;
  b.out = *out;
  b.status = dev_status;
  b.total_v = 0; b.total_e = 0;
  if (E == 0) {
    CK(cudaMemsetAsync(out->voff, 0, 8, st));
    CK(cudaMemsetAsync(out->eoff, 0, 8, st));
    CK(cudaStreamSynchronize(st));
    g->last = CallStats();
  } else {
    CallStats s;
    b.on = true;
    rc = run_staged(g, dev_targets, E, &q, nullptr, nullptr, dev_status, nullptr, nullptr, s, 0);
    b.on = false;
    g->last = s;
    if (rc == TLC_OK) {
      CK(cudaStreamSynchronize(st));
      CK(cudaGetLastError());
    }
  }
  if (total_v) *total_v = b.total_v;
  if (total_e) *total_e = b.total_e;
  return rc;
}

int tlc_ollivier_ricci(int device, int32_t N, int64_t nnz, const int32_t* rowptr, const int32_t* col, double alpha,
                       double* out_kappa, int32_t* out_iters) {
  if (N <= 0 || nnz < 0 || !rowptr || (nnz > 0 && (!col || !out_kappa))) return fail(TLC_E_INVALID, "bad arguments");
  if (!(alpha >= 0.0 && alpha <= 1.0)) return fail(TLC_E_INVALID, "alpha must lie in [0, 1]");
  int rc = check_csr(N, nnz, rowptr, col, nullptr);  // (OllivierRicci removes self-loops: none may be given)
  if (rc) return rc;
  // edge list (x < y), mirror positions, support sizes
  const int TOPK = 3000;
  std::vector<int64_t> epos, emir;
  std::vector<int32_t> esrc;
  std::vector<int64_t> esize;
  for (int32_t x = 0; x < N; x++) {
    for (int64_t e = rowptr[x]; e < rowptr[x + 1]; e++) {
      const int32_t y = col[e];
      const int32_t* lo = col + rowptr[y];
      const int32_t* hi = col + rowptr[y + 1];
      const int32_t* it = std::lower_bound(lo, hi, x);  // (present: check_csr)
      if (x < y) {
        epos.push_back(e); emir.push_back(it - col); esrc.push_back(x);
        const int64_t sa = std::min<int64_t>(rowptr[x + 1] - rowptr[x], TOPK) + 1, sb = std::min<int64_t>(rowptr[y + 1] - rowptr[y], TOPK) + 1;
        esize.push_back(std::max(sa, sb));
      }
    }
  }
  if (nnz == 0) return TLC_OK;
  if ((rc = select_device(device))) return rc;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  const int sms = prop.multiProcessorCount;
  const int64_t E = (int64_t)epos.size();
  // size classes: both supports <= 120 (vectors and the code matrix in shared memory, several CTAs per SM),
  // <= 1024 (vectors in shared memory, codes in HBM), the rest (<= 3001)
  std::vector<int64_t> order((size_t)E);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int64_t p, int64_t q) { return esize[(size_t)p] < esize[(size_t)q]; });
  std::vector<int64_t> h_pos((size_t)E), h_mir((size_t)E);
  std::vector<int32_t> h_src((size_t)E);
  int64_t c0 = 0, c1 = 0;
  for (int64_t i = 0; i < E; i++) {
    const int64_t o = order[(size_t)i];
    h_pos[(size_t)i] = epos[(size_t)o]; h_mir[(size_t)i] = emir[(size_t)o]; h_src[(size_t)i] = esrc[(size_t)o];
    if (esize[(size_t)o] <= 120) c0 = i + 1;
    if (esize[(size_t)o] <= 1024) c1 = i + 1;
  }
  const size_t Wc = ((size_t)N + 31) / 32;
  DevBuf b_rp, b_col, b_b1, b_b2, b_acc, b_state, b_list, b_cnt, b_tg, b_pos, b_mir, b_src, b_out, b_it, b_wsum, b_slab, b_bm;
  CK(b_rp.reserve((size_t)(N + 1) * 4)); CK(b_col.reserve((size_t)nnz * 4));
  CK(b_b1.reserve((size_t)N * Wc * 4)); CK(b_b2.reserve((size_t)N * Wc * 4));
  CK(b_acc.reserve((size_t)N * 16)); CK(b_state.reserve((size_t)N * 4)); CK(b_list.reserve((size_t)N * 4)); CK(b_cnt.reserve(64));
  CK(b_tg.reserve((size_t)N * 8));
  CK(b_pos.reserve((size_t)E * 8)); CK(b_mir.reserve((size_t)E * 8)); CK(b_src.reserve((size_t)E * 4));
  CK(b_out.reserve((size_t)nnz * 8)); CK(b_it.reserve((size_t)nnz * 4)); CK(b_wsum.reserve((size_t)(TOPK + 1) * 8));
  cudaStream_t st = nullptr;
  CK(cudaMemcpy(b_rp.p, rowptr, (size_t)(N + 1) * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b_col.p, col, (size_t)nnz * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b_pos.p, h_pos.data(), (size_t)E * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b_mir.p, h_mir.data(), (size_t)E * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b_src.p, h_src.data(), (size_t)E * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(b_out.p, 0, (size_t)nnz * 8));
  CK(cudaMemset(b_it.p, 0, (size_t)nnz * 4));
  {
    std::vector<int32_t> tg((size_t)N * 2);
    for (int32_t i = 0; i < N; i++) { tg[2 * (size_t)i] = i; tg[2 * (size_t)i + 1] = i; }
    CK(cudaMemcpy(b_tg.p, tg.data(), (size_t)N * 8, cudaMemcpyHostToDevice));
    // neighbour weight base ** (-(w ** exp_power)) = e ** -1 and its running sums, as python's sum() adds them
    const double wnb = std::exp(-1.0);
    std::vector<double> ws((size_t)TOPK + 1, 0.0);
    for (int k = 1; k <= TOPK; k++) ws[(size_t)k] = ws[(size_t)k - 1] + wnb;
    CK(cudaMemcpy(b_wsum.p, ws.data(), ws.size() * 8, cudaMemcpyHostToDevice));
  }
  // closed 1-hop and 2-hop balls of every node (kernel 1's ball expansion)
  GraphView gv{N, nnz, b_rp.as<int32_t>(), b_col.as<int32_t>(), nullptr, nullptr};
  for (int hop = 1; hop <= 2; hop++) {
    Params pp{hop, TLC_MODE_NODE, TLC_DESC_SUM, 5, 0, 0};
    size_t Wd = 0;
    bool smem = false;
    const int grid = vicinity_grid(device, gv, pp, &Wd, &smem);
    if (!smem && !b_bm.p) CK(b_bm.reserve((size_t)grid * 2 * Wd * 4));
    CK(cudaMemset(b_state.p, 0, (size_t)N * 4));
    VicinityScratch vs{smem ? nullptr : b_bm.as<uint32_t>(), nullptr, grid, (hop == 1 ? b_b1 : b_b2).as<uint32_t>(),
                       b_acc.as<unsigned long long>(), b_state.as<int32_t>(), b_list.as<int32_t>(), b_cnt.as<int>()};
    launch_ball_cache(gv, pp, b_tg.as<int32_t>(), N, vs, st);
  }
  const double kval[4] = {std::exp(0.0 / -1e-1), std::exp(1.0 / -1e-1), std::exp(2.0 / -1e-1), std::exp(3.0 / -1e-1)};
  const double wnb = std::exp(-1.0);
  auto run = [&](int64_t lo, int64_t hi, int cap, bool codes_smem, int per_sm) -> int {
    if (hi <= lo) return TLC_OK;
    const int grid = (int)std::min<int64_t>(hi - lo, (int64_t)sms * per_sm);
    size_t stride = 0;
    if (!codes_smem) {
      stride = ((size_t)cap * cap + 255) / 256 * 256;
      CK(b_slab.reserve(stride * (size_t)grid));
    }
    launch_ricci(b_rp.as<int32_t>(), b_col.as<int32_t>(), b_b1.as<uint32_t>(), b_b2.as<uint32_t>(), (int)Wc,
                 b_pos.as<int64_t>() + lo, b_mir.as<int64_t>() + lo, b_src.as<int32_t>() + lo, hi - lo, alpha, kval,
                 b_wsum.as<double>(), wnb, TOPK, 1000, 1e-9, cap, codes_smem, b_slab.as<uint8_t>(), stride, grid,
                 b_out.as<double>(), b_it.as<int32_t>(), st);
    return TLC_OK;
  };
  if ((rc = run(0, c0, 120, true, 8))) return rc;
  if ((rc = run(c0, c1, 1024, false, 2))) return rc;
  if ((rc = run(c1, E, TOPK + 1, false, 1))) return rc;
  CK(cudaDeviceSynchronize());
  CK(cudaGetLastError());
  CK(cudaMemcpy(out_kappa, b_out.p, (size_t)nnz * 8, cudaMemcpyDeviceToHost));
  if (out_iters) CK(cudaMemcpy(out_iters, b_it.p, (size_t)nnz * 4, cudaMemcpyDeviceToHost));
  return TLC_OK;
}

int tlc_union_find(int device, int32_t n, int32_t m, const double* fval, const int32_t* a, const int32_t* b, uint32_t flags,
                   int32_t* npairs, int32_t* pkind, int32_t* pbv, int32_t* pdv, double* pbirth, double* pdeath,
                   int32_t* npos, int32_t* pos, int32_t* nneg, int32_t* neg, uint8_t* status) {
  if (n <= 0 || m < 0 || !fval || (m > 0 && (!a || !b))) return fail(TLC_E_INVALID, "bad arguments");
  for (int32_t i = 0; i < m; i++)
    if (a[i] < 0 || a[i] >= n || b[i] < 0 || b[i] >= n) return fail(TLC_E_INVALID, "edge endpoint out of range");
  int rc = select_device(device);
  if (rc) return rc;
  DevBuf arena;
  CK(arena.reserve(chunk_bytes(1, n, m, 0)));
  ChunkView c = carve(arena.as<char>(), 1, n, m, 0, nullptr);
  cudaStream_t st = nullptr;  // legacy default stream: the plain cudaMemcpy calls below order with it
  const int64_t zero = 0, nv = n, ne = m;
  const int32_t one_n = n, one_m = m, z32 = 0;
  const uint8_t st_ok = TLC_ST_OK;
  CK(cudaMemcpy((void*)c.tidx, &zero, 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy((void*)c.voff, &zero, 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy((void*)(c.voff + 1), &nv, 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy((void*)c.eoff, &zero, 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy((void*)(c.eoff + 1), &ne, 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c.tn, &one_n, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c.tm, &one_m, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c.tnp, &z32, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c.tnpos, &z32, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c.tnneg, &z32, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c.tstatus, &st_ok, 1, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c.fval, fval, (size_t)n * 8, cudaMemcpyHostToDevice));
  if (m) {
    CK(cudaMemcpy(c.elo, a, (size_t)m * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c.ehi, b, (size_t)m * 4, cudaMemcpyHostToDevice));
  }
  Params p{0, TLC_MODE_NODE, TLC_DESC_SUM, 5, flags, 0};
  const int block = block_for(m);
  launch_sort(p, c, block, 3, 0, st);
  const int64_t uf_ints = 2 * (int64_t)n * 4 <= 96 * 1024 ? 2 * (int64_t)n : 0;
  launch_union_find(p, c, block, (int)uf_ints, 1, 3, 0, st);
  if (flags & TLC_F_EXTENDED) {
    const int64_t lp_ints = 3 * (int64_t)n * 4 <= 200 * 1024 ? 3 * (int64_t)n : 0;
    launch_loops(p, c, std::min(block, 128), (int)lp_ints, n, st);
  }
  CK(cudaDeviceSynchronize());
  CK(cudaGetLastError());
  int32_t h_np = 0, h_npos = 0, h_nneg = 0;
  uint8_t h_st = 0;
  CK(cudaMemcpy(&h_np, c.tnp, 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&h_npos, c.tnpos, 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&h_nneg, c.tnneg, 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&h_st, c.tstatus, 1, cudaMemcpyDeviceToHost));
  if (npairs) *npairs = h_np;
  if (npos) *npos = h_npos;
  if (nneg) *nneg = h_nneg;
  if (status) *status = h_st;
  if (h_np > 0) {
    if (pkind) {
      std::vector<uint8_t> k8((size_t)h_np);
      CK(cudaMemcpy(k8.data(), c.pkind, (size_t)h_np, cudaMemcpyDeviceToHost));
      for (int i = 0; i < h_np; i++) pkind[i] = k8[i];
    }
    if (pbv) CK(cudaMemcpy(pbv, c.pbv, (size_t)h_np * 4, cudaMemcpyDeviceToHost));
    if (pdv) CK(cudaMemcpy(pdv, c.pdv, (size_t)h_np * 4, cudaMemcpyDeviceToHost));
    if (pbirth) CK(cudaMemcpy(pbirth, c.pbirth, (size_t)h_np * 8, cudaMemcpyDeviceToHost));
    if (pdeath) CK(cudaMemcpy(pdeath, c.pdeath, (size_t)h_np * 8, cudaMemcpyDeviceToHost));
  }
  if (pos && h_npos > 0) CK(cudaMemcpy(pos, c.pos, (size_t)h_npos * 4, cudaMemcpyDeviceToHost));
  if (neg && h_nneg > 0) CK(cudaMemcpy(neg, c.neg, (size_t)h_nneg * 4, cudaMemcpyDeviceToHost));
  return TLC_OK;
}

int tlc_pimg_transform(int device, const double* dgm, int64_t K, int32_t resolution, double* out) {
  if (!out || (K > 0 && !dgm) || resolution < 1 || resolution > 16) return fail(TLC_E_INVALID, "bad arguments");
  int rc = select_device(device);
  if (rc) return rc;
  // one diagram of the batch imager: poff {0, K}, then the births and the deaths, uploaded in one copy
  std::vector<double> h(2 * (size_t)K + 2);
  const int64_t off[2] = {0, K};
  std::memcpy(h.data(), off, sizeof off);
  for (int64_t k = 0; k < K; k++) { h[2 + k] = dgm[2 * k]; h[2 + K + k] = dgm[2 * k + 1]; }
  DevBuf b_in, b_out;
  CK(b_in.reserve(h.size() * 8));
  CK(b_out.reserve((size_t)resolution * resolution * 8));
  CK(cudaMemcpy(b_in.p, h.data(), h.size() * 8, cudaMemcpyHostToDevice));
  const double* d_in = b_in.as<double>();
  launch_pimg_batch(b_in.as<int64_t>(), d_in + 2, d_in + 2 + K, nullptr, 0u, resolution, 1, b_out.as<double>(), nullptr);
  CK(cudaMemcpy(out, b_out.p, (size_t)resolution * resolution * 8, cudaMemcpyDeviceToHost));
  CK(cudaGetLastError());
  return TLC_OK;
}

// the checks both batch imager calls make before any CUDA call
static int check_pimg_batch(int64_t D, const int64_t* poff, const double* birth, const double* death, int32_t resolution) {
  if (D < 0 || D >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "D must be in [0, 2^31)");
  if (resolution < 1 || resolution > 16) return fail(TLC_E_INVALID, "resolution must be in 1..16");
  if (D > 0 && !poff) return fail(TLC_E_INVALID, "dev_poff is NULL");
  if (D > 0 && !birth) return fail(TLC_E_INVALID, "dev_birth is NULL");
  if (D > 0 && !death) return fail(TLC_E_INVALID, "dev_death is NULL");
  return TLC_OK;
}

int tlc_pimg_batch_dev(int device, int64_t D, const int64_t* dev_poff, const double* dev_birth, const double* dev_death,
                       const uint8_t* dev_kind, uint32_t img_mask, int32_t resolution, double* dev_out, void* stream) {
  int rc = check_pimg_batch(D, dev_poff, dev_birth, dev_death, resolution);
  if (rc) return rc;
  if (D > 0 && !dev_out) return fail(TLC_E_INVALID, "dev_out is NULL");
  if (D == 0) return TLC_OK;
  if ((rc = select_device(device))) return rc;
  launch_pimg_batch(dev_poff, dev_birth, dev_death, dev_kind, img_mask, resolution, D, dev_out, (cudaStream_t)stream);
  CK(cudaGetLastError());
  return TLC_OK;
}

int tlc_pimg_batch_grad_dev(int device, int64_t D, const int64_t* dev_poff, const double* dev_birth,
                            const double* dev_death, const uint8_t* dev_kind, uint32_t img_mask, int32_t resolution,
                            const double* dev_grad_out, double* dev_grad_birth, double* dev_grad_death, void* stream) {
  int rc = check_pimg_batch(D, dev_poff, dev_birth, dev_death, resolution);
  if (rc) return rc;
  if (D > 0 && !dev_grad_out) return fail(TLC_E_INVALID, "dev_grad_out is NULL");
  if (D == 0 || (!dev_grad_birth && !dev_grad_death)) return TLC_OK;
  if ((rc = select_device(device))) return rc;
  launch_pimg_batch_grad(dev_poff, dev_birth, dev_death, dev_kind, img_mask, resolution, D, dev_grad_out,
                         dev_grad_birth, dev_grad_death, (cudaStream_t)stream);
  CK(cudaGetLastError());
  return TLC_OK;
}

int tlc_wasserstein_workspace_bytes(int64_t D, int64_t Px, int64_t Py, uint64_t* bytes) {
  if (D < 0 || D >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "D must be in [0, 2^31)");
  if (Px < 0 || Py < 0 || Px >= ((int64_t)1 << 56) || Py >= ((int64_t)1 << 56))
    return fail(TLC_E_INVALID, "Px and Py must be in [0, 2^56)");
  if (!bytes) return fail(TLC_E_INVALID, "bytes is NULL");
  *bytes = wasserstein_workspace_bytes(D, Px, Py);
  return TLC_OK;
}

// the checks both Wasserstein calls make before any CUDA call
static int check_wasserstein(int64_t D, const int64_t* poff_x, const double* bx, const double* dx, const int64_t* poff_y,
                             const double* by, const double* dy, double order, double internal_p) {
  if (D < 0 || D >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "D must be in [0, 2^31)");
  if (!(order >= 1.0) || std::isinf(order)) return fail(TLC_E_INVALID, "order must be finite and >= 1");
  if (!(internal_p >= 1.0)) return fail(TLC_E_INVALID, "internal_p must be >= 1 or +inf");
  const char* names[6] = {"dev_poff_x", "dev_birth_x", "dev_death_x", "dev_poff_y", "dev_birth_y", "dev_death_y"};
  const void* ptrs[6] = {poff_x, bx, dx, poff_y, by, dy};
  for (int k = 0; k < 6; k++)
    if (D > 0 && !ptrs[k]) return fail(TLC_E_INVALID, std::string(names[k]) + " is NULL");
  return TLC_OK;
}

int tlc_wasserstein_batch_dev(int device, int64_t D, int64_t Px, int64_t Py, const int64_t* dev_poff_x,
                              const double* dev_birth_x, const double* dev_death_x, const uint8_t* dev_kind_x,
                              const int64_t* dev_poff_y, const double* dev_birth_y, const double* dev_death_y,
                              const uint8_t* dev_kind_y, uint32_t kind_mask, double order, double internal_p,
                              void* dev_workspace, uint64_t workspace_bytes, double* dev_dist, int64_t* dev_match_x,
                              int64_t* dev_match_y, void* stream) {
  int rc = check_wasserstein(D, dev_poff_x, dev_birth_x, dev_death_x, dev_poff_y, dev_birth_y, dev_death_y, order,
                             internal_p);
  if (rc) return rc;
  uint64_t need = 0;
  if ((rc = tlc_wasserstein_workspace_bytes(D, Px, Py, &need))) return rc;
  if (workspace_bytes < need)
    return fail(TLC_E_INVALID, "workspace_bytes is " + std::to_string(workspace_bytes) + ", the call needs " +
                                   std::to_string(need));
  if (D > 0 && need > 0 && !dev_workspace) return fail(TLC_E_INVALID, "dev_workspace is NULL");
  if (D > 0 && !dev_dist) return fail(TLC_E_INVALID, "dev_dist is NULL");
  if (D == 0) return TLC_OK;
  if ((rc = select_device(device))) return rc;
  launch_wasserstein(dev_poff_x, dev_birth_x, dev_death_x, dev_kind_x, dev_poff_y, dev_birth_y, dev_death_y,
                     dev_kind_y, kind_mask, order, internal_p, D, dev_workspace, workspace_bytes, dev_dist,
                     dev_match_x, dev_match_y, (cudaStream_t)stream);
  CK(cudaGetLastError());
  return TLC_OK;
}

int tlc_wasserstein_batch_grad_dev(int device, int64_t D, const int64_t* dev_poff_x, const double* dev_birth_x,
                                   const double* dev_death_x, const uint8_t* dev_kind_x, const int64_t* dev_poff_y,
                                   const double* dev_birth_y, const double* dev_death_y, const uint8_t* dev_kind_y,
                                   uint32_t kind_mask, double order, double internal_p, const double* dev_dist,
                                   const int64_t* dev_match_x, const int64_t* dev_match_y, const double* dev_grad_out,
                                   double* dev_grad_birth_x, double* dev_grad_death_x, double* dev_grad_birth_y,
                                   double* dev_grad_death_y, void* stream) {
  int rc = check_wasserstein(D, dev_poff_x, dev_birth_x, dev_death_x, dev_poff_y, dev_birth_y, dev_death_y, order,
                             internal_p);
  if (rc) return rc;
  if (D > 0 && !dev_dist) return fail(TLC_E_INVALID, "dev_dist is NULL");
  if (D > 0 && !dev_match_x) return fail(TLC_E_INVALID, "dev_match_x is NULL");
  if (D > 0 && !dev_match_y) return fail(TLC_E_INVALID, "dev_match_y is NULL");
  if (D > 0 && !dev_grad_out) return fail(TLC_E_INVALID, "dev_grad_out is NULL");
  if (D == 0 || (!dev_grad_birth_x && !dev_grad_death_x && !dev_grad_birth_y && !dev_grad_death_y)) return TLC_OK;
  if ((rc = select_device(device))) return rc;
  launch_wasserstein_grad(dev_poff_x, dev_birth_x, dev_death_x, dev_kind_x, dev_poff_y, dev_birth_y, dev_death_y,
                          dev_kind_y, kind_mask, order, internal_p, D, dev_dist, dev_match_x, dev_match_y,
                          dev_grad_out, dev_grad_birth_x, dev_grad_death_x, dev_grad_birth_y, dev_grad_death_y,
                          (cudaStream_t)stream);
  CK(cudaGetLastError());
  return TLC_OK;
}

int tlc_pi_gather(int device, const double* dev_table, int64_t rows, int32_t r2, const int64_t* dev_index, int64_t start,
                  int64_t n, float* dev_out_f32, void* stream) {
  if (rows < 0 || r2 < 1 || n < 0 || (n > 0 && (!dev_table || !dev_out_f32))) return fail(TLC_E_INVALID, "bad arguments");
  if (n == 0) return TLC_OK;
  const int rc = select_device(device);
  if (rc) return rc;
  // per host thread and device: the out-of-range flag and the SM count; released when the thread exits
  struct GatherScratch {
    int* d_bad[64] = {nullptr};
    int sms[64] = {0};
    ~GatherScratch() { for (int i = 0; i < 64; i++) if (d_bad[i]) cudaFree(d_bad[i]); }
  };
  static thread_local GatherScratch gs;
  int** d_bad = gs.d_bad;
  int* sms = gs.sms;
  if (device >= 64) return fail(TLC_E_INVALID, "device index out of range");
  if (!d_bad[device]) {
    CK(cudaMalloc((void**)&d_bad[device], sizeof(int)));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    sms[device] = prop.multiProcessorCount;
  }
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemsetAsync(d_bad[device], 0, sizeof(int), st));
  launch_gather_rows(dev_table, rows, r2, dev_index, start, n, dev_out_f32, d_bad[device], sms[device], st);
  int bad = 0;
  CK(cudaMemcpyAsync(&bad, d_bad[device], sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (bad) return fail(TLC_E_INVALID, "row index out of range");
  return TLC_OK;
}

// ---- multi-GPU exchange by peer stores (SURVEY.md 8e) ----
int tlc_table_create(tlc_graph* g, int64_t rows, int32_t r2, void** dev_rows, unsigned char* handle64) {
  if (!g || rows <= 0 || r2 < 1 || !handle64) return fail(TLC_E_INVALID, "bad arguments");
  CK(cudaSetDevice(g->device));
  if (g->peer_own.p) return fail(TLC_E_INVALID, "this graph already owns an exchange table");
  const size_t bytes = PEER_HEADER_BYTES + (size_t)rows * (size_t)(r2 + 1) * sizeof(float);
  CK(g->peer_own.reserve(bytes));
  CK(cudaMemset(g->peer_own.p, 0, bytes));
  if (!g->peer_ticket.p) { CK(g->peer_ticket.reserve(64)); CK(cudaMemset(g->peer_ticket.p, 0, 64)); }
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, g->peer_own.p));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
  memcpy(handle64, &h, 64);
  g->peer_rows = rows; g->peer_r2 = r2; g->peer_epoch = 0;
  g->peers.n = 0;
  if (dev_rows) *dev_rows = g->peer_own.as<unsigned char>() + PEER_HEADER_BYTES;
  return TLC_OK;
}

int tlc_table_attach(tlc_graph* g, int32_t nranks, int32_t my_rank, const unsigned char* handles64) {
  if (!g || !g->peer_own.p || nranks < 1 || nranks > PEER_MAX || my_rank < 0 || my_rank >= nranks || !handles64)
    return fail(TLC_E_INVALID, "bad arguments (create the table first; at most 16 ranks)");
  CK(cudaSetDevice(g->device));
  for (void* q : g->peer_opened) cudaIpcCloseMemHandle(q);
  g->peer_opened.clear();
  g->peers.n = nranks;
  for (int r = 0; r < nranks; r++) {
    if (r == my_rank) { g->peers.table[r] = g->peer_own.p; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles64 + (size_t)r * 64, 64);
    void* q = nullptr;
    CK(cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess));
    g->peer_opened.push_back(q);
    g->peers.table[r] = q;
  }
  return TLC_OK;
}

int tlc_vicinity_pi_exchange(tlc_graph* g, const int32_t* dev_targets, const int64_t* dev_row_index, int64_t E,
                             const tlc_params* p, int64_t* cnt_compute) {
  if (!g || (E > 0 && (!dev_targets || !dev_row_index))) return fail(TLC_E_INVALID, "NULL argument");
  if (!g->peer_own.p || g->peers.n < 1) return fail(TLC_E_INVALID, "no exchange table attached (tlc_table_create / tlc_table_attach)");
  int rc = check_params(p);
  if (rc) return rc;
  const int r2 = p->resolution * p->resolution;
  if (r2 != g->peer_r2) return fail(TLC_E_INVALID, "resolution differs from the exchange table's");
  CK(cudaSetDevice(g->device));
  if (E > g->px_cap) {
    const size_t cap = (size_t)(E + E / 8 + 256);
    CK(g->px_pi32.reserve(cap * r2 * 4));
    CK(g->px_pi.reserve(cap * r2 * 8));
    CK(g->px_st.reserve(cap));
    g->px_cap = (int64_t)cap;
  }
  float* pi32 = g->px_pi32.as<float>();
  uint8_t* sst = g->px_st.as<uint8_t>();
  if (E > 0) {
    rc = run_pipeline(g, dev_targets, E, p, g->px_pi.as<double>(), pi32, sst, cnt_compute, nullptr);
    if (rc) return rc;
  } else if (cnt_compute) *cnt_compute = 0;
  // store this rank's rows into every rank's table at their final index, then wait for everyone's arrival
  launch_peer_scatter(pi32, sst, dev_row_index, E, r2, g->peers, g->peer_ticket.as<unsigned int>(), g->sm_count, g->stream);
  g->peer_epoch++;
  launch_peer_wait(g->peer_own.as<const unsigned int>(), g->peer_epoch * (unsigned int)g->peers.n, g->stream);
  CK(cudaGetLastError());
  return TLC_OK;
}

int tlc_graph_set_hks_time(tlc_graph* g, double t) {
  if (!g) return fail(TLC_E_INVALID, "NULL graph");
  if (!(t > 0.0 && t <= 50.0)) return fail(TLC_E_INVALID, "hks time must lie in (0, 50]");
  g->hks_time = t;
  return TLC_OK;
}

int tlc_graph_set_stream(tlc_graph* g, void* stream) {
  if (!g) return fail(TLC_E_INVALID, "NULL graph");
  g->stream = stream ? (cudaStream_t)stream : g->own_stream;
  return TLC_OK;
}

int tlc_last_counts(tlc_graph* g, int64_t* out5) {  // out5: 8 slots
  if (!g || !out5) return TLC_E_INVALID;
  const CallStats& s = g->last;
  out5[0] = s.live; out5[1] = s.sum_n; out5[2] = s.sum_m; out5[3] = s.chunks; out5[4] = s.handed_back;
  out5[5] = s.general; out5[6] = s.rowcheck; out5[7] = s.blocks;
  return TLC_OK;
}

int64_t tlc_last_direct(tlc_graph* g) { return g ? g->last.direct : 0; }

int64_t tlc_last_table(tlc_graph* g) { return g ? g->last.table : 0; }
int64_t tlc_last_table_two_root(tlc_graph* g) { return g ? g->last.two_root : 0; }
double tlc_table_build_ms(tlc_graph* g) { return g ? g->sssp_build_ms : 0.0; }

int tlc_last_small(tlc_graph* g, double* out7) {
  if (!g || !out7) return TLC_E_INVALID;
  for (int i = 0; i < 3; i++) out7[i] = g->last.small_ms[i];
  for (int i = 0; i < 4; i++) out7[3 + i] = (double)g->last.small_rows[i];
  return TLC_OK;
}

int tlc_last_stage_ms(tlc_graph* g, double* out10) {
  if (!g || !out10) return 0;
  for (int i = 0; i < 10; i++) out10[i] = g->last.stage_ms[i];
  return g->last.chunks;
}

// (the BFS and union-find shares are not measured separately: 0)
int tlc_last_algorithmic_bytes(tlc_graph* g, double* bytes_total, double* bytes_bfs, double* bytes_uf) {
  if (!g) return TLC_E_INVALID;
  if (bytes_total) *bytes_total = g->last.bytes;
  if (bytes_bfs) *bytes_bfs = 0;
  if (bytes_uf) *bytes_uf = 0;
  return TLC_OK;
}

}  // extern "C"

// ---- graph batches: persistence diagrams of caller-supplied graphs (tlc_graph_batch_*, kernel 9) ----
// Each graph takes one route, fixed at creation from its size: kernel 9's fused teams (classes A / B / C) or the staged
// kernels 2 + 3 (+ 3b) over a ChunkView whose segments are the graphs'.  Two such views are carved from one arena: `large`
// (the graphs no class takes, the default route) and `all` (every graph: TLC_F_NO_SMALL).  Their per-graph tables (graph
// id, vertex / edge offsets) are uploaded once; the fill kernel writes the per-call state.
struct StagedView {
  ChunkView c{};
  int64_t n_max = 0, m_max = 0;
};

struct tlc_graph_batch {
  int device = 0, sm_count = 0;
  int64_t D = 0, N = 0, M = 0;
  DevBuf noff, eoff, soff, ea, eb;  // structure; soff[t] = noff[t] + eoff[t] + t: graph t's staging segment
  DevBuf lists;                     // the graph ids of fused classes A, B, C, one after the other
  int counts[3] = {0, 0, 0};
  DevBuf kind, bv, dv, birth, death;  // staging pairs [N + M + D]
  DevBuf np, status;                  // [D] pairs per graph, status (when the caller passes none)
  DevBuf arena, tables;
  StagedView all, large;
  DevBuf gcnt, glst;  // gradient scratch: [N], [2 (N + M + D)]
  int64_t bound() const { return N + M + D; }
};

static constexpr uint32_t GRAPH_BATCH_FLAGS = TLC_F_EXTENDED | TLC_F_KEEP_ZERO | TLC_F_ASC_ONLY | TLC_F_NO_SMALL;

// 0..2: the fused class that takes a graph of n vertices and m edges, 3: the staged kernels
static int graph_route(int64_t n, int64_t m) {
  if (n <= GRAPH_A_N && m <= GRAPH_A_M) return 0;
  if (n <= GRAPH_B_N && m <= GRAPH_B_M) return 1;
  if (n <= GRAPH_C_N && m <= GRAPH_C_M) return 2;
  return 3;
}

// the host-side part of both creations' checks: the offsets (host copies)
static int check_batch_offsets(int64_t D, const int64_t* noff, const int64_t* eoff) {
  if (noff[0] != 0 || eoff[0] != 0) return fail(TLC_E_INVALID, "noff[0] and eoff[0] must be 0");
  for (int64_t t = 0; t < D; t++) {
    if (noff[t + 1] < noff[t]) return fail(TLC_E_INVALID, "noff is not monotone at graph " + std::to_string(t));
    if (eoff[t + 1] < eoff[t]) return fail(TLC_E_INVALID, "eoff is not monotone at graph " + std::to_string(t));
  }
  if (noff[D] >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "noff[D] must be < 2^31");
  if (eoff[D] >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "eoff[D] must be < 2^31");
  return TLC_OK;
}

static int check_graph_batch(int64_t D, const int64_t* noff, const int64_t* eoff, const int32_t* ea, const int32_t* eb) {
  if (D < 0 || D >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "D must be in [0, 2^31)");
  if (!noff || !eoff) return fail(TLC_E_INVALID, "noff and eoff are required");
  const int rc = check_batch_offsets(D, noff, eoff);
  if (rc) return rc;
  const int64_t M = eoff[D];
  if (M > 0 && (!ea || !eb)) return fail(TLC_E_INVALID, "ea and eb are required when there are edges");
  std::vector<std::pair<uint64_t, int64_t>> keys((size_t)M);
  for (int64_t t = 0; t < D; t++)
    for (int64_t k = eoff[t]; k < eoff[t + 1]; k++) {
      const int64_t a = ea[k], b = eb[k];
      const std::string what = "edge " + std::to_string(k) + " (" + std::to_string(a) + ", " + std::to_string(b) +
                               ") of graph " + std::to_string(t);
      if (a < noff[t] || a >= noff[t + 1] || b < noff[t] || b >= noff[t + 1])
        return fail(TLC_E_INVALID, what + " has an endpoint outside the graph's vertices [" + std::to_string(noff[t]) +
                                       ", " + std::to_string(noff[t + 1]) + ")");
      if (a == b) return fail(TLC_E_INVALID, what + " is a self-loop");
      keys[(size_t)k] = {((uint64_t)std::min(a, b) << 32) | (uint64_t)std::max(a, b), k};
    }
  std::sort(keys.begin(), keys.end());
  int64_t dup = -1, first = -1;
  for (size_t i = 1; i < keys.size(); i++)
    if (keys[i].first == keys[i - 1].first && (dup < 0 || keys[i].second < dup)) {  // the earliest repetition
      dup = keys[i].second;
      first = keys[i - 1].second;
    }
  if (dup >= 0) {
    const int64_t t = std::upper_bound(eoff, eoff + D + 1, dup) - eoff - 1;
    return fail(TLC_E_INVALID, "edge " + std::to_string(dup) + " (" + std::to_string(ea[dup]) + ", " +
                                   std::to_string(eb[dup]) + ") of graph " + std::to_string(t) + " repeats edge " +
                                   std::to_string(first));
  }
  return TLC_OK;
}

static GraphBatchView batch_view(const tlc_graph_batch* b, const double* f, uint32_t flags, uint8_t* status) {
  GraphBatchView v{};
  v.D = b->D;
  v.noff = b->noff.as<int64_t>(); v.eoff = b->eoff.as<int64_t>(); v.soff = b->soff.as<int64_t>();
  v.ea = b->ea.as<int32_t>(); v.eb = b->eb.as<int32_t>();
  v.f = f;
  v.flags = flags;
  v.stage = DiagArea{b->kind.as<uint8_t>(), b->bv.as<int32_t>(), b->dv.as<int32_t>(), b->birth.as<double>(),
                     b->death.as<double>()};
  v.np = b->np.as<int32_t>();
  v.status = status;
  return v;
}

// the structure's device side; *b owns every allocation as soon as it exists
static int graph_batch_upload(tlc_graph_batch* b, const int64_t* noff, const int64_t* eoff, const int32_t* ea,
                              const int32_t* eb) {
  const int64_t D = b->D, N = b->N, M = b->M, P = b->bound();
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, b->device));
  b->sm_count = prop.multiProcessorCount;
  std::vector<int64_t> soff((size_t)D);
  std::vector<int32_t> lists[3];
  std::vector<int64_t> l_tidx, l_voff{0}, l_eoff{0};
  for (int64_t t = 0; t < D; t++) {
    const int64_t n = noff[t + 1] - noff[t], m = eoff[t + 1] - eoff[t];
    soff[(size_t)t] = noff[t] + eoff[t] + t;
    b->all.n_max = std::max(b->all.n_max, n); b->all.m_max = std::max(b->all.m_max, m);
    const int r = graph_route(n, m);
    if (r < 3) { lists[r].push_back((int32_t)t); continue; }
    l_tidx.push_back(t); l_voff.push_back(l_voff.back() + n); l_eoff.push_back(l_eoff.back() + m);
    b->large.n_max = std::max(b->large.n_max, n); b->large.m_max = std::max(b->large.m_max, m);
  }
  const int64_t DL = (int64_t)l_tidx.size();
  auto up = [&](DevBuf& buf, const void* src, size_t bytes) -> cudaError_t {
    cudaError_t e = buf.reserve(bytes);
    if (e == cudaSuccess && bytes) e = cudaMemcpy(buf.p, src, bytes, cudaMemcpyDefault);  // (host or device sources)
    return e;
  };
  CK(up(b->noff, noff, (size_t)(D + 1) * 8));
  CK(up(b->eoff, eoff, (size_t)(D + 1) * 8));
  CK(up(b->soff, soff.data(), (size_t)D * 8));
  CK(up(b->ea, ea, (size_t)M * 4));
  CK(up(b->eb, eb, (size_t)M * 4));
  std::vector<int32_t> all_lists;
  for (int c = 0; c < 3; c++) { b->counts[c] = (int)lists[c].size(); all_lists.insert(all_lists.end(), lists[c].begin(), lists[c].end()); }
  CK(up(b->lists, all_lists.data(), all_lists.size() * 4));
  CK(b->kind.reserve((size_t)P));
  CK(b->bv.reserve((size_t)P * 4)); CK(b->dv.reserve((size_t)P * 4));
  CK(b->birth.reserve((size_t)P * 8)); CK(b->death.reserve((size_t)P * 8));
  CK(b->np.reserve((size_t)D * 4)); CK(b->status.reserve((size_t)D));
  CK(b->gcnt.reserve((size_t)N * 4)); CK(b->glst.reserve((size_t)P * 8));
  // staged views: `all` needs the larger arena; `large` is carved from the same bytes (the two never run in one call)
  CK(b->arena.reserve(chunk_bytes(D, N, M, 0)));
  b->all.c = carve(b->arena.as<char>(), D, N, M, 0, nullptr);
  b->large.c = carve(b->arena.as<char>(), DL, l_voff.back(), l_eoff.back(), 0, nullptr);
  // their per-graph tables: all (tidx, voff, eoff), large (tidx, voff, eoff)
  std::vector<int64_t> tab;
  for (int64_t t = 0; t < D; t++) tab.push_back(t);
  tab.insert(tab.end(), noff, noff + D + 1);
  tab.insert(tab.end(), eoff, eoff + D + 1);
  tab.insert(tab.end(), l_tidx.begin(), l_tidx.end());
  tab.insert(tab.end(), l_voff.begin(), l_voff.end());
  tab.insert(tab.end(), l_eoff.begin(), l_eoff.end());
  CK(up(b->tables, tab.data(), tab.size() * 8));
  const int64_t* d_tab = b->tables.as<int64_t>();
  b->all.c.tidx = d_tab; b->all.c.voff = d_tab + D; b->all.c.eoff = d_tab + 2 * D + 1;
  const int64_t* d_l = d_tab + 3 * D + 2;
  b->large.c.tidx = d_l; b->large.c.voff = d_l + DL; b->large.c.eoff = d_l + 2 * DL + 1;
  return TLC_OK;
}

// kernels 2 + 3 (+ 3b) over one staged view, between the fill and the export
static void run_graph_staged(const tlc_graph_batch* b, const GraphBatchView& v, const StagedView& s, uint32_t flags,
                             cudaStream_t st) {
  const ChunkView& c = s.c;
  if (c.T <= 0) return;
  launch_graph_fill(v, c, b->sm_count, st);
  const Params p{0, TLC_MODE_NODE, TLC_DESC_SUM, 5, flags, 0};
  const bool ext = (flags & TLC_F_EXTENDED) != 0;
  const int mask = (flags & TLC_F_ASC_ONLY) ? 1 : 3;
  const int block = block_for(s.m_max);
  launch_sort(p, c, block, mask, 0, st);
  const int64_t uf_ints = 2 * s.n_max * 4 <= 96 * 1024 ? 2 * s.n_max : 0;
  launch_union_find(p, c, block, (int)uf_ints, ext ? 1 : 0, mask, 0, st);
  if (ext) {
    const int64_t lp_ints = 3 * s.n_max * 4 <= 200 * 1024 ? 3 * s.n_max : 0;
    launch_loops(p, c, std::min(block, 128), (int)lp_ints, s.n_max, st);
  }
  launch_graph_export(v, c, b->sm_count, st);
}

extern "C" {

int tlc_graph_batch_create(int device, int64_t D, const int64_t* noff, const int64_t* eoff, const int32_t* ea,
                           const int32_t* eb, tlc_graph_batch** out) {
  if (!out) return fail(TLC_E_INVALID, "out is NULL");
  int rc = check_graph_batch(D, noff, eoff, ea, eb);
  if (rc || (rc = select_device(device))) return rc;
  tlc_graph_batch* b = new tlc_graph_batch();
  b->device = device;
  b->D = D; b->N = noff[D]; b->M = eoff[D];
  rc = graph_batch_upload(b, noff, eoff, ea, eb);
  if (rc != TLC_OK) { delete b; return rc; }
  *out = b;
  return TLC_OK;
}

int tlc_graph_batch_create_dev(int device, int64_t D, const int64_t* dev_noff, const int64_t* dev_eoff,
                               const int32_t* dev_ea, const int32_t* dev_eb, void* stream, tlc_graph_batch** out) {
  if (!out) return fail(TLC_E_INVALID, "out is NULL");
  if (D < 0 || D >= ((int64_t)1 << 31)) return fail(TLC_E_INVALID, "D must be in [0, 2^31)");
  if (!dev_noff || !dev_eoff) return fail(TLC_E_INVALID, "noff and eoff are required");
  int rc = select_device(device);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<int64_t> noff((size_t)D + 1), eoff((size_t)D + 1);
  CK(cudaMemcpyAsync(noff.data(), dev_noff, (size_t)(D + 1) * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(eoff.data(), dev_eoff, (size_t)(D + 1) * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if ((rc = check_batch_offsets(D, noff.data(), eoff.data()))) return rc;
  const int64_t M = eoff[(size_t)D];
  if (M > 0 && (!dev_ea || !dev_eb)) return fail(TLC_E_INVALID, "ea and eb are required when there are edges");
  if (M > 0) {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    DevBuf first;
    CK(first.reserve(8));
    unsigned long long h_first = 0;
    CK(cudaMemsetAsync(first.p, 0xff, 8, st));
    launch_batch_check(D, M, dev_noff, dev_eoff, dev_ea, dev_eb, first.as<unsigned long long>(), prop.multiProcessorCount, st);
    CK(cudaMemcpyAsync(&h_first, first.p, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (h_first != ~0ull) {  // the message of tlc_graph_batch_create for the first offending edge
      const int64_t k = (int64_t)(h_first >> 2);
      const int reason = (int)(h_first & 3);
      int32_t e[4] = {0, 0, 0, 0};  // ea / eb of edges k - 1 and k
      const int64_t k0 = k > 0 ? k - 1 : k;
      CK(cudaMemcpy(e, dev_ea + k0, (size_t)(k - k0 + 1) * 4, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(e + 2, dev_eb + k0, (size_t)(k - k0 + 1) * 4, cudaMemcpyDeviceToHost));
      const int64_t a = e[k - k0], bb = e[2 + k - k0];
      const int64_t t = std::upper_bound(eoff.begin(), eoff.end(), k) - eoff.begin() - 1;
      const std::string what = "edge " + std::to_string(k) + " (" + std::to_string(a) + ", " + std::to_string(bb) +
                               ") of graph " + std::to_string(t);
      if (reason == BATCH_BAD_RANGE)
        return fail(TLC_E_INVALID, what + " has an endpoint outside the graph's vertices [" + std::to_string(noff[(size_t)t]) +
                                       ", " + std::to_string(noff[(size_t)t + 1]) + ")");
      if (reason == BATCH_BAD_LOOP) return fail(TLC_E_INVALID, what + " is a self-loop");
      if (reason == BATCH_BAD_ORIENT) return fail(TLC_E_INVALID, what + " has ea > eb (canonical form needs ea < eb)");
      if (e[0] == a && e[2] == bb) return fail(TLC_E_INVALID, what + " repeats edge " + std::to_string(k - 1));
      return fail(TLC_E_INVALID, what + " is not after edge " + std::to_string(k - 1) + " (" + std::to_string(e[0]) + ", " +
                                     std::to_string(e[2]) + "): canonical form needs the edges strictly ascending in (ea, eb)");
    }
  }
  tlc_graph_batch* b = new tlc_graph_batch();
  b->device = device;
  b->D = D; b->N = noff[(size_t)D]; b->M = M;
  rc = graph_batch_upload(b, noff.data(), eoff.data(), dev_ea, dev_eb);
  if (rc != TLC_OK) { delete b; return rc; }
  *out = b;
  return TLC_OK;
}

int tlc_graph_batch_destroy(tlc_graph_batch* b) {
  if (!b) return TLC_OK;
  cudaSetDevice(b->device);
  delete b;
  return TLC_OK;
}

int tlc_graph_batch_pair_bound(const tlc_graph_batch* b, int64_t* bound) {
  if (!b || !bound) return fail(TLC_E_INVALID, "NULL argument");
  *bound = b->bound();
  return TLC_OK;
}

int tlc_graph_batch_diagrams_dev(tlc_graph_batch* b, const double* dev_f, uint32_t flags, tlc_diagrams* out,
                                 uint8_t* dev_status, void* stream) {
  if (flags & ~GRAPH_BATCH_FLAGS)
    return fail(TLC_E_INVALID, "flags may only hold TLC_F_EXTENDED, TLC_F_KEEP_ZERO, TLC_F_ASC_ONLY and TLC_F_NO_SMALL");
  if ((flags & TLC_F_ASC_ONLY) && (flags & TLC_F_EXTENDED))
    return fail(TLC_E_INVALID, "TLC_F_ASC_ONLY excludes TLC_F_EXTENDED (the loops need the descending sweep)");
  if (!out || !out->poff) return fail(TLC_E_INVALID, "out and out->poff are required");
  if (!b) return fail(TLC_E_INVALID, "batch is NULL");
  if (b->N > 0 && !dev_f) return fail(TLC_E_INVALID, "dev_f is NULL");
  if (out->cap < b->bound())
    return fail(TLC_E_CAPACITY, "out->cap is " + std::to_string(out->cap) + ", the batch's pair bound is " +
                                    std::to_string(b->bound()));
  CK(cudaSetDevice(b->device));
  cudaStream_t st = (cudaStream_t)stream;
  const GraphBatchView v = batch_view(b, dev_f, flags, dev_status ? dev_status : b->status.as<uint8_t>());
  if (flags & TLC_F_NO_SMALL) {
    run_graph_staged(b, v, b->all, flags, st);
  } else {
    const int32_t* l = b->lists.as<int32_t>();
    const int32_t* const lists[3] = {l, l + b->counts[0], l + b->counts[0] + b->counts[1]};
    launch_graph_pd_small(v, lists, b->counts, st);
    run_graph_staged(b, v, b->large, flags, st);
  }
  launch_scan_counts(v.np, b->D, out->poff, st);
  const DiagArea dst{out->kind, out->bv, out->dv, out->birth, out->death};
  launch_gather_pairs(v.np, v.soff, out->poff, b->D, v.stage, v.stage, INT64_MAX, dst, b->sm_count, st);
  if (out->npairs && b->D > 0) CK(cudaMemcpyAsync(out->npairs, v.np, (size_t)b->D * 4, cudaMemcpyDeviceToDevice, st));
  CK(cudaGetLastError());
  return TLC_OK;
}

int tlc_graph_batch_grad_dev(tlc_graph_batch* b, const tlc_diagrams* d, const double* dev_grad_birth,
                             const double* dev_grad_death, double* dev_grad_f, void* stream) {
  if (!d || !d->poff || !d->bv || !d->dv) return fail(TLC_E_INVALID, "d, d->poff, d->bv and d->dv are required");
  if (!b) return fail(TLC_E_INVALID, "batch is NULL");
  if (b->N > 0 && !dev_grad_f) return fail(TLC_E_INVALID, "dev_grad_f is NULL");
  if (b->D == 0) return TLC_OK;
  CK(cudaSetDevice(b->device));
  const GraphBatchView v = batch_view(b, nullptr, 0, nullptr);
  launch_graph_grad(v, d->poff, d->bv, d->dv, dev_grad_birth, dev_grad_death, b->gcnt.as<int32_t>(),
                    b->glst.as<int32_t>(), dev_grad_f, b->sm_count, (cudaStream_t)stream);
  CK(cudaGetLastError());
  return TLC_OK;
}

}  // extern "C"
