// engine.cu — C ABI (include/bsched.h) of the B200 gang-scheduling feasibility engine.
//
// Host side: table validation + upload, class de-duplication of the pre-encoded
// selector/toleration masks, kernel sequencing on one CUDA stream (the queue sort
// runs concurrently on a second stream), result fetch, and the per-call mirrors of
// batchSchedulingPlugin.PreFilter / Permit / Less (batchscheduler.go:102,165,214).
// There is no CPU implementation of the path here: no device -> BS_E_NODEVICE.
#include <cuda_runtime.h>

#include <omp.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <chrono>
#include <sched.h>
#include <vector>

#include "kernels.cuh"
#include "fit.cuh"
#include "gang_state.hpp"
#include "sort.cuh"
#include "replay.cuh"

using namespace bsk;

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool owned = true;    // false: a view into an arena (alias), never freed here
  void alias(void* ptr, size_t bytes) { p = ptr; cap = bytes; owned = false; }
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p && owned) cudaFree(p);
    owned = true;
    p = nullptr;
    cap = 0;
    const size_t want = std::max<size_t>(bytes, 256);
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p && owned) cudaFree(p);
    p = nullptr;
    cap = 0;
    owned = true;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool owned = true;
  void alias(void* ptr, size_t bytes) { p = ptr; cap = bytes; owned = false; }
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p && owned) cudaFreeHost(p);
    owned = true;
    p = nullptr;
    cap = 0;
    const size_t want = std::max<size_t>(bytes, 256);
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p && owned) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    owned = true;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

// a resizable array in pinned host memory: what is DMA'd every round must not be staged through
// pageable memory
template <class T>
struct PinVec {
  PinBuf buf;
  size_t n = 0;
  bool resize(size_t count) {
    if (buf.ensure(std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) return false;
    n = count;
    return true;
  }
  T* data() const { return buf.as<T>(); }
  T& operator[](size_t i) const { return buf.as<T>()[i]; }
  size_t size() const { return n; }
  void release() { buf.release(); n = 0; }
};

// (sel, tol, non-zero scalar request mask): the pre-encoded predicates a pod class shares
struct ClassKey {
  uint64_t sel, tol;
  uint32_t nz;
  uint32_t aff;   // affinity class (row of the bs_upload_affinity table) or BS_AFF_NONE
  bool operator==(const ClassKey& o) const { return sel == o.sel && tol == o.tol && nz == o.nz && aff == o.aff; }
};

// flat open-addressing index ClassKey -> dense id (insertion order)
struct ClassIndex {
  std::vector<ClassKey> keys;
  std::vector<uint32_t> slots;  // id + 1, 0 = empty
  uint32_t mask = 0;
  ClassKey last_key{0, 0, 0xffffffffu, 0};
  uint32_t last_id = 0;
  static uint64_t hash(const ClassKey& k) {
    uint64_t h = k.sel * 0x9E3779B97F4A7C15ull ^ (k.tol + 0x7F4A7C15ull) * 0xBF58476D1CE4E5B9ull ^
                 ((uint64_t)k.nz | ((uint64_t)k.aff << 32)) * 0x94D049BB133111EBull;
    return h ^ (h >> 29);
  }
  void clear() {
    keys.clear();
    slots.assign(256, 0);
    mask = 255;
    last_key = ClassKey{0, 0, 0xffffffffu, 0};
  }
  void grow() {
    std::vector<uint32_t> ns((size_t)(mask + 1) * 2, 0);
    const uint32_t nm = (uint32_t)ns.size() - 1;
    for (uint32_t id = 0; id < keys.size(); ++id) {
      uint32_t s = (uint32_t)hash(keys[id]) & nm;
      while (ns[s]) s = (s + 1) & nm;
      ns[s] = id + 1;
    }
    slots.swap(ns);
    mask = nm;
  }
  uint32_t get_or_add(const ClassKey& k) {
    if (k == last_key) return last_id;
    if (slots.empty()) clear();
    uint32_t s = (uint32_t)hash(k) & mask;
    while (slots[s]) {
      if (keys[slots[s] - 1] == k) {
        last_key = k;
        last_id = slots[s] - 1;
        return last_id;
      }
      s = (s + 1) & mask;
    }
    const uint32_t id = (uint32_t)keys.size();
    keys.push_back(k);
    slots[s] = id + 1;
    if (keys.size() * 2 > slots.size()) grow();
    last_key = k;
    last_id = id;
    return id;
  }
  size_t size() const { return keys.size(); }
};

// Threads for the host packing passes.  Not taken from OMP_NUM_THREADS (launchers such as torchrun
// pin it to 1): BS_HOST_THREADS if set, else the cores divided by the GPUs of the box, at most 8.
inline int host_threads() {
  static int n = [] {
    if (const char* s = getenv("BS_HOST_THREADS")) return std::max(1, atoi(s));
    int ndev = 1;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) ndev = 1;
    int hw = (int)std::thread::hardware_concurrency();
    cpu_set_t set;   // cores this process may actually run on (cgroup / taskset), not the box's total
    if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) hw = std::min(hw > 0 ? hw : 1 << 20, CPU_COUNT(&set));
    return std::max(1, std::min(8, hw / ndev));
  }();
  return n;
}

// out[i] = id of key_of(i) in `global` (ids stable across calls: the index only grows).
// Two parallel passes: thread-local indices, a small sequential merge, then a remap.
template <class KeyFn>
void assign_classes(ClassIndex& global, uint32_t n, KeyFn key_of, uint32_t* out) {
  if (global.slots.empty()) global.clear();
  const int T = n < 8192 ? 1 : host_threads();
  // T fixed CHUNKS, not T threads: num_threads(T) is only a request (OMP_THREAD_LIMIT, OMP_DYNAMIC, a failed
  // thread creation give a smaller team), so the chunks are shared out with an omp for
  std::vector<ClassIndex> local(T);
  std::vector<std::vector<uint32_t>> remap(T);
  const uint32_t chunk = (n + T - 1) / T;
#pragma omp parallel for schedule(static, 1) num_threads(T)
  for (int t = 0; t < T; ++t) {
    ClassIndex& li = local[t];
    li.clear();
    const uint32_t a = std::min(n, (uint32_t)t * chunk), b = std::min(n, a + chunk);
    for (uint32_t i = a; i < b; ++i) out[i] = li.get_or_add(key_of(i));
  }
  for (int t = 0; t < T; ++t) {
    remap[t].resize(local[t].size());
    for (size_t j = 0; j < local[t].size(); ++j) remap[t][j] = global.get_or_add(local[t].keys[j]);
  }
#pragma omp parallel for schedule(static, 1) num_threads(T)
  for (int t = 0; t < T; ++t) {
    const uint32_t a = std::min(n, (uint32_t)t * chunk), b = std::min(n, a + chunk);
    const uint32_t* rm = remap[t].data();
    for (uint32_t i = a; i < b; ++i) out[i] = rm[out[i]];
  }
}

}  // namespace

struct bs_engine {
  std::mutex mu;
  int device = 0;
  uint32_t L = 0, out_flags = 0;
  cudaStream_t s = nullptr, s2 = nullptr, s3 = nullptr, s4 = nullptr;   // main; queue sort; PreFilter chain (high priority); peer wait
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_pre = nullptr, ev_push = nullptr, ev_gath = nullptr;
  std::string err;
  uint64_t launches = 0;

  // shapes
  uint32_t N = 0, Npad = 0, W = 0, P = 0, G = 0;
  bool have_nodes = false, have_pods = false, have_groups = false;
  bool nodes_dirty = true, classes_dirty = true, evaluated = false;

  // node table (device, padded to Npad) + derived
  DevBuf d_alloc, d_requested, d_pod_count, d_apres, d_rpres, d_label, d_taint, d_nflags;
  DevBuf d_left_w, d_left_n, d_left_present, d_classfit, d_left_plain, d_filter_bitmap, d_filter_code;
  LaneMap lane_map{};
  bool lane_map_valid = false;
  // per-lane maxima of |value| (lane classification wide / narrow)
  int64_t max_alloc[BS_MAX_LANES] = {}, max_requested[BS_MAX_LANES] = {}, max_req[BS_MAX_LANES] = {};
  int64_t max_pod_count = 0;
  int64_t neg_req[BS_MAX_LANES] = {};   // largest negative request per lane (0 when none)
  // scaled-lane classification: OR of every residual (percent 1.0) / request value of a lane (its
  // trailing zeros = the power of two every value is a multiple of) and max |residual|
  uint64_t or_left[BS_MAX_LANES] = {}, or_req[BS_MAX_LANES] = {};
  int64_t max_left[BS_MAX_LANES] = {};
  uint32_t score_pitch = 0;             // elements per score row: N rounded up to even
  uint32_t bitmap_pitch = 0;            // words per fit-bitmap row: ceil(N/32) rounded up to 32 (whole 128-byte lines)
  // pod table
  DevBuf d_req, d_ppres, d_gid, d_prio, d_ts, d_pflags, d_pod_fit_class, d_pod_rep_class;
  // group table
  DevBuf d_min_member, d_scheduled, d_matched, d_gflags, d_min_res, d_mrpres, d_creation, d_name_rank,
      d_group_rep_class;
  // class tables
  DevBuf d_fsel, d_ftol, d_fnz, d_faff, d_rsel, d_rtol, d_raff;
  // affinity bit table (bs_upload_affinity): [n_aff][W] host-evaluated node predicates
  DevBuf d_aff_bits;
  uint32_t n_aff = 0;
  std::vector<uint32_t> h_gaff;   // affinity class of each group's representative pod
  // gang state (SURVEY 8(f) row 3): the reference's TTL tables around Permit, see gang_state.hpp
  GangState gang;
  std::vector<uint32_t> h_min_member, h_scheduled, h_matched_up;   // group columns as uploaded
  std::vector<uint8_t> h_gflags_up;
  std::vector<uint64_t> h_pod_uid, h_pod_name;                     // bs_set_pod_ids
  int64_t cycle_now_ns = 0;
  bool gang_applied = false;     // the round's new_denied have been added to the deny table
  uint32_t n_fit_classes = 0, n_rep_classes = 0;
  // effective group state + round scratch
  DevBuf d_eflags, d_emin_res, d_emrpres, d_erep_class, d_first_pod, d_in_round, d_contrib, d_done, d_okA;
  DevBuf d_state, d_pre, d_pre_present, d_pre_stats, d_max_partial, d_pre_part, d_pre_part_pres, d_pre_cstats, d_pre_done;
  uint32_t prefix_slots = 0;
  // outputs
  DevBuf u_buf[9];        // bs_update_nodes / bs_update_groups: device scratch of the changed rows
  DevBuf d_best_packed;   // gang_fit tail pieces: max((score + 1) << 32 | ~node) per pod
  DevBuf d_prefilter, d_feasible, d_best_node, d_best_score, d_admit, d_admit_bitmap, d_new_denied,
      d_fit_bitmap, d_score, d_order, d_rank;
  // sort scratch
  DevBuf d_gk0, d_gk1, d_pk0, d_pk1, d_idx_a, d_idx_b, d_ghist, d_skip, d_group_rank, d_gorder, d_tilecnt,
      d_sort_barrier;
  uint32_t sort_max_grid = 1;
  int sort_variant = 0;           // 0: by the estimated fit time; 1 / 2: force the lean / wide sort kernel
  DevBuf d_sort_arena;            // the sort scratch buffers above are views into it
  size_t sort_arena_bytes = 0;
  size_t l2_persist_bytes = 0, l2_window_max = 0;   // persisting-L2 set-aside for the sort scratch (0 = off)

  // host copies for the per-call mirrors and class building
  std::vector<int32_t> h_gid, h_prio;
  std::vector<uint8_t> h_pflags;
  std::vector<uint64_t> h_gsel, h_gtol;
  std::vector<uint8_t> h_nflags;
  // class indices (host packing): fit classes (sel, tol, nz) of the pods; representative classes
  // (sel, tol) of pods and carried-in group representatives
  ClassIndex fit_index, rep_index;
  PinVec<uint32_t> h_pfc, h_prc, h_grc;   // pinned: DMA'd whenever the classes change
  cudaEvent_t ev_classes = nullptr;       // the last class-table DMA out of them
  bool group_classes_dirty = true;   // every group's representative id has to be looked up again
  bool group_ids_dirty = false;      // some ids in h_grc changed in place (bs_update_groups): DMA them again
  std::vector<int64_t> h_wait_ns;
  int64_t default_wait_ns = 0;
  // bits that differ between rows of each sort key word (a constant byte needs no radix pass)
  bool any_lister_miss = true;
  int32_t max_gid = -1;
  uint64_t vary_ts = ~0ull, vary_prio = ~0ull, vary_creation = ~0ull, vary_name = ~0ull;
  uint64_t g_or1 = 0, g_and1 = ~0ull, g_or0 = 0, g_and0 = ~0ull;   // OR / AND of the group key words seen so far
  bool pod_classes_dirty = true;
  double last_classes_us = 0;
  // BS_HOST_PROFILE: host-side segment times (label, us) since the last bs_evaluate, printed there
  bool host_prof = false;
  std::vector<std::pair<const char*, double>> hp_log;
  std::chrono::steady_clock::time_point hp_t;
  // pinned result cache
  PinBuf h_prefilter, h_feasible, h_best_node, h_best_score, h_admit, h_admit_bitmap, h_new_denied,
      h_order, h_rank, h_state, h_filter_code;
  bool fetched = false;
  // decision arena: every per-round decision vector lives in ONE device block and ONE pinned block with the
  // same layout (the d_* / h_* buffers above are views into them), so bs_fetch is a single D2H copy
  DevBuf d_arena;
  PinBuf h_arena;
  size_t arena_bytes = 0;

  // bs_replay scratch (kept between calls: cudaMalloc/cudaFree per call would dominate small queues)
  DevBuf r_req, r_pc, r_rp, r_matched, r_gflags, r_grc, r_minres, r_mrp, r_queue, r_pf, r_node, r_ready, r_status,
      r_sum, r_max, r_keys, r_left0, r_left1, r_both, r_fit, r_stat;

  // peer exchange (admit bitmap all-gather over NVLink peer memory)
  DevBuf d_gather, d_peer_err;
  uint32_t peer_rank = 0, peer_world = 0, peer_wpr = 0, peer_seq = 0;
  bool peer_attached = false;
  bool peer_broken = false;          // a wait timed out: every later round fails fast until detach + re-attach
  unsigned long long peer_timeout_ns = 2000000000ull;
  void* peer_ptr[PEER_MAX_WORLD] = {};

  // profiling
  bool profiling = false;
  cudaEvent_t ev_a[BS_K_COUNT] = {}, ev_b[BS_K_COUNT] = {};
  uint32_t k_launches[BS_K_COUNT] = {};
  bool k_valid[BS_K_COUNT] = {};
};

namespace {

#define CK(call)                                                                     \
  do {                                                                               \
    cudaError_t _e = (call);                                                         \
    if (_e != cudaSuccess) {                                                         \
      e->err = std::string(#call) + ": " + cudaGetErrorString(_e);                   \
      cudaGetLastError();                                                            \
      return _e == cudaErrorMemoryAllocation ? BS_E_NOMEM : BS_E_CUDA;               \
    }                                                                                \
  } while (0)

int fail(bs_engine* e, int code, const char* msg) {
  e->err = msg;
  return code;
}

// per-lane max |value| of a [L][n] table; false if any value is outside +-BS_VALUE_LIMIT
bool lane_maxima(const int64_t* a, uint32_t L, size_t n, int64_t* out) {
  bool ok = true;
  for (uint32_t d = 0; d < L; ++d) {
    const int64_t* row = a + (size_t)d * n;
    int64_t lo = 0, hi = 0;
#pragma omp parallel for reduction(min : lo) reduction(max : hi) if (n > 65536) num_threads(host_threads())
    for (size_t i = 0; i < n; ++i) {
      lo = std::min(lo, row[i]);
      hi = std::max(hi, row[i]);
    }
    ok = ok && lo >= -BS_VALUE_LIMIT && hi <= BS_VALUE_LIMIT;
    out[d] = std::max(hi, lo == INT64_MIN ? INT64_MAX : -lo);
  }
  return ok;
}

// Host restatement of singleNodeResource's per-lane residual at percent 1.0 (core.go:647-668) for the
// lane statistics only: OR of the values (common power-of-two factor) and max |value| per lane.
// (float)alloc is the RN convert, * 1.0f is exact, the cast back truncates — the device's scale_f32.
void left_stats(const bs_node_table* t, uint32_t L, uint32_t n, uint64_t* or_out, int64_t* max_out) {
  for (uint32_t d = 0; d < L; ++d) {
    uint64_t o = 0;
    int64_t mx = 0;
    const int64_t* al = t->alloc + (size_t)d * n;
    const int64_t* rq = t->requested + (size_t)d * n;
    for (uint32_t i = 0; i < n; ++i) {
      if (d >= 4 && !((t->alloc_present[i] & t->req_present[i]) >> d & 1u)) continue;   // key absent: sentinel
      int64_t used = rq[i];
      if (d == (uint32_t)LANE_PODS && used == 0) used = t->pod_count[i];
      const int64_t v = (int64_t)((float)al[i] * 1.0f) - used;
      o |= (uint64_t)v;
      mx = std::max(mx, v < 0 ? -v : v);
    }
    or_out[d] |= o;
    max_out[d] = std::max(max_out[d], mx);
  }
}

// Everything bs_upload_nodes needs from the host columns in ONE chunked pass (an omp team for big tables):
// |value| maxima of alloc / requested (range check + lane classification), max |pod_count| and the
// residual statistics of left_stats.
struct NodeHostStats {
  int64_t mx_a[BS_MAX_LANES] = {}, mx_r[BS_MAX_LANES] = {}, mx_l[BS_MAX_LANES] = {};
  uint64_t or_l[BS_MAX_LANES] = {};
  int64_t mx_pc = 0;
  bool ok = true;
};
NodeHostStats node_host_pass(const bs_node_table* t, uint32_t L, uint32_t N) {
  const int T = N < 4096 ? 1 : host_threads();
  std::vector<NodeHostStats> part(T);
  const uint32_t chunk = (N + T - 1) / std::max(T, 1);
#pragma omp parallel for schedule(static, 1) num_threads(T) if (T > 1)
  for (int tk = 0; tk < T; ++tk) {
    NodeHostStats st;
    const uint32_t a0 = std::min(N, (uint32_t)tk * chunk), a1 = std::min(N, a0 + chunk);
    for (uint32_t d = 0; d < L; ++d) {
      const int64_t* al = t->alloc + (size_t)d * N;
      const int64_t* rq = t->requested + (size_t)d * N;
      int64_t alo = 0, ahi = 0, rlo = 0, rhi = 0, mx = 0;
      uint64_t o = 0;
      for (uint32_t i = a0; i < a1; ++i) {
        alo = std::min(alo, al[i]); ahi = std::max(ahi, al[i]);
        rlo = std::min(rlo, rq[i]); rhi = std::max(rhi, rq[i]);
      }
      for (uint32_t i = a0; i < a1; ++i) {   // left_stats' body
        if (d >= 4 && !((t->alloc_present[i] & t->req_present[i]) >> d & 1u)) continue;
        int64_t used = rq[i];
        if (d == (uint32_t)LANE_PODS && used == 0) used = t->pod_count[i];
        const int64_t v = (int64_t)((float)al[i] * 1.0f) - used;
        o |= (uint64_t)v;
        mx = std::max(mx, v < 0 ? -v : v);
      }
      st.ok = st.ok && alo >= -BS_VALUE_LIMIT && ahi <= BS_VALUE_LIMIT && rlo >= -BS_VALUE_LIMIT && rhi <= BS_VALUE_LIMIT;
      st.mx_a[d] = std::max(ahi, alo == INT64_MIN ? INT64_MAX : -alo);
      st.mx_r[d] = std::max(rhi, rlo == INT64_MIN ? INT64_MAX : -rlo);
      st.or_l[d] = o;
      st.mx_l[d] = mx;
    }
    int64_t pc = 0;
    for (uint32_t i = a0; i < a1; ++i) pc = std::max<int64_t>(pc, std::abs((int64_t)t->pod_count[i]));
    st.mx_pc = pc;
    part[tk] = st;
  }
  NodeHostStats r;
  for (int tk = 0; tk < T; ++tk) {
    r.ok = r.ok && part[tk].ok;
    r.mx_pc = std::max(r.mx_pc, part[tk].mx_pc);
    for (uint32_t d = 0; d < L; ++d) {
      r.mx_a[d] = std::max(r.mx_a[d], part[tk].mx_a[d]);
      r.mx_r[d] = std::max(r.mx_r[d], part[tk].mx_r[d]);
      r.mx_l[d] = std::max(r.mx_l[d], part[tk].mx_l[d]);
      r.or_l[d] |= part[tk].or_l[d];
    }
  }
  return r;
}

// Lane classification for the fit kernel (kernels.cuh "Narrow lanes"): lane d is narrow when every
// residual |left[d]| and every request |req[d]| of the round is <= 2^27.  The narrow set must
// contain a fixed lane (always a real value) and the (LW, LN) pair must be one the dispatch
// table instantiates; otherwise every lane is wide.
LaneMap classify_lanes(const bs_engine* e);

inline uint32_t cdiv(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

// upload a [L][n] lane-major host table into a [L][npad] device table
int upload_lanes(bs_engine* e, DevBuf& dst, const int64_t* src, uint32_t L, uint32_t n, uint32_t npad) {
  CK(dst.ensure((size_t)L * npad * 8));
  if (npad != n) CK(cudaMemsetAsync(dst.p, 0, (size_t)L * npad * 8, e->s));
  if (n)
    CK(cudaMemcpy2DAsync(dst.p, (size_t)npad * 8, src, (size_t)n * 8, (size_t)n * 8, L,
                         cudaMemcpyHostToDevice, e->s));
  return BS_OK;
}

template <class T>
int upload_vec(bs_engine* e, DevBuf& dst, const T* src, uint32_t n, uint32_t npad) {
  CK(dst.ensure((size_t)npad * sizeof(T)));
  if (npad != n) CK(cudaMemsetAsync(dst.p, 0, (size_t)npad * sizeof(T), e->s));
  if (n) CK(cudaMemcpyAsync(dst.p, src, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, e->s));
  return BS_OK;
}

NodeTab node_tab(const bs_engine* e) {
  NodeTab t;
  t.alloc = e->d_alloc.as<int64_t>();
  t.requested = e->d_requested.as<int64_t>();
  t.pod_count = e->d_pod_count.as<int32_t>();
  t.alloc_present = e->d_apres.as<uint32_t>();
  t.req_present = e->d_rpres.as<uint32_t>();
  t.label = e->d_label.as<uint64_t>();
  t.taint = e->d_taint.as<uint64_t>();
  t.flags = e->d_nflags.as<uint8_t>();
  t.aff_bits = e->d_aff_bits.as<uint32_t>();
  t.aff_W = e->W;
  t.N = e->N;
  t.Npad = e->Npad;
  t.L = e->L;
  return t;
}
PodTab pod_tab(const bs_engine* e) {
  PodTab p;
  p.req = e->d_req.as<int64_t>();
  p.req_present = e->d_ppres.as<uint32_t>();
  p.gid = e->d_gid.as<int32_t>();
  p.flags = e->d_pflags.as<uint8_t>();
  p.fit_class = e->d_pod_fit_class.as<uint32_t>();
  p.rep_class = e->d_pod_rep_class.as<uint32_t>();
  p.P = e->P;
  p.L = e->L;
  return p;
}
GroupTab group_tab(const bs_engine* e) {
  GroupTab g;
  g.min_member = e->d_min_member.as<uint32_t>();
  g.scheduled = e->d_scheduled.as<uint32_t>();
  g.matched = e->d_matched.as<uint32_t>();
  g.flags = e->d_gflags.as<uint8_t>();
  g.min_res = e->d_min_res.as<int64_t>();
  g.min_res_present = e->d_mrpres.as<uint32_t>();
  g.rep_class = e->d_group_rep_class.as<uint32_t>();
  g.G = e->G;
  g.L = e->L;
  return g;
}
GroupEff group_eff(const bs_engine* e) {
  GroupEff x;
  x.flags = e->d_eflags.as<uint8_t>();
  x.min_res = e->d_emin_res.as<int64_t>();
  x.min_res_present = e->d_emrpres.as<uint32_t>();
  x.rep_class = e->d_erep_class.as<uint32_t>();
  x.first_pod = e->d_first_pod.as<uint32_t>();
  x.in_round = e->d_in_round.as<uint32_t>();
  x.contrib = e->d_contrib.as<uint32_t>();
  x.done = e->d_done.as<uint32_t>();
  return x;
}
PrefixOut prefix_out(const bs_engine* e) {
  PrefixOut o;
  o.pre = e->d_pre.as<int64_t>();
  o.present = e->d_pre_present.as<uint32_t>();
  o.stats = e->d_pre_stats.as<ClassStats>();
  return o;
}

PrefixScratch prefix_scratch(const bs_engine* e) {
  PrefixScratch sc;
  sc.part = e->d_pre_part.as<int64_t>();
  sc.part_pres = e->d_pre_part_pres.as<uint32_t>();
  sc.cstats = e->d_pre_cstats.as<ClassStats>();
  sc.done = e->d_pre_done.as<uint32_t>();
  return sc;
}

// Makes the engine's device current for the scope and restores the caller's device afterwards
// (the library must not leave the calling thread on a different device).
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) err = cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};
#define BS_DEVICE_GUARD(e)        \
  DeviceGuard _guard((e)->device); \
  CK(_guard.err)

// host-side segment timer (BS_HOST_PROFILE): HP_BEGIN at the top of an entry point, HP("what") after a segment
#define HP_BEGIN(e) do { if ((e)->host_prof) (e)->hp_t = std::chrono::steady_clock::now(); } while (0)
#define HP(e, label) do { if ((e)->host_prof) { const auto _n = std::chrono::steady_clock::now(); \
    if ((e)->hp_log.size() > 4096) (e)->hp_log.clear(); (e)->hp_log.emplace_back(label, std::chrono::duration<double, std::micro>(_n - (e)->hp_t).count()); (e)->hp_t = _n; } } while (0)

struct StageTimer {
  bs_engine* e;
  int k;
  cudaStream_t st;
  bool manual;   // the launcher records the two events itself (gang_fit: around the one kernel)
  StageTimer(bs_engine* e_, int k_, cudaStream_t st_, bool manual_ = false) : e(e_), k(k_), st(st_), manual(manual_) {
    e->k_launches[k] = 0;
    if (e->profiling && !manual) cudaEventRecord(e->ev_a[k], st);
  }
  ~StageTimer() {
    if (e->profiling && !manual) {
      cudaEventRecord(e->ev_b[k], st);
      e->k_valid[k] = true;
    }
  }
  void launched(uint32_t n = 1) {
    e->k_launches[k] += n;
    e->launches += n;
  }
};

inline int prefix_maxl(uint32_t L) {
  return L <= 4 ? 4 : L <= 5 ? 5 : L <= 6 ? 6 : L <= 8 ? 8 : L <= 9 ? 9 : L <= 12 ? 12 : 16;
}
template <int MAXL>
void launch_prefix_t(NodeTab t, PrefixSel ps, PrefixScratch sc, PrefixOut po, uint32_t n_classes, cudaStream_t s) {
  const uint32_t n_chunks = cdiv(t.N, PREFIX_CHUNK);
  dim3 grid(n_chunks, n_classes);
  prefix_partial_kernel<MAXL><<<grid, PREFIX_CHUNK, 0, s>>>(t, ps, sc, n_chunks);
  prefix_scan_kernel<MAXL><<<grid, PREFIX_CHUNK, 0, s>>>(t, ps, sc, n_chunks, po);
}
// two launches: chunk totals, then offsets + in-chunk scan + statistics
void launch_prefix(uint32_t L, NodeTab t, PrefixSel ps, PrefixScratch sc, PrefixOut po, uint32_t n_classes,
                   cudaStream_t s) {
  switch (prefix_maxl(L)) {
    case 4: launch_prefix_t<4>(t, ps, sc, po, n_classes, s); break;
    case 5: launch_prefix_t<5>(t, ps, sc, po, n_classes, s); break;
    case 6: launch_prefix_t<6>(t, ps, sc, po, n_classes, s); break;
    case 8: launch_prefix_t<8>(t, ps, sc, po, n_classes, s); break;
    case 9: launch_prefix_t<9>(t, ps, sc, po, n_classes, s); break;
    case 12: launch_prefix_t<12>(t, ps, sc, po, n_classes, s); break;
    default: launch_prefix_t<16>(t, ps, sc, po, n_classes, s); break;
  }
}

template <int MAXL>
void launch_replay_t(const ReplayArgs& a, cudaStream_t s) { replay_kernel<MAXL><<<1, REPLAY_THREADS, 0, s>>>(a); }
inline uint32_t replay_maxl(uint32_t L) { return L <= 5 ? 5u : L <= 9 ? 9u : 16u; }
void launch_replay(uint32_t L, const ReplayArgs& a, cudaStream_t s) {
  switch (replay_maxl(L)) {
    case 5: launch_replay_t<5>(a, s); break;
    case 9: launch_replay_t<9>(a, s); break;
    default: launch_replay_t<16>(a, s); break;
  }
}

cudaError_t launch_fit(const FitArgs& a, uint32_t units, cudaStream_t s, uint32_t* launches, cudaEvent_t ev_a, cudaEvent_t ev_b) {
  const int out = a.score ? FIT_OUT_SCORE : (a.fit_bitmap ? FIT_OUT_BITMAP : FIT_OUT_NONE);
  FitFn fn = fit_lookup(a.lm.LW, a.lm.LN, a.lm.LS, out);
  return fn ? fn(a, units, s, launches, ev_a, ev_b) : cudaErrorInvalidValue;
}

inline uint32_t ctz64(uint64_t v) { return v ? (uint32_t)__builtin_ctzll(v) : 63u; }

LaneMap classify_lanes(const bs_engine* e) {
  LaneMap lm{};
  const uint32_t L = e->L;
  enum { WIDE = 0, NARROW = 1, SCALED = 2 };
  int kind[BS_MAX_LANES];
  uint32_t unit[BS_MAX_LANES] = {};
  bool fixed_narrow = false;
  uint32_t ln = 0, ls = 0;
  for (uint32_t d = 0; d < L; ++d) {
    // |left| <= |scale(alloc)| + |requested| (pods lane: + len(Pods())); float32 rounding of a
    // value <= 2^26 is exact, so the bound 2^26 + 2^26 = 2^27 holds.
    int64_t used = e->max_requested[d];
    if (d == LANE_PODS) used = std::max(used, e->max_pod_count);
    const bool narrow = e->max_alloc[d] <= (NARROW_LIMIT >> 1) && used <= (NARROW_LIMIT >> 1) && e->max_req[d] <= NARROW_LIMIT;
    kind[d] = narrow ? NARROW : WIDE;
    if (narrow) {
      ++ln;
      if (d < 4) fixed_narrow = true;
      continue;
    }
    // scaled: every residual and every request of the lane is a multiple of 2^k (k from the OR of all
    // values seen at upload) and fits 2^29 in those units; the smallest such k is taken
    const uint32_t k_avail = std::min(ctz64(e->or_left[d]), ctz64(e->or_req[d]));
    const int64_t mx = std::max(e->max_left[d], e->max_req[d]);
    uint32_t k_need = 0;
    while (k_need < 63 && (mx >> k_need) > SCALED_LIMIT) ++k_need;
    if (k_need <= k_avail) {
      kind[d] = SCALED;
      unit[d] = k_need;
      ++ls;
    }
  }
  // keep at most FIT_MAX_LN narrow lanes (prefer the fixed ones)
  if (fixed_narrow && ln > (uint32_t)FIT_MAX_LN)
    for (int d = (int)L - 1; d >= 4 && ln > (uint32_t)FIT_MAX_LN; --d)
      if (kind[d] == NARROW) { kind[d] = WIDE; --ln; }
  // scaled lanes back to wide (last first) until the shape is one the variant table holds
  if (fixed_narrow) {
    for (int d = (int)L - 1; d >= 0 && !fit_variant_exists(L - ln - ls, ln, ls) && ls > 0; --d)
      if (kind[d] == SCALED) { kind[d] = WIDE; --ls; }
  }
  if (!fixed_narrow || !fit_variant_exists(L - ln - ls, ln, ls)) {
    for (uint32_t d = 0; d < L; ++d) kind[d] = WIDE;
    ln = ls = 0;
  }
  for (uint32_t d = 0; d < L; ++d) {
    if (kind[d] == NARROW) lm.narrow[lm.LN++] = (uint8_t)d;
    else if (kind[d] == SCALED) {
      const uint32_t k = unit[d];
      lm.scaled[lm.LS] = (uint8_t)d;
      lm.sunit[lm.LS] = (uint8_t)k;
      lm.sshift[lm.LS] = (uint8_t)std::min(k, (uint32_t)FIT_CAP_LOG2);
      lm.sclamp[lm.LS] = k <= (uint32_t)FIT_CAP_LOG2 ? (1u << (FIT_CAP_LOG2 - k)) : 1u;
      ++lm.LS;
    } else lm.wide[lm.LW++] = (uint8_t)d;
  }
  return lm;
}

// radix passes for the byte digits of (k0, k1) that actually vary (LSD order: k0 low..high, k1 low..high)
uint32_t build_passes(uint64_t vary0, uint64_t vary1, SortPass* out) {
  uint32_t n = 0;
  for (int sh = 0; sh < 64; sh += 8)
    if ((vary0 >> sh) & 0xffull) out[n++] = SortPass{0, (uint8_t)sh};
  for (int sh = 0; sh < 64; sh += 8)
    if ((vary1 >> sh) & 0xffull) out[n++] = SortPass{1, (uint8_t)sh};
  return n;
}

inline uint64_t low_bits_mask(uint32_t n) {  // mask covering every value in [0, n]
  uint64_t m = 0;
  while (m < n) m = (m << 1) | 1ull;
  return m;
}

int rebuild_classes(bs_engine* e) {
  // Pod classes were indexed while the pod table was uploaded; group representative classes are
  // looked up here (the representative index must already hold the pods' (sel, tol) pairs so that
  // the ids agree).  Then the class tables go to the device.
  const uint32_t P = e->P, G = e->G;
  HP_BEGIN(e);
  CK(cudaEventSynchronize(e->ev_classes));   // a previous DMA out of h_grc has finished
  HP(e, "classes:event-wait");
  const bool groups_assigned = e->group_classes_dirty;
  if (e->group_classes_dirty) {
    if (!e->h_grc.resize(G)) return fail(e, BS_E_NOMEM, "pinned host memory");
    const uint64_t* gs = e->h_gsel.data();
    const uint64_t* gt = e->h_gtol.data();
    const uint32_t* ga = e->h_gaff.data();
    assign_classes(e->rep_index, G, [=](uint32_t g) { return ClassKey{gs[g], gt[g], 0u, ga[g]}; }, e->h_grc.data());
    e->group_classes_dirty = false;
  }
  HP(e, "classes:assign-groups");
  if (e->fit_index.size() == 0) e->fit_index.get_or_add(ClassKey{0, 0, 0, BS_AFF_NONE});
  if (e->rep_index.size() == 0) e->rep_index.get_or_add(ClassKey{0, 0, 0, BS_AFF_NONE});
  e->n_fit_classes = (uint32_t)e->fit_index.size();
  e->n_rep_classes = (uint32_t)e->rep_index.size();
  std::vector<uint64_t> fsel(e->n_fit_classes), ftol(e->n_fit_classes), rsel(e->n_rep_classes), rtol(e->n_rep_classes);
  std::vector<uint32_t> fnz(e->n_fit_classes), faff(e->n_fit_classes), raff(e->n_rep_classes);
  bool aff_bad = false, any_aff = false;
  for (uint32_t c = 0; c < e->n_fit_classes; ++c) {
    fsel[c] = e->fit_index.keys[c].sel; ftol[c] = e->fit_index.keys[c].tol; fnz[c] = e->fit_index.keys[c].nz;
    faff[c] = e->fit_index.keys[c].aff;
    aff_bad = aff_bad || (faff[c] != BS_AFF_NONE && faff[c] >= e->n_aff);
  }
  for (uint32_t c = 0; c < e->n_rep_classes; ++c) {
    rsel[c] = e->rep_index.keys[c].sel; rtol[c] = e->rep_index.keys[c].tol; raff[c] = e->rep_index.keys[c].aff;
    any_aff = any_aff || raff[c] != BS_AFF_NONE;
  }
  // (stale representative classes may linger in the persistent index; only the classes in use are checked, and
  // every pod / group has its representative class in that index: no affinity id there, nothing to check)
  if (any_aff) {
    for (uint32_t p = 0; p < P && !aff_bad; ++p) {
      const uint32_t a = e->rep_index.keys[e->h_prc[p]].aff;
      aff_bad = a != BS_AFF_NONE && a >= e->n_aff;
    }
    for (uint32_t g = 0; g < G && !aff_bad; ++g) aff_bad = e->h_gaff[g] != BS_AFF_NONE && e->h_gaff[g] >= e->n_aff;
  }
  if (aff_bad) {
    if (groups_assigned) e->group_classes_dirty = true;   // their ids were not uploaded: assign again next time
    // (group_ids_dirty stays set: an in-place change is uploaded by the next successful rebuild)
    return fail(e, BS_E_INDEX, "affinity class outside the uploaded table (bs_upload_affinity after bs_upload_nodes)");
  }
  HP(e, "classes:tables+checks");
  int rc;
  // cudaMemcpyAsync from pageable memory returns once the data is staged, so the vectors may die.
  if ((rc = upload_vec(e, e->d_fsel, fsel.data(), e->n_fit_classes, e->n_fit_classes))) return rc;
  if ((rc = upload_vec(e, e->d_ftol, ftol.data(), e->n_fit_classes, e->n_fit_classes))) return rc;
  if ((rc = upload_vec(e, e->d_fnz, fnz.data(), e->n_fit_classes, e->n_fit_classes))) return rc;
  if ((rc = upload_vec(e, e->d_faff, faff.data(), e->n_fit_classes, e->n_fit_classes))) return rc;
  if ((rc = upload_vec(e, e->d_raff, raff.data(), e->n_rep_classes, e->n_rep_classes))) return rc;
  if ((rc = upload_vec(e, e->d_rsel, rsel.data(), e->n_rep_classes, e->n_rep_classes))) return rc;
  if ((rc = upload_vec(e, e->d_rtol, rtol.data(), e->n_rep_classes, e->n_rep_classes))) return rc;
  if (e->pod_classes_dirty) {   // a group-only change (bs_update_groups) leaves the pods' ids alone
    if ((rc = upload_vec(e, e->d_pod_fit_class, e->h_pfc.data(), P, std::max(P, 1u)))) return rc;
    if ((rc = upload_vec(e, e->d_pod_rep_class, e->h_prc.data(), P, std::max(P, 1u)))) return rc;
  }
  if ((groups_assigned || e->group_ids_dirty) &&
      (rc = upload_vec(e, e->d_group_rep_class, e->h_grc.data(), G, std::max(G, 1u)))) return rc;
  e->group_ids_dirty = false;
  CK(cudaEventRecord(e->ev_classes, e->s));   // the pinned id arrays are read asynchronously from here on
  HP(e, "classes:uploads");
  e->classes_dirty = false;
  e->pod_classes_dirty = false;
  return BS_OK;
}

int ensure_round_buffers(bs_engine* e) {
  const uint32_t P = std::max(e->P, 1u), G = std::max(e->G, 1u), L = e->L, N = std::max(e->N, 1u);
  CK(e->d_eflags.ensure(G));
  CK(e->d_emin_res.ensure((size_t)L * G * 8));
  CK(e->d_emrpres.ensure((size_t)G * 4));
  CK(e->d_erep_class.ensure((size_t)G * 4));
  CK(e->d_first_pod.ensure((size_t)G * 4));
  CK(e->d_in_round.ensure((size_t)G * 4));
  CK(e->d_contrib.ensure((size_t)G * 4));
  CK(e->d_done.ensure((size_t)G * 4));
  CK(e->d_okA.ensure(G));
  {
    // decision arena layout (256-byte aligned fields)
    struct F { DevBuf* d; PinBuf* h; size_t bytes; };
    F fields[] = {{&e->d_state, &e->h_state, sizeof(RoundState)},
                  {&e->d_prefilter, &e->h_prefilter, P},
                  {&e->d_feasible, &e->h_feasible, (size_t)P * 4},
                  {&e->d_best_node, &e->h_best_node, (size_t)P * 4},
                  {&e->d_best_score, &e->h_best_score, (size_t)P * 8},
                  {&e->d_admit, &e->h_admit, G},
                  {&e->d_admit_bitmap, &e->h_admit_bitmap, (size_t)cdiv(G, 32) * 4},
                  {&e->d_new_denied, &e->h_new_denied, G},
                  {&e->d_order, &e->h_order, (size_t)P * 4},
                  {&e->d_rank, &e->h_rank, (size_t)P * 4},
                  {&e->d_filter_code, &e->h_filter_code, (e->out_flags & BS_OUT_FILTER) ? (size_t)P : 0}};
    size_t total = 0;
    for (auto& f : fields) total += (f.bytes + 255) & ~(size_t)255;
    CK(e->d_arena.ensure(total));
    CK(e->h_arena.ensure(total));
    size_t off = 0;
    for (auto& f : fields) {
      f.d->alias(static_cast<char*>(e->d_arena.p) + off, f.bytes);
      f.h->alias(static_cast<char*>(e->h_arena.p) + off, f.bytes);
      off += (f.bytes + 255) & ~(size_t)255;
    }
    e->arena_bytes = total;
  }
  CK(e->d_best_packed.ensure((size_t)P * 8));
  // rows padded to a whole CTA of pods: the fit kernel writes pods >= P without a guard
  const size_t Prows = (size_t)cdiv(std::max(e->P, 1u), PODS_PER_CTA) * PODS_PER_CTA;
  if (e->out_flags & BS_OUT_FIT_BITMAP) CK(e->d_fit_bitmap.ensure(Prows * std::max(e->bitmap_pitch, 32u) * 4));
  if (e->out_flags & BS_OUT_SCORE) CK(e->d_score.ensure(Prows * std::max(e->score_pitch, 2u) * 8));
  if (e->out_flags & BS_OUT_FILTER) {
    CK(e->d_filter_bitmap.ensure(Prows * std::max(e->W, 1u) * 4));
  }
  // prefix scratch: as many rep-class slots as fit a 1 GiB budget
  const size_t per_class = (size_t)N * (8 * L + 4);
  // BS_PREFIX_BUDGET_BYTES (default 1 GiB) bounds the scratch; classes beyond it are processed in chunks
  size_t budget = (size_t)1 << 30;
  if (const char* bs = getenv("BS_PREFIX_BUDGET_BYTES")) budget = std::max<size_t>(1, strtoull(bs, nullptr, 10));
  uint32_t slots = (uint32_t)std::max<size_t>(1, std::min<size_t>(e->n_rep_classes, budget / per_class));
  slots = std::min(slots, 32768u);   // one grid row (gridDim.y <= 65535) per resident class
  e->prefix_slots = slots;
  CK(e->d_pre.ensure((size_t)slots * L * N * 8));
  CK(e->d_pre_present.ensure((size_t)slots * N * 4));
  CK(e->d_pre_stats.ensure((size_t)slots * sizeof(ClassStats)));
  {
    const size_t n_chunks = cdiv(N, PREFIX_CHUNK);
    const bool fresh = e->d_pre_done.cap < (size_t)slots * 4;
    CK(e->d_pre_part.ensure((size_t)slots * n_chunks * BS_MAX_LANES * 8));
    CK(e->d_pre_part_pres.ensure((size_t)slots * n_chunks * 4));
    CK(e->d_pre_cstats.ensure((size_t)slots * n_chunks * sizeof(ClassStats)));
    CK(e->d_pre_done.ensure((size_t)slots * 4));
    if (fresh) CK(cudaMemsetAsync(e->d_pre_done.p, 0, e->d_pre_done.cap, e->s));
    CK(e->d_max_partial.ensure((size_t)cdiv(G, FINDMAX_THREADS * FINDMAX_PER_THREAD) * sizeof(MaxState)));
  }
  // sort scratch: ONE arena, so that one L2 access-policy window on the sort stream covers it.  The queue sort
  // gathers its key words at random while gang_fit streams 8 GB of scores through the same L2: marked persisting,
  // the sort's few megabytes stay resident instead of turning into DRAM reads in the middle of a write stream.
  {
    const uint32_t M = std::max(P, G);
    struct F { DevBuf* d; size_t bytes; };
    F fields[] = {{&e->d_gk0, (size_t)G * 8}, {&e->d_gk1, (size_t)G * 8}, {&e->d_pk0, (size_t)P * 8}, {&e->d_pk1, (size_t)P * 8},
                  {&e->d_idx_a, (size_t)M * 4}, {&e->d_idx_b, (size_t)M * 4},
                  {&e->d_ghist, (size_t)3 * 256 * cdiv(M, SORT_TILE) * 4}, {&e->d_tilecnt, (size_t)cdiv(M, SORT_TILE) * 4},
                  {&e->d_sort_barrier, sizeof(unsigned int)}, {&e->d_group_rank, (size_t)G * 4}};
    size_t total = 0;
    for (auto& f : fields) total += (f.bytes + 255) & ~(size_t)255;
    const void* old_base = e->d_sort_arena.p;
    CK(e->d_sort_arena.ensure(total));
    size_t off = 0;
    for (auto& f : fields) {
      f.d->alias(static_cast<char*>(e->d_sort_arena.p) + off, f.bytes);
      off += (f.bytes + 255) & ~(size_t)255;
    }
    if (e->d_sort_arena.p != old_base || total != e->sort_arena_bytes) {
      e->sort_arena_bytes = total;
      if (e->l2_persist_bytes) {
        cudaStreamAttrValue v{};
        v.accessPolicyWindow.base_ptr = e->d_sort_arena.p;
        v.accessPolicyWindow.num_bytes = std::min(total, e->l2_window_max);
        v.accessPolicyWindow.hitRatio = total <= e->l2_persist_bytes ? 1.0f : (float)((double)e->l2_persist_bytes / (double)total);
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        if (cudaStreamSetAttribute(e->s2, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) cudaGetLastError();   // a hint only
      }
    }
  }
  return BS_OK;
}

int prepare_nodes(bs_engine* e) {
  // node_left + class fit bitmap (only when nodes or classes changed)
  NodeTab t = node_tab(e);
  StageTimer tm(e, BS_K_NODE_LEFT, e->s);
  CK(e->d_left_w.ensure((size_t)std::max(e->lane_map.LW, 1u) * e->Npad * 8));
  CK(e->d_left_n.ensure((size_t)std::max(e->lane_map.LN + e->lane_map.LS, 1u) * e->Npad * 4));
  CK(e->d_left_present.ensure((size_t)e->Npad * 4));
  if (e->out_flags & BS_OUT_FILTER) CK(e->d_left_plain.ensure((size_t)4 * e->Npad * 8));
  const uint32_t n_tiles = e->Npad / NODE_TILE;
  CK(e->d_classfit.ensure((size_t)e->n_fit_classes * n_tiles * 32 * sizeof(ColBits)));
  node_left_kernel<<<cdiv(e->Npad, 256), 256, 0, e->s>>>(t, e->lane_map, e->d_left_w.as<int64_t>(),
                                                         e->d_left_n.as<int32_t>(),
                                                         e->d_left_present.as<uint32_t>(),
                                                         (e->out_flags & BS_OUT_FILTER) ? e->d_left_plain.as<int64_t>() : nullptr);
  tm.launched();
  {
    for (uint32_t c0 = 0; c0 < e->n_fit_classes; c0 += 32768) {
      dim3 grid(cdiv(n_tiles * 32, 256), std::min(32768u, e->n_fit_classes - c0));
      class_fit_kernel<<<grid, 256, 0, e->s>>>(t, e->d_left_present.as<uint32_t>(), e->d_fsel.as<uint64_t>(),
                                               e->d_ftol.as<uint64_t>(), e->d_fnz.as<uint32_t>(), e->d_faff.as<uint32_t>(),
                                               e->n_fit_classes, n_tiles, e->d_classfit.as<ColBits>(), c0);
      tm.launched();
    }
  }
  CK(cudaGetLastError());
  e->nodes_dirty = false;
  return BS_OK;
}

int evaluate_async_locked(bs_engine* e) {
  if (!e->have_nodes || !e->have_pods || !e->have_groups)
    return fail(e, BS_E_STATE, "bs_evaluate: upload nodes, groups and pods first");
  if (e->peer_broken)
    return fail(e, BS_E_PEER, "peer exchange is broken (a rank did not arrive): bs_peer_detach on every rank, then init/attach again");
  BS_DEVICE_GUARD(e);
  int rc;
  bool reprepare = e->nodes_dirty;
  if (e->classes_dirty) {
    const bool pods_changed = e->pod_classes_dirty;   // the fit classes (class_fit bits) come from the pods only
    const auto tc0 = std::chrono::steady_clock::now();
    if ((rc = rebuild_classes(e))) return rc;
    e->last_classes_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tc0).count();
    reprepare = reprepare || pods_changed;
  }
  {
    const LaneMap lm = classify_lanes(e);
    if (!e->lane_map_valid || memcmp(&lm, &e->lane_map, sizeof(lm)) != 0) {
      e->lane_map = lm;
      e->lane_map_valid = true;
      reprepare = true;
    }
  }
  if ((rc = ensure_round_buffers(e))) return rc;
  for (int k = 0; k < BS_K_COUNT; ++k) e->k_valid[k] = false;
  if (reprepare && (rc = prepare_nodes(e))) return rc;

  const uint32_t P = e->P, G = e->G, L = e->L;
  NodeTab t = node_tab(e);
  PodTab pt = pod_tab(e);
  GroupTab gt = group_tab(e);
  GroupEff ge = group_eff(e);
  PrefixOut po = prefix_out(e);
  RoundState* st = e->d_state.as<RoundState>();

  // fork the sort stream
  CK(cudaEventRecord(e->ev_fork, e->s));
  CK(cudaStreamWaitEvent(e->s2, e->ev_fork, 0));
  CK(cudaStreamWaitEvent(e->s3, e->ev_fork, 0));
  {
    StageTimer tm(e, BS_K_SORT, e->s2);
    // one persistent kernel: group keys -> sort -> dense group rank -> pod keys -> sort -> order + rank
    if (P || G) {
      SortArgs sa{};
      sa.creation = e->d_creation.as<int64_t>();
      sa.name_rank = e->d_name_rank.as<uint32_t>();
      sa.G = G;
      sa.gk0 = e->d_gk0.as<uint64_t>();
      sa.gk1 = e->d_gk1.as<uint64_t>();
      sa.group_rank = e->d_group_rank.as<uint32_t>();
      sa.prio = e->d_prio.as<int32_t>();
      sa.gid = e->d_gid.as<int32_t>();
      sa.ts = e->d_ts.as<int64_t>();
      sa.pflags = e->d_pflags.as<uint8_t>();
      sa.P = P;
      sa.pk0 = e->d_pk0.as<uint64_t>();
      sa.pk1 = e->d_pk1.as<uint64_t>();
      sa.order = e->d_order.as<uint32_t>();
      sa.rank = e->d_rank.as<uint32_t>();
      sa.idx_a = e->d_idx_a.as<uint32_t>();
      sa.idx_b = e->d_idx_b.as<uint32_t>();
      sa.hist = e->d_ghist.as<uint32_t>();
      sa.tilecnt = e->d_tilecnt.as<uint32_t>();
      sa.barrier = e->d_sort_barrier.as<unsigned int>();
      sa.ntiles_max = cdiv(std::max(std::max(P, G), 1u), SORT_TILE);
      sa.n_gpass = build_passes(e->vary_name, e->vary_creation, sa.gpass);
      // word1 = [~biased prio : 32][grouped : 1][group rank or 0x7fffffff : 31]
      const uint64_t vary1 = (e->vary_prio << 32) | 0x80000000ull |
                             ((e->any_lister_miss || e->max_gid >= (int64_t)G) ? 0x7fffffffull : low_bits_mask(G));
      sa.n_ppass = build_passes(e->vary_ts, vary1, sa.ppass);
      if (std::max(P, G) <= (uint32_t)SORT_SMALL_MAX) {
        // small tables: one CTA, the same radix passes with the index arrays in shared memory
        const size_t smem = sort_small_smem();
        CK(cudaFuncSetAttribute(queue_sort_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        queue_sort_small_kernel<<<1, SORT_SMALL_THREADS, smem, e->s2>>>(sa);
        CK(cudaGetLastError());
      } else {
        CK(cudaMemsetAsync(sa.barrier, 0, sizeof(unsigned int), e->s2));
        const uint32_t grid = std::max(1u, std::min(sa.ntiles_max, e->sort_max_grid));
        void* params[] = {&sa};
        // Two builds of the same kernel.  Beside a long fit kernel the sort is hidden anyway and must stay out of its
        // way (32 registers: its CTAs share their SMs with the fit CTAs); when the fit kernel is the shorter of the two
        // (a small shard, few nodes) the round waits for the sort, and the build with 16 gathers in flight per thread
        // is the faster one.  Estimate: pairs x the measured per-pair time of the output mode.
        const double est_fit_ms = (double)P * (double)e->N * ((e->out_flags & BS_OUT_SCORE) ? 1.4e-9 : 0.8e-9);
        const bool lean = e->sort_variant == 1 || (e->sort_variant == 0 && est_fit_ms > 0.6);
        const void* fn = lean ? (const void*)queue_sort_kernel<SORT_LEAN_GROUP> : (const void*)queue_sort_kernel<SORT_WIDE_GROUP>;
        CK(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(SORT_THREADS), params, 0, e->s2));
      }
      tm.launched();
    }
  }
  CK(cudaEventRecord(e->ev_join, e->s2));

  // side stream (high priority): group preparation + findMaxPG, cluster scans, PreFilter.  The fit
  // kernel does not need any of it; only the per-group verdicts do, and they come after both.
  {
    StageTimer tm(e, BS_K_FIND_MAX, e->s3);
    const uint32_t gb = cdiv(std::max(G, 1u), 256);
    group_reset_kernel<<<gb, 256, 0, e->s3>>>(gt, ge, e->d_new_denied.as<uint8_t>(),
                                             e->d_admit_bitmap.as<uint32_t>(), e->d_okA.as<uint8_t>());
    tm.launched();
    if (P) {
      group_first_pod_kernel<<<cdiv(P, 256), 256, 0, e->s3>>>(pt, gt, ge);
      tm.launched();
    }
    if (G) {
      group_effective_kernel<<<gb, 256, 0, e->s3>>>(pt, gt, ge);
      tm.launched();
    }
    const uint32_t nmp = cdiv(std::max(G, 1u), FINDMAX_THREADS * FINDMAX_PER_THREAD);
    find_max_partial_kernel<<<nmp, FINDMAX_THREADS, 0, e->s3>>>(gt, ge, e->d_max_partial.as<MaxState>());
    find_max_final_kernel<<<1, 1024, 0, e->s3>>>(gt, ge, e->d_max_partial.as<MaxState>(), nmp, st, e->N);
    tm.launched(2);
  }
  // ordered cluster scans (compareClusterResourceAndRequire) per rep class
  {
    StageTimer tm(e, BS_K_CLASS_PREFIX, e->s3);
    if (e->N && G && P) {
      PrefixScratch psc = prefix_scratch(e);
      PrefixSel ps{e->d_rsel.as<uint64_t>(), e->d_rtol.as<uint64_t>(), e->d_raff.as<uint32_t>(), 0, 0, 0, 0, 0.f, st};
      for (uint32_t c0 = 0; c0 < e->n_rep_classes; c0 += e->prefix_slots) {
        const uint32_t nc = std::min(e->prefix_slots, e->n_rep_classes - c0);
        ps.c0 = c0;
        ps.mode = 0;
        launch_prefix(L, t, ps, psc, po, nc, e->s3);
        group_check_kernel<<<cdiv(G * 32, 256), 256, 0, e->s3>>>(t, gt, ge, po, c0, nc, st, e->d_okA.as<uint8_t>());
        tm.launched(3);
      }
      ps.c0 = 0;
      ps.mode = 1;
      launch_prefix(L, t, ps, psc, po, 1, e->s3);
      tm.launched(2);
    }
  }
  {
    StageTimer tm(e, BS_K_PREFILTER, e->s3);
    if (P) {
      prefilter_kernel<<<cdiv(P, PREFILTER_THREADS), PREFILTER_THREADS, 0, e->s3>>>(
          t, pt, gt, ge, po, st, e->d_okA.as<uint8_t>(), e->d_prefilter.as<uint8_t>(),
          e->d_new_denied.as<uint8_t>());
      tm.launched();
    }
    if (G) {
      group_idle_admit_kernel<<<cdiv(G, 256), 256, 0, e->s3>>>(gt, ge, e->d_admit.as<uint8_t>(),
                                                              e->d_admit_bitmap.as<uint32_t>());
      tm.launched();
    }
  }
  CK(cudaEventRecord(e->ev_pre, e->s3));
  {
    StageTimer tm(e, BS_K_GANG_FIT, e->s, true);
    if (P) {
      FitArgs a;
      a.left_w = e->d_left_w.as<int64_t>();
      a.left_n = e->d_left_n.as<int32_t>();
      a.lm = e->lane_map;
      a.left_w_pitch = (uint64_t)e->Npad * 8;
      a.left_n_pitch = (uint64_t)e->Npad * 4;
      a.classfit = e->d_classfit.as<ColBits>();
      a.req = e->d_req.as<int64_t>();
      a.req_present = e->d_ppres.as<uint32_t>();
      a.fit_class = e->d_pod_fit_class.as<uint32_t>();
      a.feasible_count = e->d_feasible.as<uint32_t>();
      a.best_node = e->d_best_node.as<int32_t>();
      a.best_score = e->d_best_score.as<int64_t>();
      a.fit_bitmap = (e->out_flags & BS_OUT_FIT_BITMAP) ? e->d_fit_bitmap.as<uint32_t>() : nullptr;
      a.score = (e->out_flags & BS_OUT_SCORE) ? e->d_score.as<int64_t>() : nullptr;
      a.score_pitch = e->score_pitch;
      a.bitmap_pitch = e->bitmap_pitch;
      a.P = P; a.N = e->N; a.Npad = e->Npad; a.W = e->W;
      a.best_packed = e->d_best_packed.as<unsigned long long>();
      uint32_t nl = 1;
      CK(launch_fit(a, cdiv(P, PODS_PER_CTA), e->s, &nl, e->profiling ? e->ev_a[BS_K_GANG_FIT] : nullptr,
                    e->profiling ? e->ev_b[BS_K_GANG_FIT] : nullptr));
      if (e->profiling) e->k_valid[BS_K_GANG_FIT] = true;
      tm.launched(nl);
    }
  }
  CK(cudaStreamWaitEvent(e->s, e->ev_pre, 0));   // PreFilter verdicts, effective group state, RoundState
  if (P && G) {
    AdmitArgs aa{};
    aa.gid = e->d_gid.as<int32_t>();
    aa.prefilter = e->d_prefilter.as<uint8_t>();
    aa.feasible_count = e->d_feasible.as<uint32_t>();
    aa.min_member = gt.min_member; aa.scheduled = gt.scheduled; aa.matched = gt.matched;
    aa.in_round = ge.in_round; aa.contrib = ge.contrib; aa.done = ge.done;
    aa.admit = e->d_admit.as<uint8_t>();
    aa.admit_bitmap = e->d_admit_bitmap.as<uint32_t>();
    aa.P = P; aa.G = G;
    gang_admit_kernel<<<cdiv(P, 256), 256, 0, e->s>>>(aa);
    e->k_launches[BS_K_GANG_FIT] += 1;
    e->launches += 1;
  }
  {
    StageTimer tm(e, BS_K_FILTER, e->s);
    if (P && (e->out_flags & BS_OUT_FILTER)) {
      FilterArgs fa;
      fa.left_plain = e->d_left_plain.as<int64_t>();
      fa.node_flags = e->d_nflags.as<uint8_t>();
      fa.req = e->d_req.as<int64_t>();
      fa.req_present = e->d_ppres.as<uint32_t>();
      fa.gid = e->d_gid.as<int32_t>();
      fa.emin_res = ge.min_res;
      fa.emin_res_present = ge.min_res_present;
      fa.eflags = ge.flags;
      fa.st = st;
      fa.filter_bitmap = e->d_filter_bitmap.as<uint32_t>();
      fa.filter_code = e->d_filter_code.as<uint8_t>();
      fa.P = P; fa.N = e->N; fa.Npad = e->Npad; fa.W = e->W; fa.G = G; fa.L = L;
      const uint32_t warps = cdiv(P, FILTER_PPW);
      filter_kernel<<<cdiv(warps * 32, 256), 256, 0, e->s>>>(fa);
      tm.launched();
    }
  }
  if (e->peer_attached) {
    // admit-bitmap all-gather over peer memory (kernels.cuh K8): the push is the round's last kernel on
    // the main stream, ordered behind the PREVIOUS round's wait (slot reuse rule); the wait for this
    // round's slots spins on the side stream s4 while the next round may already be computing.
    PeerArgs pa{};
    for (uint32_t r = 0; r < e->peer_world; ++r) pa.peer_buf[r] = reinterpret_cast<uint32_t*>(e->peer_ptr[r]);
    pa.local_bitmap = e->d_admit_bitmap.as<uint32_t>();
    pa.rank = e->peer_rank; pa.world = e->peer_world; pa.words_per_rank = e->peer_wpr;
    pa.n_words = std::min(e->peer_wpr, cdiv(std::max(G, 1u), 32));
    pa.seq = ++e->peer_seq;
    pa.err = e->d_peer_err.as<int>();
    pa.timeout_ns = e->peer_timeout_ns;
    if (pa.seq > 1) CK(cudaStreamWaitEvent(e->s, e->ev_gath, 0));
    {
      StageTimer tm(e, BS_K_PEER, e->s);
      peer_push_kernel<<<e->peer_world, 256, 0, e->s>>>(pa);
      tm.launched();
    }
    CK(cudaEventRecord(e->ev_push, e->s));
    CK(cudaStreamWaitEvent(e->s4, e->ev_push, 0));
    peer_wait_kernel<<<1, 32, 0, e->s4>>>(pa);
    e->k_launches[BS_K_PEER] += 1;
    e->launches += 1;
    CK(cudaEventRecord(e->ev_gath, e->s4));
  }
  CK(cudaStreamWaitEvent(e->s, e->ev_join, 0));
  CK(cudaGetLastError());
  e->evaluated = true;
  e->fetched = false;
  e->gang_applied = false;
  return BS_OK;
}

int fetch_locked(bs_engine* e, bs_results* out, bool view = false) {
  if (!e->evaluated) return fail(e, BS_E_STATE, "bs_fetch: nothing evaluated");
  const uint32_t P = e->P, G = e->G;
  HP_BEGIN(e);
  if (!e->fetched) {
    if (e->arena_bytes)   // every decision vector in one DMA (the arena layout is the same on both sides)
      CK(cudaMemcpyAsync(e->h_arena.p, e->d_arena.p, e->arena_bytes, cudaMemcpyDeviceToHost, e->s));
    CK(cudaStreamSynchronize(e->s));
    e->fetched = true;
  }
  HP(e, "fetch:d2h+wait");
  const RoundState* st = e->h_state.as<RoundState>();
  if (e->gang.active && e->gang.groups.size() == G && !e->gang_applied) {
    // AddToDenyCache for every group a pod of the round hit "cluster resource not enough" in (core.go:142,163)
    const uint8_t* nd = e->h_new_denied.as<uint8_t>();
    for (uint32_t g = 0; g < G; ++g)
      if (nd[g]) e->gang.deny(g, e->cycle_now_ns);
    e->gang_applied = true;
  }
  if (out && view) {
    out->prefilter = e->h_prefilter.as<uint8_t>();
    out->feasible_count = e->h_feasible.as<uint32_t>();
    out->best_node = e->h_best_node.as<int32_t>();
    out->best_score = e->h_best_score.as<int64_t>();
    out->admit = e->h_admit.as<uint8_t>();
    out->admit_bitmap = e->h_admit_bitmap.as<uint32_t>();
    out->new_denied = e->h_new_denied.as<uint8_t>();
    out->order = e->h_order.as<uint32_t>();
    out->rank = e->h_rank.as<uint32_t>();
    out->filter_code = (e->out_flags & BS_OUT_FILTER) ? e->h_filter_code.as<uint8_t>() : nullptr;
    out->max_group = st->max_group;
    out->max_finished = st->max_finished;
  } else if (out) {
    auto cp = [](void* dst, const PinBuf& src, size_t bytes) {
      if (dst && bytes) memcpy(dst, src.p, bytes);
    };
    cp(out->prefilter, e->h_prefilter, P);
    cp(out->feasible_count, e->h_feasible, (size_t)P * 4);
    cp(out->best_node, e->h_best_node, (size_t)P * 4);
    cp(out->best_score, e->h_best_score, (size_t)P * 8);
    cp(out->admit, e->h_admit, G);
    cp(out->admit_bitmap, e->h_admit_bitmap, (size_t)cdiv(G, 32) * 4);
    cp(out->new_denied, e->h_new_denied, G);
    cp(out->order, e->h_order, (size_t)P * 4);
    cp(out->rank, e->h_rank, (size_t)P * 4);
    out->max_group = st->max_group;
    out->max_finished = st->max_finished;
    if (e->out_flags & BS_OUT_FILTER) cp(out->filter_code, e->h_filter_code, P);
  }
  HP(e, "fetch:copy-out");
  if (st->ref_panic)
    return fail(e, BS_E_REF_PANIC, "findMaxPG: MinMember == 0 with Status.Scheduled != 0 (core.go:716-717 divides by zero)");
  return BS_OK;
}

}  // namespace

// ============================================================================
extern "C" {

int bs_abi_version(void) { return BS_ABI_VERSION; }

const char* bs_strerror(int err) {
  switch (err) {
    case BS_OK: return "ok";
    case BS_E_INVAL: return "invalid argument";
    case BS_E_NODEVICE: return "no CUDA device (this engine has no CPU path)";
    case BS_E_CUDA: return "CUDA runtime error";
    case BS_E_NOMEM: return "out of memory";
    case BS_E_RANGE: return "table value outside +-2^56";
    case BS_E_STATE: return "call out of order";
    case BS_E_REF_PANIC: return "reference would panic (findMaxPG divide by zero)";
    case BS_E_INDEX: return "index out of range";
    case BS_E_PEER: return "peer exchange timed out";
  }
  return "unknown error";
}

const char* bs_last_error(const bs_engine* e) { return e ? e->err.c_str() : ""; }

int bs_create(const bs_config* cfg, bs_engine** out) {
  if (!cfg || !out) return BS_E_INVAL;
  *out = nullptr;
  if (cfg->n_lanes < BS_FIXED_LANES || cfg->n_lanes > BS_MAX_LANES) return BS_E_INVAL;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return BS_E_NODEVICE;
  }
  if (cfg->device < 0 || cfg->device >= ndev) return BS_E_INVAL;
  DeviceGuard guard(cfg->device);
  if (guard.err != cudaSuccess) return BS_E_CUDA;
  bs_engine* e = new (std::nothrow) bs_engine();
  if (!e) return BS_E_NOMEM;
  e->device = cfg->device;
  e->L = cfg->n_lanes;
  e->out_flags = cfg->out_flags;
  e->host_prof = getenv("BS_HOST_PROFILE") != nullptr;
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // the small kernels of the PreFilter chain must get the
                                                          // SM slots the fit kernel's retiring CTAs free
  bool ok = cudaStreamCreateWithFlags(&e->s, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&e->s2, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithPriority(&e->s3, cudaStreamNonBlocking, prio_hi) == cudaSuccess &&
            cudaStreamCreateWithPriority(&e->s4, cudaStreamNonBlocking, prio_hi) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_pre, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_push, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_gath, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_classes, cudaEventDisableTiming) == cudaSuccess;
  for (int k = 0; ok && k < BS_K_COUNT; ++k)
    ok = cudaEventCreate(&e->ev_a[k]) == cudaSuccess && cudaEventCreate(&e->ev_b[k]) == cudaSuccess;
  if (ok) {
    int per_sm = 0, sms = 0;
    int per_sm_wide = 0;
    ok = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, queue_sort_kernel<SORT_LEAN_GROUP>, SORT_THREADS, 0) == cudaSuccess &&
         cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_wide, queue_sort_kernel<SORT_WIDE_GROUP>, SORT_THREADS, 0) == cudaSuccess &&
         cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device) == cudaSuccess;
    // the sort shares the GPU with the fit kernel on the other stream: one CTA per SM is plenty
    per_sm = std::min(per_sm, per_sm_wide);
    e->sort_max_grid = (uint32_t)std::max(1, std::min(per_sm * sms, sms));
    if (const char* sv = getenv("BS_SORT_VARIANT")) e->sort_variant = atoi(sv);   // 0 auto, 1 lean, 2 wide (measurement)
    // persisting-L2 set-aside for the sort scratch (BS_SORT_L2_PERSIST_MB, default 16, 0 = off); a hint: failures are ignored
    int max_persist = 0, max_window = 0;
    size_t want_mb = 16;
    if (const char* lp = getenv("BS_SORT_L2_PERSIST_MB")) want_mb = (size_t)std::max(0, atoi(lp));
    if (want_mb && cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, cfg->device) == cudaSuccess &&
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, cfg->device) == cudaSuccess &&
        max_persist > 0 && max_window > 0) {
      const size_t want = std::min<size_t>(want_mb << 20, (size_t)max_persist);
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
        e->l2_persist_bytes = want;
        e->l2_window_max = (size_t)max_window;
      } else {
        cudaGetLastError();
      }
    }
    if (const char* sg = getenv("BS_SORT_GRID")) e->sort_max_grid = (uint32_t)std::max(1, std::min(atoi(sg), per_sm * sms));
  }
  if (!ok) {
    bs_destroy(e);
    return BS_E_CUDA;
  }
  *out = e;
  return BS_OK;
}

void bs_destroy(bs_engine* e) {
  if (!e) return;
  DeviceGuard guard(e->device);
  if (e->s) cudaStreamSynchronize(e->s);
  if (e->s2) cudaStreamSynchronize(e->s2);
  if (e->s4) cudaStreamSynchronize(e->s4);
  for (uint32_t r = 0; r < e->peer_world; ++r)
    if (r != e->peer_rank && e->peer_ptr[r]) cudaIpcCloseMemHandle(e->peer_ptr[r]);
  e->d_gather.release();
  e->d_peer_err.release();
  DevBuf* bufs[] = {&e->d_alloc, &e->d_requested, &e->d_pod_count, &e->d_apres, &e->d_rpres, &e->d_label,
                    &e->d_taint, &e->d_nflags, &e->d_left_w, &e->d_left_n, &e->d_left_present, &e->d_left_plain, &e->d_filter_bitmap, &e->d_filter_code, &e->d_classfit, &e->d_req,
                    &e->d_ppres, &e->d_gid, &e->d_prio, &e->d_ts, &e->d_pflags, &e->d_pod_fit_class,
                    &e->d_pod_rep_class, &e->d_min_member, &e->d_scheduled, &e->d_matched, &e->d_gflags,
                    &e->d_min_res, &e->d_mrpres, &e->d_creation, &e->d_name_rank, &e->d_group_rep_class,
                    &e->d_fsel, &e->d_ftol, &e->d_fnz, &e->d_faff, &e->d_rsel, &e->d_rtol, &e->d_raff, &e->d_aff_bits, &e->d_eflags, &e->d_emin_res,
                    &e->d_emrpres, &e->d_erep_class, &e->d_first_pod, &e->d_in_round, &e->d_contrib,
                    &e->d_done, &e->d_okA, &e->d_state, &e->d_pre, &e->d_pre_present, &e->d_pre_stats, &e->d_max_partial, &e->d_pre_part,
                    &e->d_pre_part_pres, &e->d_pre_cstats, &e->d_pre_done,
                    &e->d_best_packed, &e->d_prefilter, &e->d_feasible, &e->d_best_node, &e->d_best_score, &e->d_admit,
                    &e->d_admit_bitmap, &e->d_new_denied, &e->d_fit_bitmap, &e->d_score, &e->d_order,
                    &e->d_rank, &e->d_gk0, &e->d_gk1, &e->d_pk0, &e->d_pk1, &e->d_idx_a, &e->d_idx_b,
                    &e->d_ghist, &e->d_skip, &e->d_group_rank, &e->d_gorder, &e->d_tilecnt, &e->d_sort_barrier,
                    &e->r_req, &e->r_pc, &e->r_rp, &e->r_matched, &e->r_gflags, &e->r_grc, &e->r_minres, &e->r_mrp,
                    &e->r_queue, &e->r_pf, &e->r_node, &e->r_ready, &e->r_status, &e->r_sum, &e->r_max, &e->r_keys,
                    &e->r_left0, &e->r_left1, &e->r_both, &e->r_fit, &e->r_stat};
  for (DevBuf* b : bufs) b->release();
  e->d_sort_arena.release();
  e->d_arena.release();
  e->h_arena.release();
  for (DevBuf& b : e->u_buf) b.release();
  PinBuf* pins[] = {&e->h_prefilter, &e->h_feasible, &e->h_best_node, &e->h_best_score, &e->h_admit,
                    &e->h_admit_bitmap, &e->h_new_denied, &e->h_order, &e->h_rank, &e->h_state, &e->h_filter_code};
  for (PinBuf* b : pins) b->release();
  for (int k = 0; k < BS_K_COUNT; ++k) {
    if (e->ev_a[k]) cudaEventDestroy(e->ev_a[k]);
    if (e->ev_b[k]) cudaEventDestroy(e->ev_b[k]);
  }
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  if (e->ev_pre) cudaEventDestroy(e->ev_pre);
  if (e->ev_push) cudaEventDestroy(e->ev_push);
  if (e->ev_gath) cudaEventDestroy(e->ev_gath);
  if (e->s3) cudaStreamDestroy(e->s3);
  if (e->s4) cudaStreamDestroy(e->s4);
  if (e->ev_classes) cudaEventDestroy(e->ev_classes);
  e->h_pfc.release(); e->h_prc.release(); e->h_grc.release();
  if (e->s) cudaStreamDestroy(e->s);
  if (e->s2) cudaStreamDestroy(e->s2);
  delete e;
}

int bs_upload_nodes(bs_engine* e, const bs_node_table* t) {
  if (!e || !t) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (t->n_lanes != e->L) return fail(e, BS_E_INVAL, "bs_upload_nodes: n_lanes differs from the engine's");
  const uint32_t N = t->n_nodes, L = e->L;
  if (N && (!t->alloc || !t->requested || !t->pod_count || !t->alloc_present || !t->req_present ||
            !t->label_mask || !t->taint_mask || !t->flags))
    return fail(e, BS_E_INVAL, "bs_upload_nodes: null column");
  HP_BEGIN(e);
  const NodeHostStats hs = node_host_pass(t, L, N);
  if (!hs.ok) return fail(e, BS_E_RANGE, "bs_upload_nodes: value outside +-2^56");
  HP(e, "nodes:host-pass");
  BS_DEVICE_GUARD(e);
  const uint32_t Npad = std::max(1u, cdiv(N, NODE_TILE)) * NODE_TILE;
  int rc;
  if ((rc = upload_lanes(e, e->d_alloc, t->alloc, L, N, Npad))) return rc;
  if ((rc = upload_lanes(e, e->d_requested, t->requested, L, N, Npad))) return rc;
  if ((rc = upload_vec(e, e->d_pod_count, t->pod_count, N, Npad))) return rc;
  if ((rc = upload_vec(e, e->d_apres, t->alloc_present, N, Npad))) return rc;
  if ((rc = upload_vec(e, e->d_rpres, t->req_present, N, Npad))) return rc;
  if ((rc = upload_vec(e, e->d_label, t->label_mask, N, Npad))) return rc;
  if ((rc = upload_vec(e, e->d_taint, t->taint_mask, N, Npad))) return rc;
  if ((rc = upload_vec(e, e->d_nflags, t->flags, N, Npad))) return rc;
  HP(e, "nodes:dma-enqueue");
  CK(cudaStreamSynchronize(e->s));
  HP(e, "nodes:dma-wait");
  e->h_nflags.assign(t->flags, t->flags + N);
  memcpy(e->max_alloc, hs.mx_a, sizeof(hs.mx_a));
  memcpy(e->max_requested, hs.mx_r, sizeof(hs.mx_r));
  memcpy(e->or_left, hs.or_l, sizeof(hs.or_l));
  memcpy(e->max_left, hs.mx_l, sizeof(hs.mx_l));
  e->max_pod_count = hs.mx_pc;
  e->N = N;
  e->score_pitch = (N + 1u) & ~1u;
  e->bitmap_pitch = (cdiv(N, 32) + 31u) & ~31u;
  if (e->n_aff) e->classes_dirty = true;   // class ids are validated again: the affinity table belongs to the
  e->n_aff = 0;                            // node snapshot and goes with it
  e->Npad = Npad;
  e->W = cdiv(N, 32);
  e->have_nodes = true;
  e->nodes_dirty = true;
  e->evaluated = false;
  return BS_OK;
}

int bs_update_nodes(bs_engine* e, const uint32_t* idx, const bs_node_table* t) {
  if (!e || !t || (t->n_nodes && !idx)) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_nodes) return fail(e, BS_E_STATE, "bs_update_nodes: upload nodes first");
  if (t->n_lanes != e->L) return fail(e, BS_E_INVAL, "bs_update_nodes: n_lanes differs from the engine's");
  const uint32_t n = t->n_nodes, L = e->L;
  if (!n) return BS_OK;
  if (!t->alloc || !t->requested || !t->pod_count || !t->alloc_present || !t->req_present || !t->label_mask ||
      !t->taint_mask || !t->flags)
    return fail(e, BS_E_INVAL, "bs_update_nodes: null column");
  for (uint32_t k = 0; k < n; ++k)
    if (idx[k] >= e->N) return BS_E_INDEX;
  int64_t mx_a[BS_MAX_LANES] = {}, mx_r[BS_MAX_LANES] = {};
  if (!lane_maxima(t->alloc, L, n, mx_a) || !lane_maxima(t->requested, L, n, mx_r))
    return fail(e, BS_E_RANGE, "bs_update_nodes: value outside +-2^56");
  BS_DEVICE_GUARD(e);
  HP_BEGIN(e);
  // scratch of the changed rows: kept in the engine (cudaMalloc / cudaFree per call would cost more than the scatter)
  DevBuf &da = e->u_buf[0], &dr = e->u_buf[1], &dpc = e->u_buf[2], &dap = e->u_buf[3], &drp = e->u_buf[4], &dl = e->u_buf[5],
         &dt = e->u_buf[6], &df = e->u_buf[7], &di = e->u_buf[8];
  cudaError_t er = da.ensure((size_t)L * n * 8);
  if (er == cudaSuccess) er = dr.ensure((size_t)L * n * 8);
  if (er == cudaSuccess) er = dpc.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = dap.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = drp.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = dl.ensure((size_t)n * 8);
  if (er == cudaSuccess) er = dt.ensure((size_t)n * 8);
  if (er == cudaSuccess) er = df.ensure(n);
  if (er == cudaSuccess) er = di.ensure((size_t)n * 4);
  auto h2d = [&](DevBuf& d, const void* src, size_t bytes) {
    if (er == cudaSuccess) er = cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, e->s);
  };
  h2d(da, t->alloc, (size_t)L * n * 8); h2d(dr, t->requested, (size_t)L * n * 8);
  h2d(dpc, t->pod_count, (size_t)n * 4); h2d(dap, t->alloc_present, (size_t)n * 4);
  h2d(drp, t->req_present, (size_t)n * 4); h2d(dl, t->label_mask, (size_t)n * 8);
  h2d(dt, t->taint_mask, (size_t)n * 8); h2d(df, t->flags, n); h2d(di, idx, (size_t)n * 4);
  if (er == cudaSuccess) {
    NodeTabMut dst{e->d_alloc.as<int64_t>(), e->d_requested.as<int64_t>(), e->d_pod_count.as<int32_t>(),
                   e->d_apres.as<uint32_t>(), e->d_rpres.as<uint32_t>(), e->d_label.as<uint64_t>(),
                   e->d_taint.as<uint64_t>(), e->d_nflags.as<uint8_t>()};
    NodeTab src{};
    src.alloc = da.as<int64_t>(); src.requested = dr.as<int64_t>(); src.pod_count = dpc.as<int32_t>();
    src.alloc_present = dap.as<uint32_t>(); src.req_present = drp.as<uint32_t>(); src.label = dl.as<uint64_t>();
    src.taint = dt.as<uint64_t>(); src.flags = df.as<uint8_t>();
    node_scatter_kernel<<<cdiv(n, 256), 256, 0, e->s>>>(dst, e->Npad, L, src, di.as<uint32_t>(), n);
    e->launches++;
    HP(e, "upd-nodes:enqueue");
    er = cudaStreamSynchronize(e->s);
  }
  CK(er);
  HP(e, "upd-nodes:wait");
  // lane maxima only ever grow here (a conservative bound keeps the wide/narrow split exact); the OR
  // of the residuals only gains bits (fewer common trailing zeros: a smaller unit, still exact)
  left_stats(t, L, n, e->or_left, e->max_left);
  for (uint32_t d = 0; d < L; ++d) {
    e->max_alloc[d] = std::max(e->max_alloc[d], mx_a[d]);
    e->max_requested[d] = std::max(e->max_requested[d], mx_r[d]);
  }
  for (uint32_t k = 0; k < n; ++k) {
    e->max_pod_count = std::max<int64_t>(e->max_pod_count, std::abs((int64_t)t->pod_count[k]));
    e->h_nflags[idx[k]] = t->flags[k];
  }
  e->nodes_dirty = true;
  e->evaluated = false;
  return BS_OK;
}

int bs_upload_groups(bs_engine* e, const bs_group_table* t) {
  if (!e || !t) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (t->n_lanes != e->L) return fail(e, BS_E_INVAL, "bs_upload_groups: n_lanes differs from the engine's");
  const uint32_t G = t->n_groups, L = e->L;
  if (G && (!t->min_member || !t->scheduled || !t->matched || !t->flags || !t->min_res ||
            !t->min_res_present || !t->rep_sel || !t->rep_tol || !t->creation_ns || !t->name_rank))
    return fail(e, BS_E_INVAL, "bs_upload_groups: null column");
  // the DMAs go first (asynchronous from pinned tables) and run under the host checks below; a table
  // that then fails validation is dropped (have_groups = false)
  BS_DEVICE_GUARD(e);
  HP_BEGIN(e);
  e->have_groups = false;
  e->evaluated = false;
  const uint32_t Gp = std::max(G, 1u);
  int rc;
  if ((rc = upload_vec(e, e->d_min_member, t->min_member, G, Gp))) return rc;
  if ((rc = upload_vec(e, e->d_scheduled, t->scheduled, G, Gp))) return rc;
  if ((rc = upload_vec(e, e->d_matched, t->matched, G, Gp))) return rc;
  if ((rc = upload_vec(e, e->d_gflags, t->flags, G, Gp))) return rc;
  if ((rc = upload_lanes(e, e->d_min_res, t->min_res, L, G, Gp))) return rc;
  if ((rc = upload_vec(e, e->d_mrpres, t->min_res_present, G, Gp))) return rc;
  if ((rc = upload_vec(e, e->d_creation, t->creation_ns, G, Gp))) return rc;
  if ((rc = upload_vec(e, e->d_name_rank, t->name_rank, G, Gp))) return rc;
  HP(e, "groups:dma-enqueue");
  // one chunked pass over the host columns (an omp team for big tables): |min_res| range, the varying bits of the
  // sort-key words, creation sentinel, and whether the representative columns moved since their ids were assigned
  uint64_t o1 = 0, a1 = ~0ull, o0 = 0, a0 = ~0ull;
  int bad_creation = 0, bad_range = 0, reps_differ = 0;
  {
    const bool cmp_reps = e->h_gsel.size() == G && e->h_gtol.size() == G && e->h_grc.size() == G && e->h_gaff.size() == G;
    if (!cmp_reps) reps_differ = 1;
    const int T = G < 8192 ? 1 : host_threads();
    const uint32_t chunk = (G + T - 1) / std::max(T, 1);
    const uint64_t* hs = e->h_gsel.data();
    const uint64_t* ht = e->h_gtol.data();
    const uint32_t* ha = e->h_gaff.data();
#pragma omp parallel for schedule(static, 1) num_threads(T) if (T > 1) reduction(| : o1, o0, bad_creation, bad_range, reps_differ) reduction(& : a1, a0)
    for (int tk = 0; tk < T; ++tk) {
      const uint32_t g0 = std::min(G, (uint32_t)tk * chunk), g1 = std::min(G, g0 + chunk);
      for (uint32_t d = 0; d < L; ++d) {
        const int64_t* row = t->min_res + (size_t)d * G;
        int64_t lo = 0, hi = 0;
        for (uint32_t g = g0; g < g1; ++g) { lo = std::min(lo, row[g]); hi = std::max(hi, row[g]); }
        bad_range |= (lo < -BS_VALUE_LIMIT || hi > BS_VALUE_LIMIT) ? 1 : 0;
      }
      uint64_t lo1 = 0, la1 = ~0ull, lo0 = 0, la0 = ~0ull;
      int bc = 0;
      for (uint32_t g = g0; g < g1; ++g) {
        const uint64_t c = (uint64_t)t->creation_ns[g], nm = (uint64_t)(~t->name_rank[g]);
        lo1 |= c; la1 &= c; lo0 |= nm; la0 &= nm;
        bc |= t->creation_ns[g] == INT64_MAX ? 1 : 0;
      }
      o1 |= lo1; a1 &= la1; o0 |= lo0; a0 &= la0; bad_creation |= bc;
      if (cmp_reps && g1 > g0) {
        int df = memcmp(hs + g0, t->rep_sel + g0, (size_t)(g1 - g0) * 8) != 0 || memcmp(ht + g0, t->rep_tol + g0, (size_t)(g1 - g0) * 8) != 0;
        if (t->rep_aff_class) df = df || memcmp(ha + g0, t->rep_aff_class + g0, (size_t)(g1 - g0) * 4) != 0;
        else
          for (uint32_t g = g0; g < g1 && !df; ++g) df = ha[g] != BS_AFF_NONE;
        reps_differ |= df;
      }
    }
  }
  if (bad_range) {
    cudaStreamSynchronize(e->s);
    return fail(e, BS_E_RANGE, "bs_upload_groups: value outside +-2^56");
  }
  if (bad_creation) {
    cudaStreamSynchronize(e->s);
    return fail(e, BS_E_RANGE, "bs_upload_groups: creation_ns == INT64_MAX");
  }
  e->vary_creation = G ? (o1 ^ a1) : 0;
  e->vary_name = G ? (o0 ^ a0) : 0;
  e->g_or1 = o1; e->g_and1 = a1; e->g_or0 = o0; e->g_and0 = a0;
  // representative (sel, tol, affinity) columns unchanged since the ids were assigned: nothing to look up again
  const bool same_reps = !reps_differ;
  if (!same_reps) {
    e->h_gsel.assign(t->rep_sel, t->rep_sel + G);
    e->h_gtol.assign(t->rep_tol, t->rep_tol + G);
    e->h_gaff.resize(G);
    for (uint32_t g = 0; g < G; ++g) e->h_gaff[g] = t->rep_aff_class ? t->rep_aff_class[g] : BS_AFF_NONE;
    e->group_classes_dirty = true;
    e->classes_dirty = true;
  }
  if (e->h_wait_ns.size() != G) e->h_wait_ns.assign(G, -1);
  HP(e, "groups:host-pass");
  CK(cudaStreamSynchronize(e->s));   // the caller's arrays are free again once we return
  HP(e, "groups:dma-wait");
  e->h_min_member.assign(t->min_member, t->min_member + G);
  e->h_scheduled.assign(t->scheduled, t->scheduled + G);
  e->h_matched_up.assign(t->matched, t->matched + G);
  e->h_gflags_up.assign(t->flags, t->flags + G);
  HP(e, "groups:host-copies");
  e->G = G;
  e->have_groups = true;
  e->evaluated = false;
  return BS_OK;
}

int bs_update_groups(bs_engine* e, const uint32_t* idx, const bs_group_table* t) {
  if (!e || !t || (t->n_groups && !idx)) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_groups) return fail(e, BS_E_STATE, "bs_update_groups: upload groups first");
  if (t->n_lanes != e->L) return fail(e, BS_E_INVAL, "bs_update_groups: n_lanes differs from the engine's");
  const uint32_t n = t->n_groups, L = e->L, G = e->G;
  if (!n) return BS_OK;
  if (!t->min_member || !t->scheduled || !t->matched || !t->flags || !t->min_res || !t->min_res_present ||
      !t->rep_sel || !t->rep_tol || !t->creation_ns || !t->name_rank)
    return fail(e, BS_E_INVAL, "bs_update_groups: null column");
  for (uint32_t k = 0; k < n; ++k)
    if (idx[k] >= G) return BS_E_INDEX;
  {
    int64_t mx[BS_MAX_LANES] = {};
    if (!lane_maxima(t->min_res, L, n, mx)) return fail(e, BS_E_RANGE, "bs_update_groups: value outside +-2^56");
  }
  for (uint32_t k = 0; k < n; ++k)
    if (t->creation_ns[k] == INT64_MAX) return fail(e, BS_E_RANGE, "bs_update_groups: creation_ns == INT64_MAX");
  BS_DEVICE_GUARD(e);
  HP_BEGIN(e);
  DevBuf &dmm = e->u_buf[0], &dsc = e->u_buf[1], &dma = e->u_buf[2], &dfl = e->u_buf[3], &dmr = e->u_buf[4], &dmp = e->u_buf[5],
         &dcr = e->u_buf[6], &dnr = e->u_buf[7], &di = e->u_buf[8];
  cudaError_t er = dmm.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = dsc.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = dma.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = dfl.ensure(n);
  if (er == cudaSuccess) er = dmr.ensure((size_t)L * n * 8);
  if (er == cudaSuccess) er = dmp.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = dcr.ensure((size_t)n * 8);
  if (er == cudaSuccess) er = dnr.ensure((size_t)n * 4);
  if (er == cudaSuccess) er = di.ensure((size_t)n * 4);
  auto h2d = [&](DevBuf& d, const void* src, size_t bytes) {
    if (er == cudaSuccess) er = cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, e->s);
  };
  h2d(dmm, t->min_member, (size_t)n * 4); h2d(dsc, t->scheduled, (size_t)n * 4); h2d(dma, t->matched, (size_t)n * 4);
  h2d(dfl, t->flags, n); h2d(dmr, t->min_res, (size_t)L * n * 8); h2d(dmp, t->min_res_present, (size_t)n * 4);
  h2d(dcr, t->creation_ns, (size_t)n * 8); h2d(dnr, t->name_rank, (size_t)n * 4); h2d(di, idx, (size_t)n * 4);
  if (er == cudaSuccess) {
    GroupCols dst{e->d_min_member.as<uint32_t>(), e->d_scheduled.as<uint32_t>(), e->d_matched.as<uint32_t>(),
                  e->d_gflags.as<uint8_t>(), e->d_min_res.as<int64_t>(), e->d_mrpres.as<uint32_t>(),
                  e->d_creation.as<int64_t>(), e->d_name_rank.as<uint32_t>()};
    GroupCols src{dmm.as<uint32_t>(), dsc.as<uint32_t>(), dma.as<uint32_t>(), dfl.as<uint8_t>(), dmr.as<int64_t>(),
                  dmp.as<uint32_t>(), dcr.as<int64_t>(), dnr.as<uint32_t>()};
    group_scatter_kernel<<<cdiv(n, 256), 256, 0, e->s>>>(dst, std::max(G, 1u), L, src, di.as<uint32_t>(), n);
    e->launches++;
    HP(e, "upd-groups:enqueue");
    er = cudaStreamSynchronize(e->s);
  }
  CK(er);
  HP(e, "upd-groups:wait");
  // sort-key digits that vary: the accumulated OR / AND only widen (a superset costs a pass, never an error)
  for (uint32_t k = 0; k < n; ++k) {
    const uint64_t c = (uint64_t)t->creation_ns[k], nm = (uint64_t)(~t->name_rank[k]);
    e->g_or1 |= c; e->g_and1 &= c; e->g_or0 |= nm; e->g_and0 &= nm;
    e->h_gsel[idx[k]] = t->rep_sel[k];
    e->h_gtol[idx[k]] = t->rep_tol[k];
    e->h_gaff[idx[k]] = t->rep_aff_class ? t->rep_aff_class[k] : BS_AFF_NONE;
    e->h_min_member[idx[k]] = t->min_member[k];
    e->h_scheduled[idx[k]] = t->scheduled[k];
    e->h_matched_up[idx[k]] = t->matched[k];
    e->h_gflags_up[idx[k]] = t->flags[k];
  }
  e->vary_creation = e->g_or1 ^ e->g_and1;
  e->vary_name = e->g_or0 ^ e->g_and0;
  e->classes_dirty = true;         // the class tables go to the device again (new classes may have appeared); the pods' ids stay
  if (!e->group_classes_dirty && e->h_grc.size() == G) {
    // the other groups' ids are current: look up only the changed rows (the index keeps ids stable)
    CK(cudaEventSynchronize(e->ev_classes));   // no DMA is reading h_grc
    for (uint32_t k = 0; k < n; ++k)
      e->h_grc[idx[k]] = e->rep_index.get_or_add(ClassKey{e->h_gsel[idx[k]], e->h_gtol[idx[k]], 0u, e->h_gaff[idx[k]]});
    e->group_ids_dirty = true;
  } else {
    e->group_classes_dirty = true;
  }
  e->evaluated = false;
  return BS_OK;
}

int bs_upload_pods(bs_engine* e, const bs_pod_table* t) {
  if (!e || !t) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (t->n_lanes != e->L) return fail(e, BS_E_INVAL, "bs_upload_pods: n_lanes differs from the engine's");
  const uint32_t P = t->n_pods, L = e->L;
  if (P && (!t->req || !t->req_present || !t->gid || !t->sel_mask || !t->tol_mask || !t->priority ||
            !t->ts_ns || !t->flags))
    return fail(e, BS_E_INVAL, "bs_upload_pods: null column");
  // ONE parallel pass over the table before anything is committed: per-lane maxima (range check and
  // wide/narrow lane classification), the varying bits of the sort keys, thread-local class indices
  // (fit class = (sel, tol, scalar keys requested with a non-zero amount, core.go:688-690);
  // representative class = (sel, tol)), and the host copies the per-call mirrors read.
  const int T = P < 8192 ? 1 : host_threads();
  struct Part {
    int64_t lo[BS_MAX_LANES], hi[BS_MAX_LANES];
    uint64_t orq[BS_MAX_LANES];
    uint64_t ot = 0, at = ~0ull;
    uint32_t op = 0, apr = ~0u;
    int miss = 0;
    int32_t mg = -1;
    ClassIndex fit, rep;
  };
  std::vector<Part> part(T);
  HP_BEGIN(e);
  e->h_gid.resize(P); e->h_prio.resize(P); e->h_pflags.resize(P);
  BS_DEVICE_GUARD(e);
  CK(cudaEventSynchronize(e->ev_classes));   // the class ids of the previous table are no longer being read
  if (!e->h_pfc.resize(P) || !e->h_prc.resize(P)) return fail(e, BS_E_NOMEM, "pinned host memory");
  // the DMAs go first (asynchronous from pinned tables) and run under the host pass below; a table
  // that then fails validation is dropped (have_pods = false)
  e->have_pods = false;
  e->evaluated = false;
  const uint32_t Pp = std::max(P, 1u);
  int rc;
  if ((rc = upload_lanes(e, e->d_req, t->req, L, P, Pp))) return rc;
  if ((rc = upload_vec(e, e->d_ppres, t->req_present, P, Pp))) return rc;
  if ((rc = upload_vec(e, e->d_gid, t->gid, P, Pp))) return rc;
  if ((rc = upload_vec(e, e->d_prio, t->priority, P, Pp))) return rc;
  if ((rc = upload_vec(e, e->d_ts, t->ts_ns, P, Pp))) return rc;
  if ((rc = upload_vec(e, e->d_pflags, t->flags, P, Pp))) return rc;
  HP(e, "pods:dma-enqueue");
  // T fixed chunks handed out by an omp for: a team smaller than requested still covers every chunk
  const uint32_t chunk = (P + T - 1) / std::max(T, 1);
#pragma omp parallel for schedule(static, 1) num_threads(T)
  for (int tk = 0; tk < T; ++tk) {
    Part& pt = part[tk];
    for (uint32_t d = 0; d < BS_MAX_LANES; ++d) { pt.lo[d] = 0; pt.hi[d] = 0; pt.orq[d] = 0; }
    const uint32_t a0 = std::min(P, (uint32_t)tk * chunk), a1 = std::min(P, a0 + chunk);
    for (uint32_t d = 0; d < L; ++d) {
      const int64_t* row = t->req + (size_t)d * P;
      int64_t lo = 0, hi = 0;
      uint64_t o = 0;
      for (uint32_t p = a0; p < a1; ++p) { lo = std::min(lo, row[p]); hi = std::max(hi, row[p]); o |= (uint64_t)row[p]; }
      pt.lo[d] = lo; pt.hi[d] = hi; pt.orq[d] = o;
    }
    {
      // reductions in locals and the plain column copies as memcpy: a byte store inside the loop would make the
      // compiler spill every accumulator (char stores alias everything)
      uint64_t ot = 0, at = ~0ull;
      uint32_t op = 0, apr = ~0u;
      int miss = 0;
      int32_t mg = -1;
      for (uint32_t p = a0; p < a1; ++p) {
        const uint64_t ts = (uint64_t)t->ts_ns[p];
        const uint32_t pr = (uint32_t)t->priority[p];
        const int32_t g = t->gid[p];
        ot |= ts; at &= ts; op |= pr; apr &= pr;
        miss |= ((g < BS_GID_NONE) || (t->flags[p] & BS_POD_LISTER_MISS)) ? 1 : 0;
        mg = std::max(mg, g);
      }
      pt.ot = ot; pt.at = at; pt.op = op; pt.apr = apr; pt.miss = miss; pt.mg = mg;
      if (a1 > a0) {
        memcpy(e->h_gid.data() + a0, t->gid + a0, (size_t)(a1 - a0) * 4);
        memcpy(e->h_prio.data() + a0, t->priority + a0, (size_t)(a1 - a0) * 4);
        memcpy(e->h_pflags.data() + a0, t->flags + a0, (size_t)(a1 - a0));
      }
    }
    {
      // one index lookup per pod: the representative class of a fit class is looked up once per class
      ClassIndex fit, rep;
      fit.clear();
      rep.clear();
      std::vector<uint32_t> rep_of_fit;
      uint32_t* pfc = e->h_pfc.data();
      uint32_t* prc = e->h_prc.data();
      for (uint32_t p = a0; p < a1; ++p) {
        uint32_t nz = 0;
        const uint32_t rp = t->req_present[p];
        for (uint32_t d = 4; d < L; ++d)
          if (((rp >> d) & 1u) && t->req[(size_t)d * P + p] != 0) nz |= 1u << d;
        const uint32_t af = t->aff_class ? t->aff_class[p] : BS_AFF_NONE;
        const uint32_t fc = fit.get_or_add(ClassKey{t->sel_mask[p], t->tol_mask[p], nz, af});
        if (fc >= rep_of_fit.size()) rep_of_fit.push_back(rep.get_or_add(ClassKey{t->sel_mask[p], t->tol_mask[p], 0u, af}));
        pfc[p] = fc;
        prc[p] = rep_of_fit[fc];
      }
      pt.fit = std::move(fit);
      pt.rep = std::move(rep);
    }
  }
  HP(e, "pods:host-pass");
  int64_t mx_q[BS_MAX_LANES] = {}, neg_q[BS_MAX_LANES] = {};
  uint64_t or_q[BS_MAX_LANES] = {};
  {
    uint64_t ot = 0, at = ~0ull;
    uint32_t op = 0, apr = ~0u;
    int miss = 0;
    int32_t mg = -1;
    bool ok = true;
    for (int k = 0; k < T; ++k) {
      const Part& pt = part[k];
      for (uint32_t d = 0; d < L; ++d) {
        ok = ok && pt.lo[d] >= -BS_VALUE_LIMIT && pt.hi[d] <= BS_VALUE_LIMIT;
        mx_q[d] = std::max(mx_q[d], std::max(pt.hi[d], pt.lo[d] == INT64_MIN ? INT64_MAX : -pt.lo[d]));
        neg_q[d] = std::max(neg_q[d], pt.lo[d] == INT64_MIN ? INT64_MAX : -pt.lo[d]);
        or_q[d] |= pt.orq[d];
      }
      ot |= pt.ot; at &= pt.at; op |= pt.op; apr &= pt.apr; miss |= pt.miss; mg = std::max(mg, pt.mg);
    }
    if (!ok) {   // the device and host-side columns were already overwritten: the table stays dropped
      cudaStreamSynchronize(e->s);
      return fail(e, BS_E_RANGE, "bs_upload_pods: value outside +-2^56");
    }
    e->vary_ts = P ? (ot ^ at) : 0;
    e->vary_prio = P ? (uint64_t)(op ^ apr) : 0;
    e->any_lister_miss = miss != 0;
    e->max_gid = mg;
  }
  // Merge the thread-local class indices into the engine's and remap the ids while the DMA is in
  // flight.  The engine's indices persist across uploads (ids of known classes are stable, so the
  // groups' representative ids stay valid); they restart only when mostly stale.
  {
    size_t lf = 0, lr = 0;
    for (int k = 0; k < T; ++k) { lf += part[k].fit.size(); lr += part[k].rep.size(); }
    if (e->fit_index.size() > std::max<size_t>(4096, 4 * lf)) e->fit_index.clear();
    if (e->rep_index.size() > std::max<size_t>(4096, 4 * lr)) {
      e->rep_index.clear();
      e->group_classes_dirty = true;   // the groups' ids referred to the old index
    }
  }
  {
    std::vector<std::vector<uint32_t>> rf(T), rr(T);
    for (int k = 0; k < T; ++k) {
      rf[k].resize(part[k].fit.size());
      rr[k].resize(part[k].rep.size());
      for (size_t j = 0; j < part[k].fit.size(); ++j) rf[k][j] = e->fit_index.get_or_add(part[k].fit.keys[j]);
      for (size_t j = 0; j < part[k].rep.size(); ++j) rr[k][j] = e->rep_index.get_or_add(part[k].rep.keys[j]);
    }
#pragma omp parallel for schedule(static, 1) num_threads(T)
    for (int k = 0; k < T; ++k) {
      const uint32_t a0 = std::min(P, (uint32_t)k * chunk), a1 = std::min(P, a0 + chunk);
      for (uint32_t p = a0; p < a1; ++p) {
        e->h_pfc[p] = rf[k][e->h_pfc[p]];
        e->h_prc[p] = rr[k][e->h_prc[p]];
      }
    }
  }
  HP(e, "pods:class-merge");
  CK(cudaStreamSynchronize(e->s));
  HP(e, "pods:dma-wait");
  memcpy(e->max_req, mx_q, sizeof(mx_q));
  memcpy(e->neg_req, neg_q, sizeof(neg_q));
  memcpy(e->or_req, or_q, sizeof(or_q));
  e->P = P;
  e->have_pods = true;
  e->classes_dirty = true;
  e->pod_classes_dirty = true;
  e->evaluated = false;
  return BS_OK;
}

int bs_upload_affinity(bs_engine* e, uint32_t n_classes, const uint32_t* bits) {
  if (!e || (n_classes && !bits)) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_nodes) return fail(e, BS_E_STATE, "bs_upload_affinity: upload nodes first");
  BS_DEVICE_GUARD(e);
  const size_t words = (size_t)n_classes * e->W;
  if (words) {
    CK(e->d_aff_bits.ensure(words * 4));
    CK(cudaMemcpyAsync(e->d_aff_bits.p, bits, words * 4, cudaMemcpyHostToDevice, e->s));
    CK(cudaStreamSynchronize(e->s));
  }
  e->n_aff = n_classes;
  e->nodes_dirty = true;     // class-fit bits and cluster scans follow the table
  e->classes_dirty = true;   // class ids are validated against it
  e->evaluated = false;
  return BS_OK;
}

// ---- gang state: the TTL tables around Permit as engine state (gang_state.hpp) ----
int bs_state_reset(bs_engine* e) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_groups) return fail(e, BS_E_STATE, "bs_state_reset: upload groups first");
  e->gang.reset(e->G);
  return BS_OK;
}

int bs_state_remap(bs_engine* e, uint32_t n_groups, const int32_t* old_index) {
  if (!e || (n_groups && !old_index)) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  e->gang.remap(n_groups, old_index);
  return BS_OK;
}

int bs_state_view(bs_engine* e, int64_t now_ns, uint32_t n_groups, uint32_t* matched, uint8_t* flags) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->gang.active || e->gang.groups.size() != n_groups) return fail(e, BS_E_STATE, "bs_state_view: tables of another shape");
  for (uint32_t g = 0; g < n_groups; ++g) {
    if (matched) matched[g] = e->gang.matched_count(g, now_ns);
    if (flags) flags[g] = (uint8_t)((e->gang.groups[g].scheduled ? BS_GROUP_SCHEDULED : 0u) | (e->gang.denied(g, now_ns) ? BS_GROUP_DENIED : 0u));
  }
  return BS_OK;
}

int bs_permitted_view(bs_engine* e, int64_t now_ns, const uint64_t* uids, uint32_t n, uint8_t* out) {
  if (!e || (n && (!uids || !out))) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  for (uint32_t i = 0; i < n; ++i) out[i] = e->gang.active && e->gang.permitted_recently(uids[i], now_ns) ? 1 : 0;
  return BS_OK;
}

int bs_state_move(bs_engine* dst, bs_engine* src) {
  if (!dst || !src || dst == src) return BS_E_INVAL;
  std::lock_guard<std::mutex> l1(src->mu);
  std::lock_guard<std::mutex> l2(dst->mu);
  dst->gang = std::move(src->gang);
  src->gang = GangState();
  return BS_OK;
}

int bs_set_pod_ids(bs_engine* e, const uint64_t* uid, const uint64_t* name_id) {
  if (!e || !uid || !name_id) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_pods) return fail(e, BS_E_STATE, "bs_set_pod_ids: upload pods first");
  e->h_pod_uid.assign(uid, uid + e->P);
  e->h_pod_name.assign(name_id, name_id + e->P);
  return BS_OK;
}

int bs_begin_cycle(bs_engine* e, int64_t now_ns) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_groups || !e->have_pods) return fail(e, BS_E_STATE, "bs_begin_cycle: upload groups and pods first");
  if (!e->gang.active || e->gang.groups.size() != e->G) return fail(e, BS_E_STATE, "bs_begin_cycle: bs_state_reset after the group table changed size");
  BS_DEVICE_GUARD(e);
  const uint32_t G = e->G, P = e->P;
  e->cycle_now_ns = now_ns;
  // the go-cache views at `now` become the columns the round reads: len(MatchedPodNodes.Items()), pgs.Scheduled,
  // lastDeniedPG and lastPermittedPod membership (core.go:95-110,706,711)
  std::vector<uint32_t> matched(G);
  std::vector<uint8_t> gfl(G), pfl(P);
  for (uint32_t g = 0; g < G; ++g) {
    matched[g] = e->gang.matched_count(g, now_ns);
    uint8_t f = e->h_gflags_up[g] & ~(uint8_t)(BS_GROUP_SCHEDULED | BS_GROUP_DENIED);
    if (e->gang.groups[g].scheduled) f |= BS_GROUP_SCHEDULED;
    if (e->gang.denied(g, now_ns)) f |= BS_GROUP_DENIED;
    gfl[g] = f;
  }
  const bool ids = e->h_pod_uid.size() == P && !e->gang.permitted.empty();   // an empty lastPermittedPod: no lookups
  for (uint32_t p = 0; p < P; ++p) {
    uint8_t f = e->h_pflags[p] & ~(uint8_t)BS_POD_PERMITTED_RECENTLY;
    if (ids && e->gang.permitted_recently(e->h_pod_uid[p], now_ns)) f |= BS_POD_PERMITTED_RECENTLY;
    pfl[p] = f;
  }
  if (G) {
    CK(cudaMemcpyAsync(e->d_matched.p, matched.data(), (size_t)G * 4, cudaMemcpyHostToDevice, e->s));
    CK(cudaMemcpyAsync(e->d_gflags.p, gfl.data(), G, cudaMemcpyHostToDevice, e->s));
  }
  if (P) CK(cudaMemcpyAsync(e->d_pflags.p, pfl.data(), P, cudaMemcpyHostToDevice, e->s));
  CK(cudaStreamSynchronize(e->s));
  e->evaluated = false;
  return BS_OK;
}

int bs_permit_at(bs_engine* e, uint32_t pod, uint32_t node, int64_t now_ns, bs_permit_result* r) {
  if (!e || !r) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_pods || !e->have_groups) return fail(e, BS_E_STATE, "bs_permit_at: upload groups and pods first");
  if (pod >= e->P || (e->have_nodes && node >= e->N)) return BS_E_INDEX;
  const int64_t kSecond = 1000000000ll, kDefaultWait = 60 * kSecond;  // util.DefaultWaitTime k8s.go:31
  const int32_t g = e->h_gid[pod];
  memset(r, 0, sizeof(*r));
  r->group = -1;
  if (g == BS_GID_NONE) {  // core.go:270-272 + batchscheduler.go:190-193
    r->ready = 1; r->code = BS_CODE_SUCCESS; r->wait_ns = 0;
    return BS_OK;
  }
  if (g < 0 || (uint32_t)g >= e->G) {  // core.go:275-277 + batchscheduler.go:194-195
    r->ready = 0; r->code = BS_CODE_UNSCHEDULABLE; r->wait_ns = kDefaultWait;
    return BS_OK;
  }
  if (!e->gang.active || e->gang.groups.size() != e->G || e->h_pod_uid.size() != e->P)
    return fail(e, BS_E_STATE, "bs_permit_at: bs_state_reset and bs_set_pod_ids first");
  r->group = g;
  int64_t wait = e->default_wait_ns;   // util.GetWaitTimeDuration (k8s.go:82-91)
  if ((size_t)g < e->h_wait_ns.size() && e->h_wait_ns[g] >= 0) wait = e->h_wait_ns[g];
  const bool ready = e->gang.permit((uint32_t)g, e->h_pod_uid[pod], e->h_pod_name[pod], node, now_ns, wait,
                                    e->h_min_member[g], e->h_scheduled[g]);   // core.go:283-307
  r->wait_ns = wait + kSecond;           // batchscheduler.go:180-182
  r->ready = ready ? 1 : 0;
  r->start_signal = r->ready;            // :197-199
  r->code = BS_CODE_WAIT;                // :184-187 and :201
  return BS_OK;
}

int bs_expire(bs_engine* e, int64_t now_ns, uint32_t* rej_group, uint64_t* rej_uid, uint32_t rej_cap, uint32_t* n_rejected,
              uint32_t* evicted_group, uint32_t evict_cap, uint32_t* n_evicted) {
  if (!e || !n_rejected || !n_evicted) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->gang.active) return fail(e, BS_E_STATE, "bs_expire: bs_state_reset first");
  std::vector<uint32_t> rg, ev;
  std::vector<uint64_t> ru;
  e->gang.expire(now_ns, &rg, &ru, &ev);
  *n_rejected = (uint32_t)rg.size();
  *n_evicted = (uint32_t)ev.size();
  for (uint32_t i = 0; i < rg.size() && i < rej_cap; ++i) {
    if (rej_group) rej_group[i] = rg[i];
    if (rej_uid) rej_uid[i] = ru[i];
  }
  for (uint32_t i = 0; i < ev.size() && i < evict_cap; ++i)
    if (evicted_group) evicted_group[i] = ev[i];
  return BS_OK;
}

int bs_allow_list(bs_engine* e, uint32_t group, int64_t now_ns, uint64_t* uids, uint32_t* nodes, uint32_t cap, uint32_t* n) {
  if (!e || !n) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->gang.active || e->gang.groups.size() != e->G) return fail(e, BS_E_STATE, "bs_allow_list: bs_state_reset first");
  if (group >= e->G) return BS_E_INDEX;
  std::vector<uint64_t> u;
  std::vector<uint32_t> nd;
  e->gang.allow_list(group, now_ns, e->h_min_member[group], e->h_scheduled[group], &u, &nd);
  *n = (uint32_t)u.size();
  for (uint32_t i = 0; i < u.size() && i < cap; ++i) {
    if (uids) uids[i] = u[i];
    if (nodes) nodes[i] = nd[i];
  }
  return BS_OK;
}

int bs_deny(bs_engine* e, uint32_t group, int64_t now_ns) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->gang.active || e->gang.groups.size() != e->G) return fail(e, BS_E_STATE, "bs_deny: bs_state_reset first");
  if (group >= e->G) return BS_E_INDEX;
  e->gang.deny(group, now_ns);
  return BS_OK;
}

int bs_mark_permitted(bs_engine* e, uint64_t uid, int64_t now_ns) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->gang.active) return fail(e, BS_E_STATE, "bs_mark_permitted: bs_state_reset first");
  e->gang.mark_permitted(uid, now_ns);
  return BS_OK;
}

int bs_group_state(bs_engine* e, uint32_t group, int64_t now_ns, uint32_t* matched, int32_t* scheduled_flag, int32_t* denied) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->gang.active || e->gang.groups.size() != e->G) return fail(e, BS_E_STATE, "bs_group_state: bs_state_reset first");
  if (group >= e->G) return BS_E_INDEX;
  if (matched) *matched = e->gang.matched_count(group, now_ns);
  if (scheduled_flag) *scheduled_flag = e->gang.groups[group].scheduled ? 1 : 0;
  if (denied) *denied = e->gang.denied(group, now_ns) ? 1 : 0;
  return BS_OK;
}

int bs_set_wait_time(bs_engine* e, int64_t default_ns, const int64_t* per_group_ns, uint32_t n_groups) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  e->default_wait_ns = default_ns;
  if (per_group_ns) e->h_wait_ns.assign(per_group_ns, per_group_ns + n_groups);
  return BS_OK;
}

int bs_evaluate_async(bs_engine* e) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  return evaluate_async_locked(e);
}

// checks the sticky error word of the peer exchange; on a timeout the exchange is marked broken
static int peer_check_locked(bs_engine* e) {
  if (!e->peer_attached) return BS_OK;
  CK(cudaStreamSynchronize(e->s4));
  int bad = 0;
  CK(cudaMemcpy(&bad, e->d_peer_err.p, sizeof(int), cudaMemcpyDeviceToHost));
  if (bad) {
    e->peer_broken = true;
    return fail(e, BS_E_PEER, "peer exchange timed out: a rank did not arrive (detach and re-attach every rank)");
  }
  return BS_OK;
}

int bs_sync(bs_engine* e) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  CK(cudaStreamSynchronize(e->s));
  return peer_check_locked(e);
}

int bs_fetch(bs_engine* e, bs_results* out) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  return fetch_locked(e, out);
}

int bs_fetch_view(bs_engine* e, bs_results* out) {
  if (!e || !out) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  return fetch_locked(e, out, true);
}

int bs_evaluate_view(bs_engine* e, bs_results* out) {
  if (!e || !out) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  int rc = evaluate_async_locked(e);
  if (rc) return rc;
  BS_DEVICE_GUARD(e);
  return fetch_locked(e, out, true);
}

int bs_evaluate(bs_engine* e, bs_results* out) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  static const bool prof = getenv("BS_HOST_PROFILE") != nullptr;   // host-side stage times on stderr
  const auto t0 = std::chrono::steady_clock::now();
  int rc = evaluate_async_locked(e);
  if (rc) return rc;
  if (!prof) return fetch_locked(e, out);
  const auto t1 = std::chrono::steady_clock::now();
  {
    BS_DEVICE_GUARD(e);
    CK(cudaStreamSynchronize(e->s));
  }
  const auto t2 = std::chrono::steady_clock::now();
  rc = fetch_locked(e, out);
  const auto t3 = std::chrono::steady_clock::now();
  auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double, std::micro>(b - a).count();
  };
  fprintf(stderr, "[bs_evaluate] enqueue %.0f us (classes %.0f us)  device wait %.0f us  fetch %.0f us |", us(t0, t1),
          e->last_classes_us, us(t1, t2), us(t2, t3));
  for (auto& kv : e->hp_log) fprintf(stderr, " %s %.0f", kv.first, kv.second);
  fprintf(stderr, "\n");
  e->hp_log.clear();
  return rc;
}

int bs_prefilter(bs_engine* e, uint32_t pod, bs_status* st) {
  if (!e || !st) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->evaluated) return fail(e, BS_E_STATE, "bs_prefilter: evaluate first");
  if (pod >= e->P) return BS_E_INDEX;
  if (!e->fetched) {
    int rc = fetch_locked(e, nullptr);
    if (rc) return rc;
  }
  const uint8_t reason = e->h_prefilter.as<uint8_t>()[pod];
  st->reason = reason;
  // batchscheduler.go:104-107: nil -> Success, any error -> Unschedulable
  st->code = reason == BS_PF_PASS ? BS_CODE_SUCCESS : BS_CODE_UNSCHEDULABLE;
  const int32_t g = e->h_gid[pod];
  st->group = (g >= 0 && (uint32_t)g < e->G) ? g : -1;
  return BS_OK;
}

int bs_permit(bs_engine* e, uint32_t pod, uint32_t node, bs_permit_result* r) {
  if (!e || !r) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->evaluated) return fail(e, BS_E_STATE, "bs_permit: evaluate first");
  if (pod >= e->P || node >= e->N) return BS_E_INDEX;
  if (!e->fetched) {
    int rc = fetch_locked(e, nullptr);
    if (rc) return rc;
  }
  const int64_t kSecond = 1000000000ll, kDefaultWait = 60 * kSecond;  // util.DefaultWaitTime k8s.go:31
  const int32_t g = e->h_gid[pod];
  memset(r, 0, sizeof(*r));
  r->group = -1;
  if (g == BS_GID_NONE) {  // core.go:270-272 + batchscheduler.go:190-193
    r->ready = 1;
    r->code = BS_CODE_SUCCESS;
    r->wait_ns = 0;
    return BS_OK;
  }
  if (g < 0 || (uint32_t)g >= e->G) {  // core.go:275-277 + batchscheduler.go:194-195
    r->ready = 0;
    r->code = BS_CODE_UNSCHEDULABLE;
    r->wait_ns = kDefaultWait;
    return BS_OK;
  }
  r->group = g;
  // util.GetWaitTimeDuration (k8s.go:82-91) + 1s (batchscheduler.go:180-182)
  int64_t wait = e->default_wait_ns;
  if ((size_t)g < e->h_wait_ns.size() && e->h_wait_ns[g] >= 0) wait = e->h_wait_ns[g];
  r->wait_ns = wait + kSecond;
  const uint8_t a = e->h_admit.as<uint8_t>()[g];
  r->ready = a == BS_ADMIT;              // core.go:303-307
  r->start_signal = r->ready;            // batchscheduler.go:197-199
  r->code = BS_CODE_WAIT;                // :184-187 and :201
  return BS_OK;
}

int bs_less(bs_engine* e, uint32_t a, uint32_t b) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->evaluated) return fail(e, BS_E_STATE, "bs_less: evaluate first");
  if (a >= e->P || b >= e->P) return BS_E_INDEX;
  if (!e->fetched) {
    int rc = fetch_locked(e, nullptr);
    if (rc) return rc;
  }
  // core.go:395-399: at equal priority, two grouped pods where a lister lookup fails
  // compare false both ways; everything else is the rank order of the device sort.
  auto miss = [&](uint32_t p) {
    const int32_t g = e->h_gid[p];
    return g != BS_GID_NONE && (g < 0 || (uint32_t)g >= e->G || (e->h_pflags[p] & BS_POD_LISTER_MISS));
  };
  if (e->h_prio[a] == e->h_prio[b] && e->h_gid[a] != BS_GID_NONE && e->h_gid[b] != BS_GID_NONE &&
      (miss(a) || miss(b)))
    return 0;
  const uint32_t* rank = e->h_rank.as<uint32_t>();
  return rank[a] < rank[b] ? 1 : 0;
}

int bs_format_message(const bs_status* st, const char* ns_name, const char* occupied_by, char* buf,
                      size_t buf_len) {
  if (!st || !buf || !buf_len) return BS_E_INVAL;
  const char* n = ns_name ? ns_name : "";
  const char* o = occupied_by ? occupied_by : "";
  switch (st->reason) {
    case BS_PF_PASS: snprintf(buf, buf_len, "%s", ""); break;
    case BS_PF_ERR_NOT_FOUND: snprintf(buf, buf_len, "can not found pod group: %s", n); break;           // core.go:102
    case BS_PF_ERR_DENIED: snprintf(buf, buf_len, "pod with pgName: %s last failed in 20s, deny", n); break;  // :107
    case BS_PF_ERR_OCCUPIED_NOREFS: snprintf(buf, buf_len, "pod group %s has been occupied by %s", n, o); break;  // :505
    case BS_PF_ERR_OCCUPIED: snprintf(buf, buf_len, "pod group has been occupied by %s", o); break;      // :509
    case BS_PF_ERR_NOT_ENOUGH: snprintf(buf, buf_len, "cluster resource not enough"); break;             // :143,:164
    default: return BS_E_INVAL;
  }
  return BS_OK;
}

int bs_node_left(bs_engine* e, uint64_t sel, uint64_t tol, float percent, int64_t* left, uint32_t* present) {
  if (!e || !left || !present) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_nodes) return fail(e, BS_E_STATE, "bs_node_left: upload nodes first");
  BS_DEVICE_GUARD(e);
  const uint32_t N = e->N, L = e->L;
  if (!N) return BS_OK;
  DevBuf dl, dp;
  CK(dl.ensure((size_t)L * N * 8));
  CK(dp.ensure((size_t)N * 4));
  node_left_class_kernel<<<cdiv(N, 256), 256, 0, e->s>>>(node_tab(e), sel, tol, percent, dl.as<int64_t>(),
                                                         dp.as<uint32_t>());
  e->launches++;
  cudaError_t er = cudaMemcpyAsync(left, dl.p, (size_t)L * N * 8, cudaMemcpyDeviceToHost, e->s);
  if (er == cudaSuccess) er = cudaMemcpyAsync(present, dp.p, (size_t)N * 4, cudaMemcpyDeviceToHost, e->s);
  if (er == cudaSuccess) er = cudaStreamSynchronize(e->s);
  dl.release();
  dp.release();
  CK(er);
  return BS_OK;
}

int bs_cluster_check(bs_engine* e, uint64_t sel, uint64_t tol, float percent, const int64_t* need,
                     const uint32_t* need_present, uint32_t n_needs, uint8_t* ok) {
  if (!e || (n_needs && (!need || !need_present || !ok))) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_nodes) return fail(e, BS_E_STATE, "bs_cluster_check: upload nodes first");
  BS_DEVICE_GUARD(e);
  const uint32_t N = e->N, L = e->L;
  if (!n_needs) return BS_OK;
  if (!N) {
    memset(ok, 0, n_needs);  // empty snapshot list: the loop never runs (core.go:604,631)
    return BS_OK;
  }
  DevBuf pre, pp, stats, dn, dnp, dok, spart, spres, scst, sdone;
  const size_t n_chunks = cdiv(N, PREFIX_CHUNK);
  cudaError_t er = pre.ensure((size_t)L * N * 8);
  if (er == cudaSuccess) er = spart.ensure(n_chunks * BS_MAX_LANES * 8);
  if (er == cudaSuccess) er = spres.ensure(n_chunks * 4);
  if (er == cudaSuccess) er = scst.ensure(n_chunks * sizeof(ClassStats));
  if (er == cudaSuccess) er = sdone.ensure(4);
  if (er == cudaSuccess) er = cudaMemsetAsync(sdone.p, 0, 4, e->s);
  if (er == cudaSuccess) er = pp.ensure((size_t)N * 4);
  if (er == cudaSuccess) er = stats.ensure(sizeof(ClassStats));
  if (er == cudaSuccess) er = dn.ensure((size_t)L * n_needs * 8);
  if (er == cudaSuccess) er = dnp.ensure((size_t)n_needs * 4);
  if (er == cudaSuccess) er = dok.ensure(n_needs);
  if (er == cudaSuccess) er = cudaMemcpyAsync(dn.p, need, (size_t)L * n_needs * 8, cudaMemcpyHostToDevice, e->s);
  if (er == cudaSuccess) er = cudaMemcpyAsync(dnp.p, need_present, (size_t)n_needs * 4, cudaMemcpyHostToDevice, e->s);
  if (er == cudaSuccess) {
    PrefixOut po{pre.as<int64_t>(), pp.as<uint32_t>(), stats.as<ClassStats>()};
    NodeTab t = node_tab(e);
    PrefixSel ps{nullptr, nullptr, nullptr, 0, 2, sel, tol, percent, nullptr};
    PrefixScratch psc{spart.as<int64_t>(), spres.as<uint32_t>(), scst.as<ClassStats>(), sdone.as<uint32_t>()};
    launch_prefix(L, t, ps, psc, po, 1, e->s);
    const uint64_t threads = (uint64_t)n_needs * 32;
    needs_check_kernel<<<(uint32_t)((threads + 255) / 256), 256, 0, e->s>>>(
        t, po, dn.as<int64_t>(), dnp.as<uint32_t>(), n_needs, dok.as<uint8_t>());
    e->launches += 3;
    er = cudaMemcpyAsync(ok, dok.p, n_needs, cudaMemcpyDeviceToHost, e->s);
  }
  if (er == cudaSuccess) er = cudaStreamSynchronize(e->s);
  if (er == cudaSuccess) er = cudaGetLastError();
  pre.release(); pp.release(); stats.release(); dn.release(); dnp.release(); dok.release();
  spart.release(); spres.release(); scst.release(); sdone.release();
  CK(er);
  return BS_OK;
}

int bs_replay(bs_engine* e, const uint32_t* queue, uint32_t n_queue, bs_replay_result* out) {
  if (!e || !out) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_nodes || !e->have_pods || !e->have_groups)
    return fail(e, BS_E_STATE, "bs_replay: upload nodes, groups and pods first");
  BS_DEVICE_GUARD(e);
  const uint32_t N = e->N, Npad = e->Npad, P = e->P, G = e->G, L = e->L;
  if (!queue) n_queue = P;
  if (n_queue && (!out->prefilter || !out->node || !out->ready)) return BS_E_INVAL;
  if (queue)
    for (uint32_t i = 0; i < n_queue; ++i)
      if (queue[i] >= P) return fail(e, BS_E_INDEX, "bs_replay: queue entry is not a pod of the table");
  int rc;
  if (e->classes_dirty && (rc = rebuild_classes(e))) return rc;

  // scratch copies of everything the cycle mutates
  DevBuf &s_req = e->r_req, &s_pc = e->r_pc, &s_rp = e->r_rp, &s_matched = e->r_matched, &s_gflags = e->r_gflags,
         &s_grc = e->r_grc, &s_minres = e->r_minres, &s_mrp = e->r_mrp, &d_queue = e->r_queue, &d_pf = e->r_pf,
         &d_node = e->r_node, &d_ready = e->r_ready, &d_status = e->r_status, &c_sum = e->r_sum, &c_max = e->r_max,
         &c_keys = e->r_keys, &n_left0 = e->r_left0, &n_left1 = e->r_left1, &n_both = e->r_both, &n_fit = e->r_fit,
         &n_stat = e->r_stat;
  const uint32_t Gp = std::max(G, 1u), Qp = std::max(n_queue, 1u);
  cudaError_t er = s_req.ensure((size_t)L * Npad * 8);
  auto dup = [&](DevBuf& dst, const DevBuf& src, size_t bytes) {
    if (er == cudaSuccess) er = dst.ensure(std::max<size_t>(bytes, 4));
    if (er == cudaSuccess && bytes) er = cudaMemcpyAsync(dst.p, src.p, bytes, cudaMemcpyDeviceToDevice, e->s);
  };
  dup(s_req, e->d_requested, (size_t)L * Npad * 8);
  dup(s_pc, e->d_pod_count, (size_t)Npad * 4);
  dup(s_rp, e->d_rpres, (size_t)Npad * 4);
  dup(s_matched, e->d_matched, (size_t)G * 4);
  dup(s_gflags, e->d_gflags, (size_t)G);
  dup(s_grc, e->d_group_rep_class, (size_t)G * 4);
  dup(s_minres, e->d_min_res, (size_t)L * G * 8);
  dup(s_mrp, e->d_mrpres, (size_t)G * 4);
  if (er == cudaSuccess) er = d_queue.ensure((size_t)Qp * 4);
  if (er == cudaSuccess && queue && n_queue)
    er = cudaMemcpyAsync(d_queue.p, queue, (size_t)n_queue * 4, cudaMemcpyHostToDevice, e->s);
  if (er == cudaSuccess) er = d_pf.ensure(Qp);
  if (er == cudaSuccess) er = d_node.ensure((size_t)Qp * 4);
  if (er == cudaSuccess) er = d_ready.ensure(Qp);
  if (er == cudaSuccess) er = d_status.ensure(128);
  if (er == cudaSuccess) er = cudaMemsetAsync(d_status.p, 0, 128, e->s);
  int32_t status = 0;
  if (er == cudaSuccess) {
    ReplayArgs a{};
    a.nt = node_tab(e);
    a.nt.requested = s_req.as<int64_t>();
    a.nt.pod_count = s_pc.as<int32_t>();
    a.nt.req_present = s_rp.as<uint32_t>();
    a.requested = s_req.as<int64_t>();
    a.pod_count = s_pc.as<int32_t>();
    a.req_present = s_rp.as<uint32_t>();
    a.pt = pod_tab(e);
    // compact node state the kernel builds and maintains (replay.cuh)
    er = n_left0.ensure((size_t)L * Npad * 8);
    if (er == cudaSuccess) er = n_left1.ensure((size_t)L * Npad * 8);
    if (er == cudaSuccess) er = n_both.ensure((size_t)Npad * 4);
    if (er == cudaSuccess) er = n_stat.ensure((size_t)Npad);
    if (er == cudaSuccess && e->n_rep_classes <= (uint32_t)REPLAY_MAX_CLASSES) er = n_fit.ensure((size_t)Npad * 4);
    a.left[0] = n_left0.as<int64_t>();
    a.left[1] = n_left1.as<int64_t>();
    a.both = n_both.as<uint32_t>();
    a.nstat = n_stat.as<uint8_t>();
    a.fitmask = e->n_rep_classes <= (uint32_t)REPLAY_MAX_CLASSES ? n_fit.as<uint32_t>() : nullptr;
    a.rsel = e->d_rsel.as<uint64_t>();
    a.rtol = e->d_rtol.as<uint64_t>();
    a.raff = e->d_raff.as<uint32_t>();
    a.n_rep = e->n_rep_classes;
    {
      // block cache of the cluster scan (replay.cuh): every running sum must stay below 2^62.
      // A pod is only assumed where it fits, so a node's `requested` never passes its capacity by
      // more than one request; only negative requests accumulate without that limit.
      long double worst = 0;
      for (uint32_t d = 0; d < L; ++d)
        worst = std::max(worst, (long double)e->max_alloc[d] + (long double)e->max_requested[d] + (long double)e->max_req[d] +
                                    (long double)e->neg_req[d] * (long double)n_queue + (long double)e->max_pod_count + n_queue);
      const bool safe = worst * (long double)std::max(N, 1u) < 4.0e18L;
      const uint32_t n_blocks = cdiv(N, REPLAY_BLOCK);
      const uint32_t maxl = replay_maxl(L);
      a.cache_ok = 0;
      if (er == cudaSuccess && safe && a.n_rep <= (uint32_t)REPLAY_MAX_CLASSES && n_blocks >= 1 && n_blocks <= (uint32_t)REPLAY_MAX_BLOCKS) {
        const size_t rows = (size_t)2 * a.n_rep * n_blocks;
        er = c_sum.ensure(rows * maxl * 8);
        if (er == cudaSuccess) er = c_max.ensure(rows * maxl * 8);
        if (er == cudaSuccess) er = c_keys.ensure(rows * 4);
        a.blk_sum = c_sum.as<int64_t>();
        a.blk_max = c_max.as<int64_t>();
        a.blk_keys = c_keys.as<uint32_t>();
        a.cache_ok = 1;
      }
    }
    a.min_member = e->d_min_member.as<uint32_t>();
    a.scheduled = e->d_scheduled.as<uint32_t>();
    a.matched = s_matched.as<uint32_t>();
    a.gflags = s_gflags.as<uint8_t>();
    a.grc = s_grc.as<uint32_t>();
    a.min_res = s_minres.as<int64_t>();
    a.mrpres = s_mrp.as<uint32_t>();
    a.G = G;
    a.queue = queue ? d_queue.as<uint32_t>() : nullptr;
    a.n_queue = n_queue;
    a.prefilter = d_pf.as<uint8_t>();
    a.node = d_node.as<int32_t>();
    a.ready = d_ready.as<uint8_t>();
    a.status = d_status.as<int32_t>();
    if (er == cudaSuccess) {
      StageTimer tm(e, BS_K_REPLAY, e->s);
      launch_replay(L, a, e->s);
      tm.launched();
      er = cudaGetLastError();
    }
  }
  std::vector<uint32_t> grc;
  auto d2h = [&](void* dst, const DevBuf& src, size_t bytes) {
    if (er == cudaSuccess && dst && bytes) er = cudaMemcpyAsync(dst, src.p, bytes, cudaMemcpyDeviceToHost, e->s);
  };
  d2h(&status, d_status, 4);
#ifdef BS_REPLAY_PROFILE
  long long rp[8] = {};
  d2h(rp, d_status, 0);
  if (er == cudaSuccess) er = cudaMemcpyAsync(rp, (char*)d_status.p + 8, 64, cudaMemcpyDeviceToHost, e->s);
#endif
  d2h(out->prefilter, d_pf, n_queue);
  d2h(out->node, d_node, (size_t)n_queue * 4);
  d2h(out->ready, d_ready, n_queue);
  if (er == cudaSuccess && out->node_requested && N)
    er = cudaMemcpy2DAsync(out->node_requested, (size_t)N * 8, s_req.p, (size_t)Npad * 8, (size_t)N * 8, L,
                           cudaMemcpyDeviceToHost, e->s);
  d2h(out->node_pod_count, s_pc, (size_t)N * 4);
  d2h(out->node_req_present, s_rp, (size_t)N * 4);
  d2h(out->group_matched, s_matched, (size_t)G * 4);
  d2h(out->group_flags, s_gflags, (size_t)G);
  d2h(out->group_min_res, s_minres, (size_t)L * G * 8);
  d2h(out->group_min_res_present, s_mrp, (size_t)G * 4);
  if (out->group_rep_sel || out->group_rep_tol) {
    grc.resize(Gp);
    d2h(grc.data(), s_grc, (size_t)G * 4);
  }
  if (er == cudaSuccess) er = cudaStreamSynchronize(e->s);
  CK(er);
  (void)Gp;
#ifdef BS_REPLAY_PROFILE
  fprintf(stderr, "replay clocks: init %lld pre %lld fill %lld findmax %lld cluster %lld misc %lld firstfit %lld commit %lld\n", rp[7], rp[0], rp[1], rp[2], rp[3], rp[4], rp[5], rp[6]);
#endif
  if (status) return fail(e, BS_E_REF_PANIC, "bs_replay: findMaxPG would divide by MinMember == 0 (core.go:716)");
  for (uint32_t g = 0; g < G && (out->group_rep_sel || out->group_rep_tol); ++g) {
    const ClassKey& k = e->rep_index.keys[grc[g]];
    if (out->group_rep_sel) out->group_rep_sel[g] = k.sel;
    if (out->group_rep_tol) out->group_rep_tol[g] = k.tol;
  }
  return BS_OK;
}

int bs_device_buffer(bs_engine* e, int which, void** dev_ptr, size_t* bytes) {
  if (!e || !dev_ptr || !bytes) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  const uint32_t P = e->P, G = e->G;
  switch (which) {
    case BS_BUF_FIT_BITMAP: *dev_ptr = e->d_fit_bitmap.p; *bytes = (size_t)P * e->bitmap_pitch * 4; break;   // rows of bs_bitmap_pitch words
    case BS_BUF_SCORE: *dev_ptr = e->d_score.p; *bytes = (size_t)P * e->score_pitch * 8; break;   // rows of bs_score_pitch elements
    case BS_BUF_ADMIT_BITMAP: *dev_ptr = e->d_admit_bitmap.p; *bytes = (size_t)cdiv(G, 32) * 4; break;
    case BS_BUF_PREFILTER: *dev_ptr = e->d_prefilter.p; *bytes = P; break;
    case BS_BUF_ADMIT: *dev_ptr = e->d_admit.p; *bytes = G; break;
    case BS_BUF_ORDER: *dev_ptr = e->d_order.p; *bytes = (size_t)P * 4; break;
    case BS_BUF_GATHERED_ADMIT:   // the slot set of the last round (they alternate with the parity of the round number)
      *dev_ptr = e->d_gather.p ? e->d_gather.as<uint32_t>() + (size_t)(e->peer_seq & 1u) * e->peer_world * e->peer_wpr : nullptr;
      *bytes = (size_t)e->peer_world * e->peer_wpr * 4;
      break;
    default: return BS_E_INVAL;
  }
  return BS_OK;
}

void* bs_stream(bs_engine* e) { return e ? (void*)e->s : nullptr; }

uint32_t bs_score_pitch(const bs_engine* e) { return e ? e->score_pitch : 0; }
uint32_t bs_bitmap_pitch(const bs_engine* e) { return e ? e->bitmap_pitch : 0; }

int bs_fetch_fit_rows(bs_engine* e, uint32_t pod0, uint32_t n, uint32_t* words) {
  if (!e || !words) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->evaluated || !(e->out_flags & BS_OUT_FIT_BITMAP)) return fail(e, BS_E_STATE, "no fit bitmap materialised");
  if ((uint64_t)pod0 + n > e->P) return BS_E_INDEX;
  BS_DEVICE_GUARD(e);
  if (n && e->W)
    CK(cudaMemcpy2DAsync(words, (size_t)e->W * 4, e->d_fit_bitmap.as<uint32_t>() + (size_t)pod0 * e->bitmap_pitch,
                         (size_t)e->bitmap_pitch * 4, (size_t)e->W * 4, n, cudaMemcpyDeviceToHost, e->s));
  CK(cudaStreamSynchronize(e->s));
  return BS_OK;
}

int bs_fetch_filter_rows(bs_engine* e, uint32_t pod0, uint32_t n, uint32_t* words) {
  if (!e || !words) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->evaluated || !(e->out_flags & BS_OUT_FILTER)) return fail(e, BS_E_STATE, "no filter matrix materialised");
  if ((uint64_t)pod0 + n > e->P) return BS_E_INDEX;
  BS_DEVICE_GUARD(e);
  if (n && e->W)
    CK(cudaMemcpyAsync(words, e->d_filter_bitmap.as<uint32_t>() + (size_t)pod0 * e->W, (size_t)n * e->W * 4,
                       cudaMemcpyDeviceToHost, e->s));
  CK(cudaStreamSynchronize(e->s));
  return BS_OK;
}

int bs_filter(bs_engine* e, uint32_t pod, uint32_t node, bs_status* st) {
  if (!e || !st) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->evaluated || !(e->out_flags & BS_OUT_FILTER)) return fail(e, BS_E_STATE, "bs_filter: evaluate with BS_OUT_FILTER first");
  if (pod >= e->P || node >= e->N) return BS_E_INDEX;
  if (!e->fetched) {
    int rc = fetch_locked(e, nullptr);
    if (rc) return rc;
  }
  BS_DEVICE_GUARD(e);
  uint32_t word = 0;
  const uint8_t nflag = e->h_nflags[node];
  CK(cudaMemcpyAsync(&word, e->d_filter_bitmap.as<uint32_t>() + (size_t)pod * e->W + (node >> 5), 4,
                     cudaMemcpyDeviceToHost, e->s));
  CK(cudaStreamSynchronize(e->s));
  const int32_t g = e->h_gid[pod];
  st->group = (g >= 0 && (uint32_t)g < e->G) ? g : -1;
  const uint8_t pcode = e->h_filter_code.as<uint8_t>()[pod];
  if ((word >> (node & 31)) & 1u) st->reason = BS_FILTER_PASS;
  else if (pcode != BS_FILTER_PASS) st->reason = pcode;
  else st->reason = (nflag & BS_NODE_NIL) ? BS_FILTER_ERR_NO_SNAPSHOT : BS_FILTER_ERR_NOT_ENOUGH;
  st->code = st->reason == BS_FILTER_PASS ? BS_CODE_SUCCESS : BS_CODE_UNSCHEDULABLE;   // batchscheduler.go:153-156
  return BS_OK;
}

int bs_fetch_score_rows(bs_engine* e, uint32_t pod0, uint32_t n, int64_t* scores) {
  if (!e || !scores) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->evaluated || !(e->out_flags & BS_OUT_SCORE)) return fail(e, BS_E_STATE, "no score matrix materialised");
  if ((uint64_t)pod0 + n > e->P) return BS_E_INDEX;
  BS_DEVICE_GUARD(e);
  if (n && e->N)
    CK(cudaMemcpy2DAsync(scores, (size_t)e->N * 8, e->d_score.as<int64_t>() + (size_t)pod0 * e->score_pitch,
                         (size_t)e->score_pitch * 8, (size_t)e->N * 8, n, cudaMemcpyDeviceToHost, e->s));
  CK(cudaStreamSynchronize(e->s));
  return BS_OK;
}

int bs_peer_init(bs_engine* e, uint32_t rank, uint32_t world, uint32_t words_per_rank) {
  if (!e || world == 0 || world > PEER_MAX_WORLD || rank >= world || words_per_rank == 0) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  if (e->peer_attached) return fail(e, BS_E_STATE, "bs_peer_init: detach first");
  const size_t bytes = peer_buf_words(world, words_per_rank) * 4;
  e->d_gather.release();   // a fresh allocation: the IPC handle names this exact block
  CK(e->d_gather.ensure(bytes));
  CK(e->d_peer_err.ensure(sizeof(int)));
  CK(cudaMemsetAsync(e->d_gather.p, 0, e->d_gather.cap, e->s));
  CK(cudaMemsetAsync(e->d_peer_err.p, 0, sizeof(int), e->s));
  CK(cudaStreamSynchronize(e->s));
  e->peer_rank = rank; e->peer_world = world; e->peer_wpr = words_per_rank; e->peer_seq = 0;
  e->peer_broken = false;
  if (const char* t = getenv("BS_PEER_TIMEOUT_MS")) e->peer_timeout_ns = (unsigned long long)std::max(1, atoi(t)) * 1000000ull;
  return BS_OK;
}

int bs_peer_handle(bs_engine* e, unsigned char handle[64]) {
  if (!e || !handle) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  if (!e->d_gather.p) return fail(e, BS_E_STATE, "bs_peer_handle: bs_peer_init first");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, e->d_gather.p));
  memcpy(handle, &h, 64);
  return BS_OK;
}

int bs_peer_attach(bs_engine* e, const unsigned char* handles) {
  if (!e || !handles) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  if (!e->d_gather.p) return fail(e, BS_E_STATE, "bs_peer_attach: bs_peer_init first");
  if (e->peer_attached) return fail(e, BS_E_STATE, "bs_peer_attach: already attached");
  for (uint32_t r = 0; r < e->peer_world; ++r) {
    if (r == e->peer_rank) { e->peer_ptr[r] = e->d_gather.p; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * 64, 64);
    void* p = nullptr;
    cudaError_t er = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (er != cudaSuccess) {
      for (uint32_t q = 0; q < r; ++q)
        if (q != e->peer_rank && e->peer_ptr[q]) { cudaIpcCloseMemHandle(e->peer_ptr[q]); e->peer_ptr[q] = nullptr; }
      e->err = std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(er);
      cudaGetLastError();
      return BS_E_CUDA;
    }
    e->peer_ptr[r] = p;
  }
  e->peer_attached = true;
  return BS_OK;
}

int bs_peer_detach(bs_engine* e) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  if (e->s) cudaStreamSynchronize(e->s);
  if (e->s4) cudaStreamSynchronize(e->s4);
  for (uint32_t r = 0; r < e->peer_world; ++r) {
    if (r != e->peer_rank && e->peer_ptr[r]) cudaIpcCloseMemHandle(e->peer_ptr[r]);
    e->peer_ptr[r] = nullptr;
  }
  e->peer_attached = false;
  e->peer_broken = false;
  e->peer_seq = 0;
  return BS_OK;
}

int bs_peer_join(bs_engine* e) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  BS_DEVICE_GUARD(e);
  if (e->peer_attached && e->peer_seq) CK(cudaStreamWaitEvent(e->s, e->ev_gath, 0));
  return BS_OK;
}

int bs_fetch_gathered_admit(bs_engine* e, uint32_t* words) {
  if (!e || !words) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->peer_attached || !e->peer_seq) return fail(e, BS_E_STATE, "bs_fetch_gathered_admit: no exchanged round");
  BS_DEVICE_GUARD(e);
  int rc = peer_check_locked(e);   // waits for the round's slots to land (stream s4)
  if (rc) return rc;
  const size_t n = (size_t)e->peer_world * e->peer_wpr;
  CK(cudaMemcpyAsync(words, e->d_gather.as<uint32_t>() + (size_t)(e->peer_seq & 1u) * n, n * 4, cudaMemcpyDeviceToHost, e->s4));
  CK(cudaStreamSynchronize(e->s4));
  return BS_OK;
}

int bs_set_profiling(bs_engine* e, int on) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  e->profiling = on != 0;
  return BS_OK;
}

int bs_kernel_ms(bs_engine* e, int k, float* ms, uint32_t* launches) {
  if (!e || k < 0 || k >= BS_K_COUNT) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (launches) *launches = e->k_launches[k];
  if (ms) {
    *ms = 0.f;
    if (e->profiling && e->k_valid[k]) {
      BS_DEVICE_GUARD(e);
      CK(cudaEventSynchronize(e->ev_b[k]));
      CK(cudaEventElapsedTime(ms, e->ev_a[k], e->ev_b[k]));
    }
  }
  return BS_OK;
}

uint64_t bs_launch_count(const bs_engine* e) { return e ? e->launches : 0; }

int bs_fit_shape(bs_engine* e, uint32_t* wide, uint32_t* narrow, uint32_t* scaled) {
  if (!e) return BS_E_INVAL;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->lane_map_valid) return fail(e, BS_E_STATE, "bs_fit_shape: evaluate first");
  if (wide) *wide = e->lane_map.LW;
  if (narrow) *narrow = e->lane_map.LN;
  if (scaled) *scaled = e->lane_map.LS;
  return BS_OK;
}

}  // extern "C"
