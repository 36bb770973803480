// ust_api.cu — host side of libust.so: the C ABI of include/ust.h over the kernels of ust_kernels.cu.
// No node is ever evaluated on the CPU here; without an sm_100 device every computing call fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types only; the library is resolved with dlopen when ust_comm_init is called

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <mutex>
#include <string>
#include <vector>

#include "ust_dev.h"

namespace {

thread_local std::string g_create_error;

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool load(std::string* err) {
    if (lib) return true;
    // prefer a copy already mapped into the process (e.g. the one PyTorch ships), then the system one
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL | RTLD_NOLOAD);
      if (lib) break;
    }
    for (const char* n : names) {
      if (lib) break;
      lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    }
    if (!lib) { *err = std::string("cannot load libnccl: ") + dlerror(); return false; }
    GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
    AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
    AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
    CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
    GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
    if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) { *err = "libnccl lacks required symbols"; return false; }
    return true;
  }
};
NcclApi g_nccl;
std::mutex g_nccl_mu;

// A device array that grows and is freed with its owner. Growing frees the old array at once: nothing may still use it.
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;  // elements
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    size_t want = cap ? cap : 1024;
    while (want < n) want += want / 2 + 1024;  // geometric growth
    return resize(want);
  }
  // exactly n elements; the contents are not kept
  cudaError_t resize(size_t n) {
    T* q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T));
    if (e != cudaSuccess) return e;
    if (p) cudaFree(p);
    p = q;
    cap = n;
    return cudaSuccess;
  }
};

// A CUDA resource of fixed size (device or pinned allocation, stream, event) that `Free` releases with its owner.
// It reads as the raw handle.
template <class T, auto Free>
struct Owned {
  T p{};
  Owned() = default;
  Owned(const Owned&) = delete;
  Owned& operator=(const Owned&) = delete;
  ~Owned() { if (p) Free(p); }
  operator T() const { return p; }
  T operator->() const { return p; }
};
template <class T> using DevPtr = Owned<T*, cudaFree>;
template <class T> using PinnedPtr = Owned<T*, cudaFreeHost>;
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;

}  // namespace

struct ust_handle {
  int device = -1;
  Stream stream;
  Stream stream_d2h;   // pipelined host path: downloads, kernels and uploads on three streams
  Stream stream_h2d;
  Event seg_done[16];
  Event seg_up[16];
  Event d2h_done;
  std::mutex mu;
  std::string err;
  int64_t launches = 0;
  int num_sms = 0;
  bool ws_dirty = false;
  bool pdl = true;          // launch the kernels of a call with programmatic dependent launch (UST_PDL=0 turns it off: tuning)
  bool stamps = false;      // UST_STAMPS: per-CTA %globaltimer stamps (diagnostics)
  int static_pct = 75;      // share of a launch's tile rounds taken in stride order before the ticket (UST_STATIC_PCT: tuning)
  unsigned call_seq = 0;    // calls whose kernels were launched: call k uses accumulator set k & 1 of the workspace
  // the previous call's buffers, when its kernels are the last thing enqueued on the handle's own stream (else n = -1):
  // a call that touches none of them does not wait for it (UstParams::relaxed)
  struct Span { const char* p; size_t len; };
  Span prev_in[4] = {}, prev_out[3] = {};
  int64_t prev_n = -1;
  int64_t relaxed_calls = 0;   // diagnostics
  bool overlap_calls = true;  // UST_OVERLAP=0 turns the overlap of independent back-to-back calls off (tuning)
  cudaStream_t last_stream = nullptr;  // stream of the previous device-resident call (calls on another stream are ordered behind it)
  int64_t resident_n = -1;  // nodes of the snapshot the last ust_apply_state left in the staging arrays (-1 = none)
  int32_t resident_n_ds = 0;  // ... and the size of its DaemonSet table
  DevBuf<ust_counters> hist;  // rollout simulation: one ust_counters per simulated reconcile
  int segments = 6;      // upload / compute / download pipeline depth of the host path (UST_SEGMENTS, tuning)
  bool no_hint = false;  // UST_NO_HINT=1 (tuning): every call speculates from the policy default, never from the previous call

  DevPtr<UstWorkspace> ws;
  DevPtr<uint32_t> lut_dev;         // UST_LUT_WORDS words
  DevPtr<uint8_t> podlut_dev;
  PinnedPtr<uint32_t> lut_host;     // staging copy
  PinnedPtr<uint8_t> podlut_host;
  ust_policy lut_policy;            // policy the device tables were built for
  bool lut_valid = false;
  DevPtr<ust_counters> counters_dev;
  PinnedPtr<ust_counters> counters_host;
  DevPtr<long long> xchg_dev;
  DevBuf<unsigned long long> ds_count;  // BuildState: pods per DaemonSet (zeroed whenever it is reallocated)

  // staging for the host-pointer API
  DevBuf<uint8_t> s_hot, s_next, s_outcome;
  DevBuf<uint32_t> s_flags;
  DevBuf<int32_t> s_rev, s_ds, s_dsrev, s_podoff, s_dsdesired;
  DevBuf<uint16_t> s_rev16;          // packed host format: interned pod revisions / DaemonSet indices as uploaded
  DevBuf<int8_t> s_ds8;
  DevBuf<uint16_t> s_actions, s_podflags;
  DevBuf<uint8_t> s_podsum;
  DevBuf<unsigned int> s_candtile[2];   // upgrade candidates per tile of the current call (by call parity: the previous
                                        // call's verification kernel may still be reading its own)
  // sparse delta outputs: the previous call's outputs, block counts, compacted entries
  DevBuf<uint8_t> s_next_prev, sp_next;
  DevBuf<uint16_t> s_actions_prev, sp_actions;
  DevBuf<unsigned int> sp_blocks;
  DevBuf<long long> sp_idx;
  DevPtr<long long> sp_count_dev;
  PinnedPtr<long long> sp_count_host;
  bool outputs_resident = false;       // s_next / s_actions hold the outputs of the last call on the resident snapshot
  DevBuf<uint64_t> s_uid, s_dsuid;   // BuildState owner join: pod owner UIDs, DaemonSet UID hash table (+ s_dsorder: slot -> index)
  DevBuf<int32_t> s_dsorder;
  DevBuf<long long> d_idx;           // delta updates: indices and values of the changed nodes
  DevBuf<uint8_t> d_state;
  DevBuf<uint32_t> d_flags;
  DevBuf<int32_t> d_rev, d_ds;
  DevBuf<int32_t> sim_entered, sim_wait, sim_valid;  // timed rollout simulation: per-node clocks

  // multi-GPU
  int rank = 0, world = 1, comm_mode = 0;
  ncclComm_t comm = nullptr;
  // fused exchange: own mailbox + the peers' mailboxes mapped through CUDA IPC
  DevPtr<UstMailbox> mbox_own;
  UstMailbox* mbox[UST_MAX_WORLD] = {};
  bool mbox_ready = false;
  long long epoch = 0;

  int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    err = buf;
    return code;
  }
};

#define UST_CUDA(h, call)                                                                                   \
  do {                                                                                                      \
    cudaError_t e_ = (call);                                                                                \
    if (e_ != cudaSuccess) return (h)->fail(UST_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

static bool policy_active(const ust_policy* p) { return p != nullptr && p->auto_upgrade != 0; }

// tables depend on these fields only
static ust_policy table_key(const ust_policy* p) {
  ust_policy k;
  memset(&k, 0, sizeof(k));
  if (!policy_active(p)) return k;  // all-noop tables
  k = *p;
  k.max_parallel_upgrades = 0;
  k.max_unavailable_kind = 0;
  k.max_unavailable_value = 0;
  return k;
}

static int ensure_tables(ust_handle* h, const ust_policy* p, cudaStream_t st) {
  const ust_policy key = table_key(p);
  if (h->lut_valid && memcmp(&key, &h->lut_policy, sizeof(key)) == 0) return UST_OK;
  UST_CUDA(h, cudaStreamSynchronize(st));  // the pinned staging copy may still be in flight
  if (policy_active(p)) {
    ust_build_lut(&key, h->lut_host);
    ust_build_pod_lut256(&key, h->podlut_host);
  } else {
    ust_build_lut(nullptr, h->lut_host);
    memset(h->podlut_host, 0, UST_PODLUT_ENTRIES);
  }
  UST_CUDA(h, cudaMemcpyAsync(h->lut_dev, h->lut_host, UST_LUT_WORDS * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  UST_CUDA(h, cudaMemcpyAsync(h->podlut_dev, h->podlut_host, UST_PODLUT_ENTRIES, cudaMemcpyHostToDevice, st));
  h->lut_policy = key;
  h->lut_valid = true;
  return UST_OK;
}

// Tiling of a shard: tiles of UST_TILE_NODES nodes; smaller tiles (halved, multiples of 128) when the snapshot is so small that
// full-size tiles would leave SMs without work. One persistent CTA per SM, never more CTAs than tiles.
static int pick_tile_nodes(const ust_handle* h, int64_t n) {
  int tn = UST_TILE_NODES;
  // at least one tile per SM; a CTA keeps up to UST_STAGES tiles in flight at once, so a small snapshot is one load
  // round trip whatever its tile size - and larger tiles mean larger (more efficient) bulk copies
  while (tn > 128 && n / tn < (int64_t)h->num_sms) { tn = (tn / 2) & ~127; if (tn < 128) tn = 128; }  // multiples of 128 nodes
  return tn;
}
static int pick_grid(const ust_handle* h, int tiles) {
  const int g = tiles < h->num_sms ? tiles : h->num_sms;
  return g < 1 ? 1 : g;
}
// rounds of a launch's tile range that a CTA takes in stride order before it starts claiming tiles by ticket
static int pick_static_rounds(const ust_handle* h, int tiles, int grid) {
  const int rounds = tiles / grid;
  int r = (int)((int64_t)rounds * h->static_pct / 100);
  if (rounds - r < 2) r = rounds - 2;
  if (r < 1 && rounds >= 1) r = 1;  // the first round never waits for a ticket
  return r < 0 ? 0 : r;
}

static int check_aligned(ust_handle* h, const void* p, const char* what) {
  if (((uintptr_t)p & 15u) != 0) return h->fail(UST_ERR_INVALID_ARGUMENT, "%s must be 16-byte aligned", what);
  return UST_OK;
}

// Everything a call does before its streaming launches: order it behind the previous call, reset the workspace, build
// the tables, fill the launch parameters, launch the pod summary (pod lists only) and give the call its collective
// number and accumulator parity. The number is taken after the pod-summary launch: a call that fails before it leaves
// epoch and call_seq as they were.
static int begin_call(ust_handle* h, const ust_policy* policy, cudaStream_t st, int64_t n, const uint8_t* state,
                      const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx, int32_t n_ds, const int32_t* ds_rev,
                      const int32_t* pod_off, const uint16_t* pod_flags, int64_t n_pods, uint8_t* next_state, uint16_t* actions,
                      uint8_t* outcome, ust_counters* out_dev, UstParams* out, int* grid_out) {
  // a handle's workspace, tables and counters serve one call at a time: a call on another stream than the previous
  // one is ordered behind it (calls on the same stream are ordered by the stream)
  if (h->last_stream && h->last_stream != st) UST_CUDA(h, cudaStreamSynchronize(h->last_stream));
  h->last_stream = st;
  if (h->ws_dirty) {
    UST_CUDA(h, cudaMemsetAsync(h->ws, 0, sizeof(UstWorkspace), st));
    h->ws_dirty = false;
  }
  int rc = ensure_tables(h, policy, st);
  if (rc) return rc;

  const bool active = policy_active(policy);
  UstParams P;
  memset(&P, 0, sizeof(P));
  P.n = n;
  P.hot = state; P.flags = flags; P.pod_rev = pod_rev; P.ds_idx = ds_idx;
  P.ds_rev = ds_rev; P.n_ds = n_ds;
  P.pod_off = pod_off; P.pod_flags = pod_flags;
  P.next = next_state; P.actions = actions; P.outcome = outcome;
  P.lut = h->lut_dev; P.podlut = h->podlut_dev;
  P.ws = h->ws; P.xchg = h->xchg_dev;
  P.out = out_dev ? out_dev : h->counters_dev;
  P.active = active ? 1 : 0;
  if (active) {
    P.max_parallel = policy->max_parallel_upgrades;
    P.max_unav_value = policy->max_unavailable_value;
    P.max_unav_kind = policy->max_unavailable_kind;
    P.requestor = policy->use_maintenance_operator != 0;
    P.pd_enabled = policy->pod_deletion_enabled != 0;
    P.pd_spec_present = policy->pod_deletion_spec_present != 0;
    // pod lists given (even empty ones: "no pods" is an answer, not "unknown") and actuator evaluation asked for
    P.eval_pods = (policy->evaluate_actuators != 0 && pod_off) ? 1 : 0;
  }
  P.rank = h->rank;
  P.world = h->world;
  if (h->world > 1 && h->comm_mode == 1 && h->mbox_ready) {
    P.fused_exchange = 1;
    for (int r = 0; r < h->world; r++) P.mbox[r] = h->mbox[r];
  }
  P.split = (h->world > 1 && !P.fused_exchange) ? 1 : 0;
  // Speculative slot grant (verified by the call's last CTA, so only speed depends on it):
  // with no MaxParallelUpgrades / MaxUnavailable limit every candidate gets a slot (upgrade_inplace.go:49-62);
  // with limits the budget is normally tiny next to the number of candidates.
  P.spec_cut_tile = (active && policy->max_parallel_upgrades == 0 && policy->max_unavailable_kind == UST_MAXUNAVAIL_NIL) ? 0x7FFFFFFF : 0;
  const int tn = pick_tile_nodes(h, n);
  const int64_t tiles64 = (n + tn - 1) / tn;
  const int tiles = (int)tiles64;
  const int grid = pick_grid(h, tiles);
  if (active && !P.requestor && !h->no_hint) {
    // signature of everything the cut position depends on besides the data itself (FNV-1a)
    unsigned long long sig = 1469598103934665603ull;
    const long long parts[6] = {n, tn, policy->max_parallel_upgrades, policy->max_unavailable_kind, policy->max_unavailable_value, h->world * 64 + h->rank};
    for (long long v : parts) { sig ^= (unsigned long long)v; sig *= 1099511628211ull; }
    P.spec_sig = sig ? sig : 1;
  }
  P.tile_nodes = tn;
  P.n_tiles = tiles;
  P.tile_begin = 0;
  P.tile_end = tiles;
  P.static_rounds = pick_static_rounds(h, tiles, grid);
  P.publish = 1;
  P.stamps = (h->stamps && grid <= UST_MAX_CTAS) ? 1 : 0;
  for (auto& b : h->s_candtile) {
    // growing a buffer frees the old one: nothing of an earlier call may still be using it
    if ((size_t)tiles + 1 > b.cap && h->last_stream) cudaStreamSynchronize(h->last_stream);
    cudaError_t ce = b.reserve((size_t)tiles + 1);
    if (ce != cudaSuccess) return h->fail(UST_ERR_CUDA, "cudaMalloc failed: %s", cudaGetErrorString(ce));
  }

  h->ws_dirty = true;  // cleared again once every launch of this call has been enqueued successfully
  if (P.eval_pods) {
    // pod lists: one byte per node first (only the nodes whose actuator looks at its pods are read),
    // then the ordinary streaming pass with that byte as a fifth input stream
    UST_CUDA(h, h->s_podsum.reserve((size_t)n + 16));
    P.podsum = h->s_podsum.p;
    int e = ust_launch_pod_summary(n, P.active, P.hot, P.pod_off, P.pod_flags, n_pods, P.podlut, P.podsum, h->num_sms * 6, st);
    if (e) return h->fail(UST_ERR_CUDA, "pod-summary kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    h->launches += 1;
  }
  if (P.fused_exchange) P.epoch = ++h->epoch;  // collective call number: identical on every rank
  P.parity = (int)(h->call_seq++ & 1u);
  P.cand_tile = h->s_candtile[P.parity].p;
  *out = P;
  *grid_out = grid;
  return UST_OK;
}

// the verification kernel behind the streaming launches of a call (+ the collective, split mode)
static int launch_verify(ust_handle* h, UstParams& P, cudaStream_t st, bool pdl) {
  if (P.split) {
    ncclResult_t r = g_nccl.AllReduce(h->xchg_dev, h->xchg_dev, UST_V_LEN, ncclInt64, ncclSum, h->comm, st);
    if (r != ncclSuccess) return h->fail(UST_ERR_COMM, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  }
  int e = ust_launch_verify(P, h->num_sms, st, (pdl && !P.split) ? 1 : 0);
  if (e) return h->fail(UST_ERR_CUDA, "verification kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
  h->launches += 1;
  return UST_OK;
}

// The pod CSR must be well-formed before a kernel walks it: pod_off[0] == 0, non-decreasing, pod_off[n] == n_pods.
static int check_pod_offsets_host(ust_handle* h, int64_t n, const int32_t* pod_off, int64_t n_pods) {
  if (n == 0) return UST_OK;
  if (pod_off[0] != 0) return h->fail(UST_ERR_INVALID_ARGUMENT, "pod_off[0] must be 0");
  for (int64_t i = 0; i < n; i++)
    if (pod_off[i + 1] < pod_off[i]) return h->fail(UST_ERR_INVALID_ARGUMENT, "pod_off must not decrease (node %lld)", (long long)i);
  if ((int64_t)pod_off[n] != n_pods) return h->fail(UST_ERR_INVALID_ARGUMENT, "pod_off[n_nodes] must equal n_pods");
  return UST_OK;
}

// core: everything device-resident, enqueue on `st`. `chain`: called by ust_apply_state_device, whose calls may
// overlap the previous one.
static int apply_device(ust_handle* h, bool chain, const ust_policy* policy, int64_t n, const uint8_t* state,
                        const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx, int32_t n_ds, const int32_t* ds_rev,
                        const int32_t* pod_off, const uint16_t* pod_flags, int64_t n_pods, uint8_t* next_state,
                        uint16_t* actions, uint8_t* outcome, ust_counters* out_dev, cudaStream_t st) {
  if (n < 0) return h->fail(UST_ERR_NIL_STATE, "currentState should not be empty");
  if (n > 0 && (!state || !flags || !pod_rev || !ds_idx || !next_state || !actions))
    return h->fail(UST_ERR_NIL_STATE, "currentState should not be empty");
  if (n_ds < 0 || (n_ds > 0 && !ds_rev)) return h->fail(UST_ERR_INVALID_ARGUMENT, "bad DaemonSet table");
  if (n >= (1LL << 40)) return h->fail(UST_ERR_INVALID_ARGUMENT, "too many nodes");
  const void* ptrs[] = {state, flags, pod_rev, ds_idx, next_state, actions, outcome};
  const char* names[] = {"state", "flags", "pod_rev", "ds_idx", "next_state", "actions", "actuator_outcome"};
  for (int i = 0; i < 7; i++)
    if (ptrs[i]) { int rc = check_aligned(h, ptrs[i], names[i]); if (rc) return rc; }
  if (pod_off && pod_flags) { int rc = check_aligned(h, pod_flags, "pod_flags"); if (rc) return rc; }
  UST_CUDA(h, cudaSetDevice(h->device));
  UstParams P;
  int grid = 0;
  int rc = begin_call(h, policy, st, n, state, flags, pod_rev, ds_idx, n_ds, ds_rev, pod_off, pod_flags, n_pods, next_state,
                      actions, outcome, out_dev, &P, &grid);
  if (rc) return rc;
  // Independent back-to-back calls overlap: when the last thing enqueued on the handle's own stream is the previous
  // call's verification kernel and this call reads nothing that call writes and writes nothing that call reads or
  // writes, its streaming kernel does not wait for it (programmatic dependent launch without the initial wait: the
  // CTAs of this call take over the SMs as the CTAs of that one run out of tiles, and that call's decision and exchange
  // run beside them). Everything else - another stream, pod lists, shared output arrays - keeps the strict order.
  ust_handle::Span in[4] = {{(const char*)state, (size_t)n}, {(const char*)flags, (size_t)n * 4}, {(const char*)pod_rev, (size_t)n * 4},
                            {(const char*)ds_idx, (size_t)n * 4}};
  ust_handle::Span outs[3] = {{(const char*)next_state, (size_t)n}, {(const char*)actions, (size_t)n * 2},
                             {(const char*)outcome, outcome ? (size_t)n : 0}};
  auto overlaps = [](const ust_handle::Span& a, const ust_handle::Span& b) {
    return a.len && b.len && a.p < b.p + b.len && b.p < a.p + a.len;
  };
  bool relaxed = chain && h->pdl && h->overlap_calls && st == h->stream && h->prev_n >= 0 && !P.eval_pods && !P.split;
  for (int i = 0; relaxed && i < 3; i++) {
    for (int j = 0; j < 3; j++) relaxed = relaxed && !overlaps(outs[i], h->prev_out[j]);   // write / write
    for (int j = 0; j < 4; j++) relaxed = relaxed && !overlaps(outs[i], h->prev_in[j]);    // write / read (that call's redo)
  }
  for (int i = 0; relaxed && i < 4; i++)
    for (int j = 0; j < 3; j++) relaxed = relaxed && !overlaps(in[i], h->prev_out[j]);     // read / write
  P.relaxed = relaxed ? 1 : 0;
  h->relaxed_calls += relaxed ? 1 : 0;
  if (relaxed) P.static_rounds = P.n_tiles / grid + 3;  // no tickets: a CTA's tiles are fixed, the next call fills the tail
  h->prev_n = -1;
  int e = ust_launch_stream(P, grid, st, h->pdl ? 1 : 0);
  if (e) return h->fail(UST_ERR_CUDA, "streaming kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
  h->launches += 1;
  rc = launch_verify(h, P, st, h->pdl);
  if (rc) return rc;
  h->ws_dirty = false;
  if (chain && st == h->stream && !P.eval_pods) {
    for (int i = 0; i < 4; i++) h->prev_in[i] = in[i];
    for (int i = 0; i < 3; i++) h->prev_out[i] = outs[i];
    h->prev_n = n;
  }
  return UST_OK;
}

static int finish_with_counters(ust_handle* h, cudaStream_t st, ust_counters* out, bool fetched = false) {
  if (!fetched) UST_CUDA(h, cudaMemcpyAsync(h->counters_host, h->counters_dev, sizeof(ust_counters), cudaMemcpyDeviceToHost, st));
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    h->ws_dirty = true;
    return h->fail(UST_ERR_CUDA, "kernel execution failed: %s", cudaGetErrorString(e));
  }
  if (out) *out = *h->counters_host;
  const int code = (int)h->counters_host->error_code;
  if (code != UST_OK) {
    switch (code) {
      case UST_ERR_REVISION_HASH:
        return h->fail(code, "failed to get daemonset template/pod revision hash (node index %lld, pass %lld)",
                       (long long)h->counters_host->error_index, (long long)h->counters_host->error_pass);
      case UST_ERR_MAX_UNAVAILABLE: return h->fail(code, "failed to compute maxUnavailable from the current total nodes");
      case UST_ERR_POD_DELETION_SPEC: return h->fail(code, "pod deletion spec should not be empty");
      case UST_ERR_DS_UNSCHEDULED: return h->fail(code, "driver DaemonSet should not have Unscheduled pods");
      case UST_ERR_COMM: return h->fail(code, "multi-GPU exchange timed out: a peer rank did not take part in the call");
      default: return h->fail(code, "ApplyState aborted with code %d", code);
    }
  }
  return UST_OK;
}

static void drain_streams(ust_handle* h) {
  if (h->stream_h2d) cudaStreamSynchronize(h->stream_h2d);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->stream_d2h) cudaStreamSynchronize(h->stream_d2h);
}

// Host-pointer entry points hand caller-owned buffers to asynchronous copies: whatever way such a call ends, nothing
// of it may still be in flight when it returns (the caller may free or reuse the buffers).
struct StreamDrain {
  ust_handle* h;
  explicit StreamDrain(ust_handle* hh) : h(hh) {}
  ~StreamDrain() { drain_streams(h); }
};

// Every entry point that takes a handle starts with UST_ENTER (after checks that touch nothing): one call at a time
// per handle, and whatever the call enqueues sits between two device calls, which therefore keep the strict order.
// Only ust_apply_state_device continues the overlap chain (chain = true).
struct CallGuard {
  std::lock_guard<std::mutex> lock;
  CallGuard(ust_handle* h, bool chain) : lock(h->mu) { if (!chain) h->prev_n = -1; }
};
#define UST_ENTER(h)                          \
  if (!(h)) return UST_ERR_INVALID_ARGUMENT; \
  CallGuard call_guard_((h), false)

// The resident snapshot: the staging arrays hold a snapshot that the delta calls, ust_fetch_outputs and the rollout
// simulation may use. A call that stages into those arrays drops it first.
static void drop_resident(ust_handle* h) {
  h->resident_n = -1;
  h->outputs_resident = false;
}
// Whether the snapshot a call has staged survives the call's return code: it does unless the call itself failed (CUDA,
// the multi-GPU exchange). A reference-level abort (UST_ERR_REVISION_HASH, _MAX_UNAVAILABLE, _POD_DELETION_SPEC) is an
// answer about the data and keeps it. Argument errors are returned before anything is staged or dropped: they leave the
// previous snapshot as it was and never reach this rule.
static bool snapshot_survives(int rc) { return rc != UST_ERR_CUDA && rc != UST_ERR_COMM; }
static int keep_resident(ust_handle* h, int rc, int64_t n, int32_t n_ds) {
  if (snapshot_survives(rc)) {
    h->resident_n = n;
    h->resident_n_ds = n_ds;
    h->outputs_resident = true;
  }
  return rc;
}

// The dense outputs of nodes [n0, n0 + len) from the staging arrays to the caller's (actuator outcomes when asked for).
static int download_outputs(ust_handle* h, int64_t n0, size_t len, uint8_t* next_state, uint16_t* actions, uint8_t* outcome,
                            cudaStream_t st) {
  if (!len) return UST_OK;
  UST_CUDA(h, cudaMemcpyAsync(next_state + n0, h->s_next.p + n0, len, cudaMemcpyDeviceToHost, st));
  UST_CUDA(h, cudaMemcpyAsync(actions + n0, h->s_actions.p + n0, len * 2, cudaMemcpyDeviceToHost, st));
  if (outcome) UST_CUDA(h, cudaMemcpyAsync(outcome + n0, h->s_outcome.p + n0, len, cudaMemcpyDeviceToHost, st));
  return UST_OK;
}

// The node columns of a host-staged ApplyState: wide (int32 pod_rev / ds_idx, as the kernels read them) or packed
// (uint16 rev16 / int8 ds8: 3 instead of 8 bytes per node over PCIe, widened on the device).
struct HostNodes {
  ust_handle* h;
  bool packed;
  const uint8_t* state;
  const uint32_t* flags;
  const int32_t* pod_rev;
  const int32_t* ds_idx;
  const uint16_t* rev16;
  const int8_t* ds8;

  // copies nodes [n0, n0 + len) into the staging arrays
  int upload_nodes(int64_t n0, size_t len, cudaStream_t st) const {
    if (!len) return UST_OK;
    UST_CUDA(h, cudaMemcpyAsync(h->s_hot.p + n0, state + n0, len, cudaMemcpyHostToDevice, st));
    UST_CUDA(h, cudaMemcpyAsync(h->s_flags.p + n0, flags + n0, len * 4, cudaMemcpyHostToDevice, st));
    if (packed) {
      UST_CUDA(h, cudaMemcpyAsync(h->s_rev16.p + n0, rev16 + n0, len * 2, cudaMemcpyHostToDevice, st));
      UST_CUDA(h, cudaMemcpyAsync(h->s_ds8.p + n0, ds8 + n0, len, cudaMemcpyHostToDevice, st));
    } else {
      UST_CUDA(h, cudaMemcpyAsync(h->s_rev.p + n0, pod_rev + n0, len * 4, cudaMemcpyHostToDevice, st));
      UST_CUDA(h, cudaMemcpyAsync(h->s_ds.p + n0, ds_idx + n0, len * 4, cudaMemcpyHostToDevice, st));
    }
    return UST_OK;
  }
  // packed: widens the uploaded nodes [n0, n0 + len) into the int32 staging arrays
  int widen_nodes(int64_t n0, size_t len, cudaStream_t st) const {
    if (!packed || !len) return UST_OK;
    int e = ust_launch_widen((long long)len, h->s_rev16.p + n0, h->s_ds8.p + n0, h->s_rev.p + n0, h->s_ds.p + n0, 4 * h->num_sms, st);
    if (e) return h->fail(UST_ERR_CUDA, "widen kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    h->launches += 1;
    return UST_OK;
  }
};

// Pipelined host path: the snapshot is cut into segments of whole tiles; segment s+1 uploads while segment
// s streams through the kernel and segment s-1's results download (PCIe is full duplex). The streaming pass
// is speculative, so a segment's outputs are final unless the end-of-call verification had to redo tiles —
// then (rare) the outputs are downloaded again.
static int apply_pipelined(ust_handle* h, const HostNodes& nodes, const ust_policy* policy, int64_t n, int32_t n_ds,
                           uint8_t* next_state, uint16_t* actions, uint8_t* outcome, ust_counters* out) {
  cudaStream_t up = h->stream, down = h->stream_d2h, h2d = h->stream_h2d;  // up = compute stream of the call
  UstParams P;
  int grid = 0;
  int rc = begin_call(h, policy, up, n, h->s_hot.p, h->s_flags.p, h->s_rev.p, h->s_ds.p, n_ds, h->s_dsrev.p, nullptr, nullptr, 0,
                      h->s_next.p, h->s_actions.p, outcome ? h->s_outcome.p : nullptr, nullptr, &P, &grid);
  if (rc) return rc;
  const int tiles = P.n_tiles;
  // Segments: the uploads are the critical path (PCIe), every segment costs ~25 us of copy-engine turnarounds (measured:
  // 6 / 8 / 12 / 16 segments -> 1.80 / 1.87 / 1.95 / 2.06 ms at 10 M nodes), and what follows the last upload - its
  // kernels and the download of its outputs - is exposed. So: few segments, and a last one of 1/16 of the tiles.
  const int kSegments = h->segments;  // <= UST_MAX_SEGMENTS: one ticket counter and one event pair per streaming launch
  const int last_tiles = (kSegments > 1 && tiles >= 64) ? tiles / 16 : 0;
  const int per = last_tiles ? (tiles - last_tiles + kSegments - 2) / (kSegments - 1) : (tiles + kSegments - 1) / kSegments;
  // uploads start once the compute stream has reached this call (tables, DaemonSet table, previous call's reads)
  UST_CUDA(h, cudaEventRecord(h->d2h_done, up));
  UST_CUDA(h, cudaStreamWaitEvent(h2d, h->d2h_done, 0));
  int seg = 0;
  for (int c0 = 0, c1 = 0; c0 < tiles; c0 = c1, seg++) {
    c1 = c0 + per < tiles - last_tiles ? c0 + per : (c0 < tiles - last_tiles ? tiles - last_tiles : tiles);
    const int64_t n0 = (int64_t)c0 * P.tile_nodes, n1 = c1 == tiles ? n : (int64_t)c1 * P.tile_nodes;
    const size_t len = (size_t)(n1 - n0);
    if ((rc = nodes.upload_nodes(n0, len, h2d))) return rc;
    UST_CUDA(h, cudaEventRecord(h->seg_up[seg], h2d));
    UST_CUDA(h, cudaStreamWaitEvent(up, h->seg_up[seg], 0));
    if ((rc = nodes.widen_nodes(n0, len, up))) return rc;
    UstParams Ps = P;
    Ps.tile_begin = c0;
    Ps.tile_end = c1;
    Ps.publish = c1 == tiles;
    Ps.seg = seg;
    const int g = pick_grid(h, c1 - c0);
    Ps.static_rounds = pick_static_rounds(h, c1 - c0, g);
    Ps.stamps = 0;
    int e = ust_launch_stream(Ps, g, up, 0);
    if (e) return h->fail(UST_ERR_CUDA, "streaming kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    h->launches += 1;
    UST_CUDA(h, cudaEventRecord(h->seg_done[seg], up));
    UST_CUDA(h, cudaStreamWaitEvent(down, h->seg_done[seg], 0));
    if ((rc = download_outputs(h, n0, len, next_state, actions, outcome, down))) return rc;
  }
  rc = launch_verify(h, P, up, false);
  if (rc) return rc;
  h->ws_dirty = false;
  UST_CUDA(h, cudaMemcpyAsync(h->counters_host, h->counters_dev, sizeof(ust_counters), cudaMemcpyDeviceToHost, up));
  cudaError_t ce = cudaStreamSynchronize(up);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(down);
  if (ce != cudaSuccess) {
    h->ws_dirty = true;
    return h->fail(UST_ERR_CUDA, "kernel execution failed: %s", cudaGetErrorString(ce));
  }
  const bool redone = h->counters_host->reserved[0] != 0;  // the verification redid tiles: fetch the final outputs
  if (redone && (rc = download_outputs(h, 0, (size_t)n, next_state, actions, outcome, up))) return rc;
  return finish_with_counters(h, up, out, !redone);
}

// ust_apply_state and ust_apply_state_packed, once their arguments have been checked: stage the snapshot, evaluate it,
// return the outputs. Without pod lists the staged snapshot stays resident (see keep_resident); with pod lists it does
// not, because the calls on the resident snapshot evaluate no pod lists.
static int apply_host(ust_handle* h, const ust_policy* policy, int64_t n, const HostNodes& nodes, int32_t n_ds,
                      const int32_t* ds_rev, const ust_pods* pods, uint8_t* next_state, uint16_t* actions, uint8_t* outcome,
                      ust_counters* out) {
  UST_CUDA(h, cudaSetDevice(h->device));
  StreamDrain drain(h);
  cudaStream_t st = h->stream;
  const size_t N = (size_t)n;
  UST_CUDA(h, h->s_hot.reserve(N + 16));
  UST_CUDA(h, h->s_flags.reserve(N + 4));
  UST_CUDA(h, h->s_rev.reserve(N + 4));
  UST_CUDA(h, h->s_ds.reserve(N + 4));
  if (nodes.packed) {
    UST_CUDA(h, h->s_rev16.reserve(N + 8));
    UST_CUDA(h, h->s_ds8.reserve(N + 16));
  }
  UST_CUDA(h, h->s_next.reserve(N + 16));
  UST_CUDA(h, h->s_actions.reserve(N + 8));
  UST_CUDA(h, h->s_dsrev.reserve((size_t)n_ds + 1));
  if (outcome) UST_CUDA(h, h->s_outcome.reserve(N + 16));
  if (pods) {
    UST_CUDA(h, h->s_podoff.reserve(N + 1));
    UST_CUDA(h, h->s_podflags.reserve((size_t)pods->n_pods + 8));
  }
  if (n_ds) UST_CUDA(h, cudaMemcpyAsync(h->s_dsrev.p, ds_rev, (size_t)n_ds * 4, cudaMemcpyHostToDevice, st));
  drop_resident(h);
  if (!pods && n >= (1 << 19))
    return keep_resident(h, apply_pipelined(h, nodes, policy, n, n_ds, next_state, actions, outcome, out), n, n_ds);
  int rc = nodes.upload_nodes(0, N, st);
  if (rc) return rc;
  if (pods) {
    UST_CUDA(h, cudaMemcpyAsync(h->s_podoff.p, pods->pod_off, (N + 1) * 4, cudaMemcpyHostToDevice, st));
    if (pods->n_pods) UST_CUDA(h, cudaMemcpyAsync(h->s_podflags.p, pods->pod_flags, (size_t)pods->n_pods * 2, cudaMemcpyHostToDevice, st));
  }
  if ((rc = nodes.widen_nodes(0, N, st))) return rc;
  rc = apply_device(h, false, policy, n, h->s_hot.p, h->s_flags.p, h->s_rev.p, h->s_ds.p, n_ds, h->s_dsrev.p,
                    pods ? h->s_podoff.p : nullptr, pods ? h->s_podflags.p : nullptr, pods ? pods->n_pods : 0, h->s_next.p,
                    h->s_actions.p, outcome ? h->s_outcome.p : nullptr, nullptr, st);
  if (rc) return rc;
  if ((rc = download_outputs(h, 0, N, next_state, actions, outcome, st))) return rc;
  rc = finish_with_counters(h, st, out);
  return pods ? rc : keep_resident(h, rc, n, n_ds);
}

// BuildState staging shared by both forms: pod columns, DaemonSet sizes, per-DaemonSet counters and a clean workspace
static int stage_build_state(ust_handle* h, size_t n_pods, int32_t n_ds, cudaStream_t st) {
  UST_CUDA(h, h->s_hot.reserve(n_pods + 16));
  UST_CUDA(h, h->s_ds.reserve(n_pods + 4));
  UST_CUDA(h, h->s_dsdesired.reserve((size_t)n_ds + 1));
  if ((size_t)n_ds + 1 > h->ds_count.cap) {
    UST_CUDA(h, h->ds_count.resize((size_t)n_ds + 64));
    UST_CUDA(h, cudaMemsetAsync(h->ds_count.p, 0, h->ds_count.cap * sizeof(unsigned long long), st));
  }
  if (h->ws_dirty) { UST_CUDA(h, cudaMemsetAsync(h->ws, 0, sizeof(UstWorkspace), st)); h->ws_dirty = false; }
  return UST_OK;
}
static int build_state_grid(const ust_handle* h, int64_t n_pods) {
  int64_t grid = (n_pods + 1023) / 1024;  // 256 threads x 4 pods per iteration
  if (grid < 1) grid = 1;
  if (grid > 8 * h->num_sms) grid = 8 * h->num_sms;
  return (int)grid;
}

#pragma GCC visibility push(default)

extern "C" {

int ust_abi_version(void) { return UST_ABI_VERSION; }
const char* ust_create_error(void) { return g_create_error.c_str(); }
const char* ust_last_error(const ust_handle* h) { return h ? h->err.c_str() : "null handle"; }
int64_t ust_launch_count(const ust_handle* h) { return h ? h->launches : 0; }

int ust_create(ust_handle** out, int device) {
  if (!out) return UST_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
    return UST_ERR_CUDA;
  }
  if (device < 0 || device >= count) { g_create_error = "device index out of range"; return UST_ERR_INVALID_ARGUMENT; }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return UST_ERR_CUDA; }
  if (prop.major != 10) {
    g_create_error = "libust.so carries sm_100a code only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor);
    return UST_ERR_CUDA;
  }
  ust_handle* h = new ust_handle();
  h->device = device;
  h->no_hint = getenv("UST_NO_HINT") != nullptr;
  if (const char* sg = getenv("UST_SEGMENTS")) { int v = atoi(sg); if (v >= 1 && v <= UST_MAX_SEGMENTS) h->segments = v; }
  auto bail = [&](const char* what, cudaError_t err) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
    ust_destroy(h);
    return UST_ERR_CUDA;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
  if ((e = cudaStreamCreateWithFlags(&h->stream.p, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaStreamCreateWithFlags(&h->stream_d2h.p, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaStreamCreateWithFlags(&h->stream_h2d.p, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  for (auto& ev : h->seg_up)
    if ((e = cudaEventCreateWithFlags(&ev.p, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  for (auto& ev : h->seg_done)
    if ((e = cudaEventCreateWithFlags(&ev.p, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&h->d2h_done.p, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaMalloc(&h->ws.p, sizeof(UstWorkspace))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMemset(h->ws, 0, sizeof(UstWorkspace))) != cudaSuccess) return bail("cudaMemset", e);
  if ((e = cudaMalloc(&h->lut_dev.p, UST_LUT_WORDS * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMalloc(&h->podlut_dev.p, UST_PODLUT_ENTRIES)) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMallocHost(&h->lut_host.p, UST_LUT_WORDS * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMallocHost", e);
  if ((e = cudaMallocHost(&h->podlut_host.p, UST_PODLUT_ENTRIES)) != cudaSuccess) return bail("cudaMallocHost", e);
  if ((e = cudaMalloc(&h->counters_dev.p, sizeof(ust_counters))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMallocHost(&h->counters_host.p, sizeof(ust_counters))) != cudaSuccess) return bail("cudaMallocHost", e);
  if ((e = cudaMalloc(&h->xchg_dev.p, UST_V_LEN * sizeof(long long))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMalloc(&h->sp_count_dev.p, sizeof(long long))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMallocHost(&h->sp_count_host.p, sizeof(long long))) != cudaSuccess) return bail("cudaMallocHost", e);
  if ((e = cudaMemset(h->xchg_dev, 0, UST_V_LEN * sizeof(long long))) != cudaSuccess) return bail("cudaMemset", e);
  if (const char* v = getenv("UST_PDL")) h->pdl = atoi(v) != 0;
  if (const char* v = getenv("UST_STATIC_PCT")) { h->static_pct = atoi(v); if (h->static_pct < 0) h->static_pct = 0; if (h->static_pct > 100) h->static_pct = 100; }
  h->stamps = getenv("UST_STAMPS") != nullptr;
  if (const char* v = getenv("UST_OVERLAP")) h->overlap_calls = atoi(v) != 0;
  size_t stream_smem = 0;  // dynamic shared memory of the streaming kernel (largest variant)
  int rc = ust_stream_config(device, &h->num_sms, &stream_smem);
  if (rc != 0 || h->num_sms < 1) {
    g_create_error = std::string("no sm_100a kernel image usable on this device: ") + cudaGetErrorString((cudaError_t)rc);
    ust_destroy(h);
    return UST_ERR_CUDA;
  }
  *out = h;
  return UST_OK;
}

// What needs an order: nothing in flight, the peers' mailboxes unmapped, the communicator gone. The handle's members
// free its buffers, events and streams.
void ust_destroy(ust_handle* h) {
  if (!h) return;
  if (h->device >= 0) cudaSetDevice(h->device);
  drain_streams(h);
  if (h->last_stream) cudaStreamSynchronize(h->last_stream);
  for (int r = 0; r < UST_MAX_WORLD; r++)
    if (h->mbox[r] && h->mbox[r] != h->mbox_own) cudaIpcCloseMemHandle(h->mbox[r]);
  if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  delete h;
}

void* ust_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
  return p;
}
void ust_host_free(void* p) { if (p) cudaFreeHost(p); }

void* ust_stream(ust_handle* h) { return h ? (void*)h->stream : nullptr; }

int ust_sync(ust_handle* h) {
  UST_ENTER(h);
  UST_CUDA(h, cudaSetDevice(h->device));
  cudaError_t e = cudaStreamSynchronize(h->stream);
  if (e == cudaSuccess && h->last_stream && h->last_stream != h->stream) e = cudaStreamSynchronize(h->last_stream);
  if (e != cudaSuccess) { h->ws_dirty = true; return h->fail(UST_ERR_CUDA, "stream sync failed: %s", cudaGetErrorString(e)); }
  return UST_OK;
}

int ust_apply_state_device(ust_handle* h, const ust_policy* policy, int64_t n_nodes, const uint8_t* state,
                           const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx, int32_t n_ds,
                           const int32_t* ds_rev, const ust_pods* pods, uint8_t* next_state, uint16_t* actions,
                           uint8_t* actuator_outcome, ust_counters* out_device, void* stream) {
  if (!h) return UST_ERR_INVALID_ARGUMENT;
  CallGuard call_guard(h, true);  // the one entry point whose calls may overlap the previous call's tail (apply_device)
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  if (pods && (!pods->pod_off || pods->n_pods < 0 || (pods->n_pods > 0 && !pods->pod_flags)))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "bad pod lists");
  return apply_device(h, true, policy, n_nodes, state, flags, pod_rev, ds_idx, n_ds, ds_rev, pods ? pods->pod_off : nullptr,
                      pods ? pods->pod_flags : nullptr, pods ? pods->n_pods : 0, next_state, actions, actuator_outcome,
                      out_device, st);
}

int ust_apply_state(ust_handle* h, const ust_policy* policy, int64_t n, const uint8_t* state, const uint32_t* flags,
                    const int32_t* pod_rev, const int32_t* ds_idx, int32_t n_ds, const int32_t* ds_rev,
                    const ust_pods* pods, uint8_t* next_state, uint16_t* actions, uint8_t* actuator_outcome,
                    ust_counters* out) {
  UST_ENTER(h);
  if (n < 0 || (n > 0 && (!state || !flags || !pod_rev || !ds_idx || !next_state || !actions)))
    return h->fail(UST_ERR_NIL_STATE, "currentState should not be empty");
  if (n_ds < 0 || (n_ds > 0 && !ds_rev)) return h->fail(UST_ERR_INVALID_ARGUMENT, "bad DaemonSet table");
  if (pods && (!pods->pod_off || pods->n_pods < 0 || (pods->n_pods > 0 && !pods->pod_flags)))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "bad pod lists");
  if (pods) { int prc = check_pod_offsets_host(h, n, pods->pod_off, pods->n_pods); if (prc) return prc; }
  const HostNodes nodes{h, false, state, flags, pod_rev, ds_idx, nullptr, nullptr};
  return apply_host(h, policy, n, nodes, n_ds, ds_rev, pods, next_state, actions, actuator_outcome, out);
}

int ust_apply_state_packed(ust_handle* h, const ust_policy* policy, int64_t n, const uint8_t* state, const uint32_t* flags,
                           const uint16_t* pod_rev16, const int8_t* ds_idx8, int32_t n_ds, const int32_t* ds_rev,
                           uint8_t* next_state, uint16_t* actions, uint8_t* actuator_outcome, ust_counters* out) {
  UST_ENTER(h);
  if (n < 0 || (n > 0 && (!state || !flags || !pod_rev16 || !ds_idx8 || !next_state || !actions)))
    return h->fail(UST_ERR_NIL_STATE, "currentState should not be empty");
  if (n_ds < 0 || n_ds > 127 || (n_ds > 0 && !ds_rev)) return h->fail(UST_ERR_INVALID_ARGUMENT, "bad DaemonSet table (the packed format holds at most 127 DaemonSets)");
  const HostNodes nodes{h, true, state, flags, nullptr, nullptr, pod_rev16, ds_idx8};
  return apply_host(h, policy, n, nodes, n_ds, ds_rev, nullptr, next_state, actions, actuator_outcome, out);
}

// ust_apply_state_delta and ust_apply_state_delta_sparse: scatter the re-encoded nodes into the resident snapshot,
// evaluate everything, return all outputs (dense) or the outputs that differ from the previous call's (sparse).
static int delta_common(ust_handle* h, const ust_policy* policy, int64_t n_changed, const int64_t* idx, const uint8_t* state,
                        const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx, int32_t n_ds, const int32_t* ds_rev,
                        bool sparse, uint8_t* next_state, uint16_t* actions, uint8_t* actuator_outcome, int64_t max_out,
                        int64_t* out_idx, int64_t* n_out, ust_counters* out) {
  const int64_t n = h->resident_n;
  if (n < 0) return h->fail(UST_ERR_INVALID_ARGUMENT, "no resident snapshot: call ust_apply_state (without pod lists) first");
  if (sparse && !h->outputs_resident)
    return h->fail(UST_ERR_INVALID_ARGUMENT, "no resident outputs to compare with: the previous call must be an ApplyState on this snapshot");
  if (n_changed < 0 || (n_changed > 0 && (!idx || !state || !flags || !pod_rev || !ds_idx)))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "bad arguments");
  if (!sparse && n > 0 && (!next_state || !actions)) return h->fail(UST_ERR_INVALID_ARGUMENT, "bad arguments");
  if (sparse && (max_out < 0 || !n_out || (max_out > 0 && (!out_idx || !next_state || !actions))))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "bad arguments");
  if (n_ds < 0 || (n_ds > 0 && !ds_rev)) return h->fail(UST_ERR_INVALID_ARGUMENT, "bad DaemonSet table");
  for (int64_t k = 0; k < n_changed; k++)
    if (idx[k] < 0 || idx[k] >= n) return h->fail(UST_ERR_INVALID_ARGUMENT, "changed node %lld has index %lld outside the snapshot of %lld nodes", (long long)k, (long long)idx[k], (long long)n);
  UST_CUDA(h, cudaSetDevice(h->device));
  StreamDrain drain(h);
  cudaStream_t st = h->stream;
  const size_t N = (size_t)n, M = (size_t)n_changed;
  UST_CUDA(h, h->s_dsrev.reserve((size_t)n_ds + 1));
  if (actuator_outcome) UST_CUDA(h, h->s_outcome.reserve(N + 16));
  UST_CUDA(h, h->d_idx.reserve(M + 1)); UST_CUDA(h, h->d_state.reserve(M + 16)); UST_CUDA(h, h->d_flags.reserve(M + 4));
  UST_CUDA(h, h->d_rev.reserve(M + 4)); UST_CUDA(h, h->d_ds.reserve(M + 4));
  if (sparse) {
    UST_CUDA(h, h->s_next_prev.reserve(h->s_next.cap));
    UST_CUDA(h, h->s_actions_prev.reserve(h->s_actions.cap));
    UST_CUDA(h, h->sp_blocks.reserve((size_t)ust_diff_blocks(n) + 1));
    UST_CUDA(h, h->sp_idx.reserve((size_t)max_out + 1));
    UST_CUDA(h, h->sp_next.reserve((size_t)max_out + 16));
    UST_CUDA(h, h->sp_actions.reserve((size_t)max_out + 8));
  }
  drop_resident(h);  // until the patched snapshot has been evaluated
  if (n_ds) UST_CUDA(h, cudaMemcpyAsync(h->s_dsrev.p, ds_rev, (size_t)n_ds * 4, cudaMemcpyHostToDevice, st));
  if (M) {
    static_assert(sizeof(long long) == sizeof(int64_t), "index width");
    UST_CUDA(h, cudaMemcpyAsync(h->d_idx.p, idx, M * 8, cudaMemcpyHostToDevice, st));
    UST_CUDA(h, cudaMemcpyAsync(h->d_state.p, state, M, cudaMemcpyHostToDevice, st));
    UST_CUDA(h, cudaMemcpyAsync(h->d_flags.p, flags, M * 4, cudaMemcpyHostToDevice, st));
    UST_CUDA(h, cudaMemcpyAsync(h->d_rev.p, pod_rev, M * 4, cudaMemcpyHostToDevice, st));
    UST_CUDA(h, cudaMemcpyAsync(h->d_ds.p, ds_idx, M * 4, cudaMemcpyHostToDevice, st));
    int e = ust_launch_patch((long long)n_changed, h->d_idx.p, h->d_state.p, h->d_flags.p, h->d_rev.p, h->d_ds.p, h->s_hot.p,
                             h->s_flags.p, h->s_rev.p, h->s_ds.p, st);
    if (e) return h->fail(UST_ERR_CUDA, "patch kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    h->launches += 1;
  }
  if (sparse) {  // the previous call's outputs step aside; this call writes the other pair of arrays
    std::swap(h->s_next, h->s_next_prev);
    std::swap(h->s_actions, h->s_actions_prev);
  }
  int rc = apply_device(h, false, policy, n, h->s_hot.p, h->s_flags.p, h->s_rev.p, h->s_ds.p, n_ds, h->s_dsrev.p, nullptr, nullptr,
                        0, h->s_next.p, h->s_actions.p, actuator_outcome ? h->s_outcome.p : nullptr, nullptr, st);
  if (rc) return rc;
  if (!sparse) {
    if ((rc = download_outputs(h, 0, N, next_state, actions, actuator_outcome, st))) return rc;
  } else {
    int e = ust_launch_diff((long long)n, h->s_next.p, h->s_actions.p, h->s_next_prev.p, h->s_actions_prev.p, h->sp_blocks.p,
                            h->sp_count_dev, (long long)max_out, h->sp_idx.p, h->sp_next.p, h->sp_actions.p, st);
    if (e) return h->fail(UST_ERR_CUDA, "diff kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    h->launches += 3;
    UST_CUDA(h, cudaMemcpyAsync(h->sp_count_host, h->sp_count_dev, sizeof(long long), cudaMemcpyDeviceToHost, st));
    UST_CUDA(h, cudaStreamSynchronize(st));
    const int64_t cnt = *h->sp_count_host;
    *n_out = cnt;
    if (cnt <= max_out && cnt > 0) {
      UST_CUDA(h, cudaMemcpyAsync(out_idx, h->sp_idx.p, (size_t)cnt * 8, cudaMemcpyDeviceToHost, st));
      UST_CUDA(h, cudaMemcpyAsync(next_state, h->sp_next.p, (size_t)cnt, cudaMemcpyDeviceToHost, st));
      UST_CUDA(h, cudaMemcpyAsync(actions, h->sp_actions.p, (size_t)cnt * 2, cudaMemcpyDeviceToHost, st));
    }
  }
  rc = keep_resident(h, finish_with_counters(h, st, out), n, n_ds);
  if (sparse && (rc == UST_OK) && *n_out > max_out)
    return h->fail(UST_ERR_TRUNCATED, "%lld outputs changed, the caller's arrays hold %lld: fetch them with ust_fetch_outputs", (long long)*n_out, (long long)max_out);
  return rc;
}

int ust_apply_state_delta(ust_handle* h, const ust_policy* policy, int64_t n_changed, const int64_t* idx, const uint8_t* state,
                          const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx, int32_t n_ds,
                          const int32_t* ds_rev, uint8_t* next_state, uint16_t* actions, uint8_t* actuator_outcome,
                          ust_counters* out) {
  UST_ENTER(h);
  return delta_common(h, policy, n_changed, idx, state, flags, pod_rev, ds_idx, n_ds, ds_rev, false, next_state, actions,
                      actuator_outcome, 0, nullptr, nullptr, out);
}

int ust_apply_state_delta_sparse(ust_handle* h, const ust_policy* policy, int64_t n_changed, const int64_t* idx,
                                 const uint8_t* state, const uint32_t* flags, const int32_t* pod_rev, const int32_t* ds_idx,
                                 int32_t n_ds, const int32_t* ds_rev, int64_t max_out, int64_t* out_idx,
                                 uint8_t* out_next_state, uint16_t* out_actions, int64_t* n_out, ust_counters* out) {
  UST_ENTER(h);
  return delta_common(h, policy, n_changed, idx, state, flags, pod_rev, ds_idx, n_ds, ds_rev, true, out_next_state, out_actions,
                      nullptr, max_out, out_idx, n_out, out);
}

int ust_fetch_outputs(ust_handle* h, uint8_t* next_state, uint16_t* actions) {
  UST_ENTER(h);
  if (h->resident_n < 0 || !h->outputs_resident) return h->fail(UST_ERR_INVALID_ARGUMENT, "no resident outputs");
  if (h->resident_n > 0 && (!next_state || !actions)) return h->fail(UST_ERR_INVALID_ARGUMENT, "bad arguments");
  UST_CUDA(h, cudaSetDevice(h->device));
  int rc = download_outputs(h, 0, (size_t)h->resident_n, next_state, actions, nullptr, h->stream);
  if (rc) return rc;
  UST_CUDA(h, cudaStreamSynchronize(h->stream));
  return UST_OK;
}

static int simulate_common(ust_handle* h, const ust_policy* policy, const ust_sim_options* opt, int32_t steps, ust_counters* history,
                           uint8_t* final_state, uint32_t* final_flags, int32_t* final_pod_rev, int32_t* steps_done) {
  const int64_t n = h->resident_n;
  if (n < 0) return h->fail(UST_ERR_INVALID_ARGUMENT, "no resident snapshot: call ust_apply_state (without pod lists) first");
  if (steps < 0 || steps > (1 << 20)) return h->fail(UST_ERR_INVALID_ARGUMENT, "bad step count");
  if (h->world > 1) return h->fail(UST_ERR_INVALID_ARGUMENT, "rollout simulation runs on one GPU");
  if (opt && (opt->seconds_per_reconcile < 0 || opt->wait_timeout_seconds < 0 || opt->job_seconds < 0 || opt->validation_timeout_seconds < 0 ||
              opt->maintenance_seconds < 0 || (int64_t)steps * opt->seconds_per_reconcile >= (1LL << 29)))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "bad simulation options (times are non-negative; the horizon stays below 2^29 seconds)");
  if (opt && policy && (policy->wait_timeout_nonzero != 0) != (opt->wait_timeout_seconds != 0))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "policy.wait_timeout_nonzero must say whether wait_timeout_seconds != 0");
  ust_policy pol;
  if (policy) { pol = *policy; pol.evaluate_actuators = 1; }  // the asynchronous actuators' results are what is fed back
  UST_CUDA(h, cudaSetDevice(h->device));
  StreamDrain drain(h);
  cudaStream_t st = h->stream;
  const size_t N = (size_t)n;
  UST_CUDA(h, h->s_outcome.reserve(N + 16));
  if ((size_t)steps + 1 > h->hist.cap) UST_CUDA(h, h->hist.resize((size_t)steps + 64));
  drop_resident(h);
  int grid = 8 * h->num_sms;
  UstSimParams sp;
  memset(&sp, 0, sizeof(sp));
  if (opt) {
    sp.timed = 1;
    sp.dt = opt->seconds_per_reconcile;
    sp.wait_timeout = opt->wait_timeout_seconds; sp.job_seconds = opt->job_seconds; sp.validation_seconds = opt->validation_seconds;
    sp.validation_timeout = opt->validation_timeout_seconds; sp.maintenance_seconds = opt->maintenance_seconds;
    UST_CUDA(h, h->sim_entered.reserve(N + 1)); UST_CUDA(h, h->sim_wait.reserve(N + 1)); UST_CUDA(h, h->sim_valid.reserve(N + 1));
    int e = ust_launch_sim_init(n, h->s_flags.p, h->sim_entered.p, h->sim_wait.p, h->sim_valid.p, grid, st);
    if (e) return h->fail(UST_ERR_CUDA, "simulation init kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    h->launches += 1;
  }
  for (int32_t k = 0; k < steps; k++) {
    int rc = apply_device(h, false, policy ? &pol : nullptr, n, h->s_hot.p, h->s_flags.p, h->s_rev.p, h->s_ds.p, h->resident_n_ds,
                          h->s_dsrev.p, nullptr, nullptr, 0, h->s_next.p, h->s_actions.p, h->s_outcome.p, h->hist.p + k, st);
    if (rc) return rc;
    sp.now = (long long)k * sp.dt;
    int e = ust_launch_feedback(n, h->s_hot.p, h->s_flags.p, h->s_rev.p, h->s_ds.p, h->resident_n_ds, h->s_dsrev.p, h->s_next.p,
                                h->s_actions.p, h->s_outcome.p, h->hist.p + k, sp, h->sim_entered.p, h->sim_wait.p, h->sim_valid.p,
                                grid, st);
    if (e) return h->fail(UST_ERR_CUDA, "feedback kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    h->launches += 1;
  }
  std::vector<ust_counters> hist((size_t)steps);
  if (steps) UST_CUDA(h, cudaMemcpyAsync(hist.data(), h->hist.p, (size_t)steps * sizeof(ust_counters), cudaMemcpyDeviceToHost, st));
  if (N && final_state) UST_CUDA(h, cudaMemcpyAsync(final_state, h->s_hot.p, N, cudaMemcpyDeviceToHost, st));
  if (N && final_flags) UST_CUDA(h, cudaMemcpyAsync(final_flags, h->s_flags.p, N * 4, cudaMemcpyDeviceToHost, st));
  if (N && final_pod_rev) UST_CUDA(h, cudaMemcpyAsync(final_pod_rev, h->s_rev.p, N * 4, cudaMemcpyDeviceToHost, st));
  cudaError_t ce = cudaStreamSynchronize(st);
  if (ce != cudaSuccess) { h->ws_dirty = true; return h->fail(UST_ERR_CUDA, "kernel execution failed: %s", cudaGetErrorString(ce)); }
  h->resident_n = n;  // the snapshot now holds the simulated state
  h->outputs_resident = false;
  int32_t done = steps;
  int rc = UST_OK;
  for (int32_t k = 0; k < steps; k++)
    if (hist[(size_t)k].error_code != UST_OK) { done = k; rc = (int)hist[(size_t)k].error_code; break; }
  if (history) memcpy(history, hist.data(), (size_t)steps * sizeof(ust_counters));
  if (steps_done) *steps_done = done;
  if (rc) return h->fail(rc, "the simulated reconcile %d returned an error (code %d); the state before it is kept", (int)done, rc);
  return UST_OK;
}

int ust_simulate_rollout(ust_handle* h, const ust_policy* policy, int32_t steps, ust_counters* history, uint8_t* final_state,
                         uint32_t* final_flags, int32_t* final_pod_rev, int32_t* steps_done) {
  UST_ENTER(h);
  return simulate_common(h, policy, nullptr, steps, history, final_state, final_flags, final_pod_rev, steps_done);
}

int ust_simulate_rollout_timed(ust_handle* h, const ust_policy* policy, const ust_sim_options* options, int32_t steps,
                               ust_counters* history, uint8_t* final_state, uint32_t* final_flags, int32_t* final_pod_rev,
                               int32_t* steps_done) {
  if (!options) return UST_ERR_INVALID_ARGUMENT;
  UST_ENTER(h);
  return simulate_common(h, policy, options, steps, history, final_state, final_flags, final_pod_rev, steps_done);
}

int ust_build_state(ust_handle* h, int64_t n_pods, const uint8_t* state, const int32_t* ds_idx, int32_t n_ds,
                    const int32_t* ds_desired, ust_counters* out) {
  UST_ENTER(h);
  if (n_pods < 0 || (n_pods > 0 && (!state || !ds_idx)) || n_ds < 0 || (n_ds > 0 && !ds_desired))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "bad arguments");
  drop_resident(h);  // shares the staging arrays
  UST_CUDA(h, cudaSetDevice(h->device));
  StreamDrain drain(h);
  cudaStream_t st = h->stream;
  const size_t N = (size_t)n_pods;
  int rc = stage_build_state(h, N, n_ds, st);
  if (rc) return rc;
  if (N) {
    UST_CUDA(h, cudaMemcpyAsync(h->s_hot.p, state, N, cudaMemcpyHostToDevice, st));
    UST_CUDA(h, cudaMemcpyAsync(h->s_ds.p, ds_idx, N * 4, cudaMemcpyHostToDevice, st));
  }
  if (n_ds) UST_CUDA(h, cudaMemcpyAsync(h->s_dsdesired.p, ds_desired, (size_t)n_ds * 4, cudaMemcpyHostToDevice, st));
  h->ws_dirty = true;
  int e = ust_launch_build_state(n_pods, h->s_hot.p, h->s_ds.p, n_ds, h->s_dsdesired.p, h->ds_count.p, h->ws, h->counters_dev,
                                 build_state_grid(h, n_pods), st);
  if (e) return h->fail(UST_ERR_CUDA, "build-state kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
  h->ws_dirty = false;
  h->launches += 2;
  return finish_with_counters(h, st, out);
}

int ust_build_state_uids(ust_handle* h, int64_t n_pods, const uint8_t* state, const uint64_t* owner_uid, int32_t n_ds,
                         const uint64_t* ds_uid, const int32_t* ds_desired, int32_t* ds_idx_out, ust_counters* out) {
  UST_ENTER(h);
  if (n_pods < 0 || (n_pods > 0 && (!state || !owner_uid || !ds_idx_out)) || n_ds < 0 || (n_ds > 0 && (!ds_uid || !ds_desired)))
    return h->fail(UST_ERR_INVALID_ARGUMENT, "bad arguments");
  // the DaemonSet map is keyed by UID (common_manager.go:181-185): an open-addressing table at load factor <= 1/4
  size_t slots = 8;
  while (slots < 4 * (size_t)n_ds) slots <<= 1;
  std::vector<uint64_t> tab(2 * slots, 0);
  std::vector<int32_t> tab_idx(slots, -2);
  for (int32_t d = 0; d < n_ds; d++) {
    const uint64_t x = ds_uid[2 * (size_t)d], y = ds_uid[2 * (size_t)d + 1];
    if ((x | y) == 0) return h->fail(UST_ERR_INVALID_ARGUMENT, "DaemonSet %d has an empty UID", (int)d);
    size_t s = ust_uid_hash(x, y) & (slots - 1);
    while ((tab[2 * s] | tab[2 * s + 1]) != 0) {
      if (tab[2 * s] == x && tab[2 * s + 1] == y)
        return h->fail(UST_ERR_INVALID_ARGUMENT, "DaemonSets %d and %d share a UID", (int)tab_idx[s], (int)d);
      s = (s + 1) & (slots - 1);
    }
    tab[2 * s] = x; tab[2 * s + 1] = y; tab_idx[s] = d;
  }
  drop_resident(h);  // shares the staging arrays
  UST_CUDA(h, cudaSetDevice(h->device));
  StreamDrain drain(h);
  cudaStream_t st = h->stream;
  const size_t N = (size_t)n_pods;
  UST_CUDA(h, h->s_uid.reserve(2 * N + 2));
  UST_CUDA(h, h->s_dsuid.reserve(2 * slots));
  UST_CUDA(h, h->s_dsorder.reserve(slots));
  int rc = stage_build_state(h, N, n_ds, st);
  if (rc) return rc;
  if (N) {
    UST_CUDA(h, cudaMemcpyAsync(h->s_hot.p, state, N, cudaMemcpyHostToDevice, st));
    UST_CUDA(h, cudaMemcpyAsync(h->s_uid.p, owner_uid, N * 16, cudaMemcpyHostToDevice, st));
  }
  UST_CUDA(h, cudaMemcpyAsync(h->s_dsuid.p, tab.data(), slots * 16, cudaMemcpyHostToDevice, st));
  UST_CUDA(h, cudaMemcpyAsync(h->s_dsorder.p, tab_idx.data(), slots * 4, cudaMemcpyHostToDevice, st));
  if (n_ds) UST_CUDA(h, cudaMemcpyAsync(h->s_dsdesired.p, ds_desired, (size_t)n_ds * 4, cudaMemcpyHostToDevice, st));
  h->ws_dirty = true;
  int e = ust_launch_build_state_uids(n_pods, h->s_hot.p, h->s_uid.p, n_ds, h->s_dsuid.p, h->s_dsorder.p, (int)slots,
                                      h->s_dsdesired.p, h->s_ds.p, h->ds_count.p, h->ws, h->counters_dev,
                                      build_state_grid(h, n_pods), st);
  if (e) return h->fail(UST_ERR_CUDA, "build-state kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
  h->ws_dirty = false;
  h->launches += 2;
  if (N) UST_CUDA(h, cudaMemcpyAsync(ds_idx_out, h->s_ds.p, N * 4, cudaMemcpyDeviceToHost, st));
  return finish_with_counters(h, st, out);  // synchronises the stream: `tab` / `tab_idx` outlive their copies
}

uint32_t ust_table_entry(const ust_policy* policy, unsigned state_code, uint32_t w) {
  // the very table the kernels stage and the very lookup they make (ust_lut.h), built for `policy` (cached per thread)
  static thread_local std::vector<uint32_t> lut;
  static thread_local ust_policy cached;
  static thread_local bool have = false;
  state_code &= 15u;
  const ust_policy key = table_key(policy);
  if (!have || memcmp(&key, &cached, sizeof(key)) != 0) {
    lut.assign(UST_LUT_WORDS, 0u);
    ust_build_lut(policy_active(policy) ? &key : nullptr, lut.data());
    cached = key;
    have = true;
  }
  return ust_lut_lookup(lut.data(), state_code, w);
}
int ust_table_window_shift(unsigned state_code) { return ust_window_shift[state_code & 15u]; }

// audit: entries of the 2048-entry pod table (ust_build_pod_lut) that T[pf & 255] & gate(pf) disagrees with
int ust_debug_podlut_mismatches(const ust_policy* p) {
  if (!p) return -1;
  uint8_t full[UST_PODLUT_ENTRIES], T[256];
  ust_build_pod_lut(p, full);
  ust_build_pod_lut256(p, T);
  int bad = 0;
  for (unsigned pf = 0; pf < UST_PODLUT_ENTRIES; pf++) bad += (T[pf & 255u] & ust_pod_gate(pf)) != full[pf];
  return bad;
}

long long ust_debug_relaxed_calls(ust_handle* h) { return h ? (long long)h->relaxed_calls : -1; }

// diagnostics (not in include/ust.h): %globaltimer stamps taken by CTA 0 of the last fused launch
int ust_debug_stamps(ust_handle* h, unsigned long long* out, int n_ctas) {
  if (!out || n_ctas < 1 || n_ctas > UST_MAX_CTAS) return UST_ERR_INVALID_ARGUMENT;
  UST_ENTER(h);
  UST_CUDA(h, cudaSetDevice(h->device));
  UST_CUDA(h, cudaDeviceSynchronize());
  UST_CUDA(h, cudaMemcpy(out, h->ws->dbg, (size_t)n_ctas * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  UST_CUDA(h, cudaMemcpy(out + (size_t)n_ctas * 4, h->ws->dbg2, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));  // verification kernel
  return UST_OK;
}

int ust_get_unique_id(void* out_bytes) {
  if (!out_bytes) return UST_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(g_nccl_mu);
  std::string err;
  if (!g_nccl.load(&err)) { g_create_error = err; return UST_ERR_COMM; }
  ncclUniqueId id;
  static_assert(sizeof(ncclUniqueId) == UST_UNIQUE_ID_BYTES, "ncclUniqueId size");
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return UST_ERR_COMM; }
  memcpy(out_bytes, &id, sizeof(id));
  return UST_OK;
}

int ust_comm_init(ust_handle* h, int rank, int world_size, const void* unique_id_bytes) {
  UST_ENTER(h);
  if (world_size < 1 || world_size > UST_MAX_WORLD || rank < 0 || rank >= world_size)
    return h->fail(UST_ERR_INVALID_ARGUMENT, "world size must be 1..%d", UST_MAX_WORLD);
  if (world_size == 1) { h->rank = 0; h->world = 1; return UST_OK; }
  if (!unique_id_bytes) return h->fail(UST_ERR_INVALID_ARGUMENT, "unique id required");
  {
    std::lock_guard<std::mutex> g2(g_nccl_mu);
    std::string err;
    if (!g_nccl.load(&err)) return h->fail(UST_ERR_COMM, "%s", err.c_str());
  }
  UST_CUDA(h, cudaSetDevice(h->device));
  ncclUniqueId id;
  memcpy(&id, unique_id_bytes, sizeof(id));
  ncclResult_t r = g_nccl.CommInitRank(&h->comm, world_size, id, rank);
  if (r != ncclSuccess) return h->fail(UST_ERR_COMM, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  h->rank = rank;
  h->world = world_size;
  // Mailboxes for the fused exchange: allocate, all-gather the CUDA IPC handles over the new communicator, map the
  // peers' buffers. Any failure leaves the NCCL exchange (mode 0) as the only mode.
  h->mbox_ready = false;
  do {
    if (!g_nccl.AllGather) break;
    if (cudaMalloc(&h->mbox_own.p, sizeof(UstMailbox)) != cudaSuccess) break;
    if (cudaMemset(h->mbox_own, 0, sizeof(UstMailbox)) != cudaSuccess) break;
    cudaIpcMemHandle_t mine;
    if (cudaIpcGetMemHandle(&mine, h->mbox_own) != cudaSuccess) { cudaGetLastError(); break; }
    cudaIpcMemHandle_t* dev = nullptr;
    if (cudaMalloc(&dev, sizeof(cudaIpcMemHandle_t) * (size_t)(world_size + 1)) != cudaSuccess) break;
    cudaMemcpy(dev + world_size, &mine, sizeof(mine), cudaMemcpyHostToDevice);
    ncclResult_t g = g_nccl.AllGather(dev + world_size, dev, sizeof(mine), ncclChar, h->comm, h->stream);
    cudaError_t ce = cudaStreamSynchronize(h->stream);
    std::vector<cudaIpcMemHandle_t> all((size_t)world_size);
    if (g == ncclSuccess && ce == cudaSuccess) cudaMemcpy(all.data(), dev, sizeof(mine) * (size_t)world_size, cudaMemcpyDeviceToHost);
    cudaFree(dev);
    if (g != ncclSuccess || ce != cudaSuccess) break;
    bool ok = true;
    for (int r = 0; r < world_size && ok; r++) {
      if (r == rank) { h->mbox[r] = h->mbox_own; continue; }
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, all[(size_t)r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
      h->mbox[r] = (UstMailbox*)p;
    }
    h->mbox_ready = ok;
  } while (0);
  h->epoch = 0;
  return UST_OK;
}

int ust_comm_set_mode(ust_handle* h, int mode) {
  UST_ENTER(h);
  if (mode != 0 && mode != 1) return h->fail(UST_ERR_INVALID_ARGUMENT, "unknown exchange mode %d", mode);
  if (mode == 1 && !(h->world > 1 && h->mbox_ready))
    return h->fail(UST_ERR_COMM, "fused exchange unavailable: peer mailboxes could not be mapped (CUDA IPC)");
  h->comm_mode = mode;
  return UST_OK;
}

}  // extern "C"
#pragma GCC visibility pop
