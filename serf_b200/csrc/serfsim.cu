// serfsim.cu — host side of the simulator and its C ABI (include/serfsim.h).
//
// The reference's host code is Rust; Rust is not available in this build environment, so the
// host layer above the C ABI is C++ and mirrors the reference's names: Options/MemberlistOptions
// fields (serf-core/src/options.rs:495-530), Serf::{join,leave,remove_failed_node,members,stats}
// (serf/api.rs), MemberStatus (types/member.rs:54-58), MemberEventType (event.rs:325-328).
// Device memory, streams and the per-tick launch sequence live here; the kernels are in
// tick_kernel.cu.  There is no CPU execution path: without a CUDA device every entry point fails.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_set>
#include <vector>

#include "../../include/serfsim.h"
#include "tick_kernel.cuh"

using namespace sfs;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(SERFSIM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));        \
  } while (0)

struct HostOp { u32 tick, op, node, slot; u64 seq; };

// memberlist retransmit limit: retransmit_mult * ceil(log10(n + 1))  [external crate, restated]
u32 retransmit_limit(u32 mult, u64 n) {
  u32 digits = 0;
  u64 p = 1;
  while (p < n + 1) { p *= 10; ++digits; }
  return mult * digits;
}

// memberlist suspicion timeouts (Lifeguard), in ticks  [external crate, restated]:
//   min = suspicion_mult · max(1, log10 n) · probe_interval, max = suspicion_max_timeout_mult · min,
//   k = suspicion_mult − 2 (0 if n − 2 < k), timeout(c) = max − log(c+1)/log(k+1)·(max − min) ≥ min.
// The only floating point on the whole path; it runs once on the host and yields integers.
std::vector<u32> suspicion_table(u32 susp_mult, u32 max_mult, u32 probe_ticks, u32 tick_ms, u64 n) {
  const double node_scale = std::max(1.0, std::log10(std::max(1.0, (double)n)));
  const int64_t interval_ms = (int64_t)probe_ticks * tick_ms;
  const int64_t min_ms = (int64_t)susp_mult * (int64_t)(node_scale * 1000.0) * interval_ms / 1000;
  const int64_t max_ms = (int64_t)max_mult * min_ms;
  int64_t k = (int64_t)susp_mult - 2;
  if ((int64_t)n - 2 < k) k = 0;
  if (k < 0) k = 0;
  std::vector<u32> tab;
  for (int64_t c = 0; c <= k; ++c) {
    int64_t ms = min_ms;
    if (k >= 1) {
      const double frac = std::log((double)c + 1.0) / std::log((double)k + 1.0);
      ms = (int64_t)std::floor((double)max_ms - frac * (double)(max_ms - min_ms));
      if (ms < min_ms) ms = min_ms;
    }
    int64_t ticks = (ms + tick_ms - 1) / tick_ms;
    if (ticks < 1) ticks = 1;
    tab.push_back((u32)ticks);
  }
  return tab;
}

}  // namespace

struct serfsim {
  serfsim_config_t cfg{};
  u32 N = 0, R = 0, first = 0, count = 0, shard_size = 0;
  u32 stride = 0;                  // count rounded up to a whole 256-node tile: stride of every per-slot plane
  Rules rules{};
  // device state
  uint4* d_rec = nullptr;          // [R][stride] × 32 B (transmit-budget bytes zero)
  u32* d_qword = nullptr;          // [R][stride] queue words (transmit budgets)
  u32* d_inbox[2] = {nullptr, nullptr};   // [3][R][count]
  u64* d_node = nullptr;           // [count]
  u8* d_busy = nullptr;            // [stride] per-node busy byte
  u16* d_watch = nullptr;          // [stride] per-node watcher mask (subjects among the node's neighbours)
  bool watch_dirty = true;
  uint4* d_snap_rec = nullptr;     // push-pull rounds: end-of-tick snapshot of the records …
  u64* d_snap_node = nullptr;      // … and of the node words
  const uint4** d_peer_snap_rec = nullptr;   // sharded push-pull: device arrays of every rank's snapshot pointers
  const u64** d_peer_snap_node = nullptr;
  u8* d_hot[2] = {nullptr, nullptr};      // [n_tiles] per tick parity
  u8* d_hot_static = nullptr;             // [n_tiles] tiles that hold a watcher (never consumed)
  u32* d_node_due = nullptr;              // [stride] per-node earliest suspicion deadline (tick_kernel.cuh)
  u32* d_tile_due = nullptr;              // [n_tiles] earliest suspicion deadline of a tile's nodes (the timer wheel)
  u32* d_sched = nullptr;                 // scheduler words (tick_kernel.cuh: SCHED_*)
  u32 n_tiles = 0;
  u32* d_rowptr = nullptr;         // [count+1]
  u32* d_col = nullptr;
  u32 *d_ev_node = nullptr, *d_ev_op = nullptr, *d_ev_slot = nullptr;
  size_t ev_cap = 0;
  u64* d_trace = nullptr;          // [trace_cap][8]
  u32* d_kinds = nullptr;          // [trace_cap+1][4]; row t+1 = messages by kind sent in tick t
  u32* d_ones = nullptr;           // [4] non-zero (multi-GPU: never skip an inbox plane)
  u32 trace_cap = 0;
  u32* d_overflow = nullptr;       // device address of pin_overflow (mapped pinned host memory: written by kernels on the rare error paths, read by the host without a copy)
  u32* pin_overflow = nullptr;
  u32* d_subj = nullptr;
  u64* d_scratch = nullptr;        // summary / hash output
  void* d_stage = nullptr;         // getter staging, count × 8 B
  // user events (SURVEY §8f row 3): allocated by serfsim_set_user_events
  UeTable ue_table{};              // n = 0: user events off
  uint4* d_ue_state = nullptr;     // [stride] 16-byte event records
  u32* d_ue_inbox[2] = {nullptr, nullptr};   // [stride] arrived-event masks per tick parity
  u32* d_ue_ltime = nullptr;       // [MAX_UEVENTS]
  u64* d_ue_totals = nullptr;      // [8]
  u32 ue_injected = 0;             // tracked events already scheduled (each may be injected once)
  uint4* d_ue_snap = nullptr;      // push-pull rounds: snapshot of the event records (partners read it)
  const uint4** d_peer_ue_snap = nullptr;
  u32 ue_origin[MAX_UEVENTS] = {0};
  u32 ue_fire_tick[MAX_UEVENTS] = {0};  // origin node of each scheduled event (its shard is the one that stamps the Lamport time)
  // byzantine injectors (BASELINE configs[4]): allocated by serfsim_set_byzantine
  u32 byz_n = 0, byz_delta = 2;    // byz_n: injectors of THIS shard
  bool byz_on = false;             // any injector anywhere (all ranks agree): changes the convergence rule and the drain kernel
  u8** d_peer_anomaly = nullptr;   // sharded runs: device array of every rank's flag array
  u32* d_byz_ids = nullptr;        // [byz_n] ascending
  u8* d_anomaly = nullptr;         // [stride] sender flags
  u64* d_byz_totals = nullptr;     // [4]
  // host state
  std::vector<HostOp> ops;         // sorted by (tick, seq)
  std::unordered_set<u64> op_keys; // (tick << 32 | node): at most one operation per node per tick
  bool ops_dirty = false;
  u64 op_seq = 0;
  std::vector<u32> subj;
  u32 up_mask = 0;
  u32 ever_down = 0;               // subjects that have been down at some tick since the reset (only those are probed, suspected, run timers)
  u32 sv = 1;                      // single-view ticks of multi-slot runs: 1 = dual launch, 2 = check mode, 0 = off (SERFSIM_SV, tick_kernel.cuh)
  int grid_sv = 0;                 // grid of the single-view kernel
  u32 tick = 0;
  bool has_topo = false;
  u32 ahead = 1;                   // multi-slot tick kernel: software pipelining of saturated ticks (SERFSIM_AHEAD=0 / 1 / 2, tick_kernel.cuh)
  u32 udeg = 0;                    // uniform out-degree of the shard's rows (0: degrees differ)
  std::vector<serfsim_tick_row_t> rows;   // rows pulled from the device so far (global sums when sharded)
  // device-side convergence gate (tick_kernel.cuh: Gate)
  u32* d_runctl = nullptr;         // [0] done flag, [1] first quiescent tick
  u32* pin_ctl = nullptr;          // the verdict in mapped pinned host memory (written by the gate's leader thread), read once per chunk
  u32* d_pin_ctl = nullptr;        // its device address
  u64* d_grow = nullptr;           // sharded runs: [trace_cap][8] global trace rows, summed on the device by the drain kernel
  bool gate_on = false;
  u32 gate_first = 0;              // first tick of the current run_until_converged call (it always runs)
  std::vector<u32> launch_log;     // kernels launched per tick since the timing window opened (ticks past the quiescent one do not count)
  u32 launch_log_first = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timing_open = false;
  double last_ms = 0.0;
  u64 last_launches = 0, launches = 0;
  serfsim_event_cb cb = nullptr;
  void* cb_user = nullptr;
  std::vector<u8> reported;        // last status reported per slot
  int grid = 1;
  int ctas_per_sm = 4;
  // multi-GPU
  u64* d_win_data[2] = {nullptr, nullptr};     // my receive windows [parity][world][win_cap]  (IPC-exported)
  u32* d_ctrl = nullptr;                       // my control block [parity][counts[8] | flags[8]] (IPC-exported)
  u32* d_send_count = nullptr;                 // [world] entries written into each peer's window this tick
  u64** d_peer_data[2] = {nullptr, nullptr};   // device arrays of peer window pointers, per parity
  u32** d_peer_ctrl = nullptr;                 // device array of peer control-block pointers
  u32 xepoch = 0;                              // executed-tick counter of the exchange (never rewinds): stamps and parity
  u32 win_cap = 0;
  u32 win_cap_base = 0;                        // capacity sized for the membership entries alone (serfsim_create)
  bool connected = false;
  bool loopback = false;                       // serfsim_comm_loopback: profiling aid, the handle exchanges with itself
  serfsim_barrier_fn barrier = nullptr; serfsim_allreduce_u64_fn allreduce = nullptr; void* comm_user = nullptr;
  std::vector<void*> ipc_opened;
  bool tick_timing = false;
  bool no_skip = false;             // SERFSIM_NO_SKIP=1: process every tile every tick (A/B measurements)
  bool compact = true;              // SERFSIM_COMPACT=0: tile-by-tile walk in unsaturated ticks too (A/B measurements)
  // asynchronous result read-back (serfsim_results_async): extraction into a ring of staging buffers on the launch stream,
  // device→host copies on a second stream so that they overlap the ticks of the caller's next step
  struct ResBuf { unsigned char* d = nullptr; cudaEvent_t copied = nullptr; bool used = false; };
  ResBuf res[4];
  u32 res_next = 0;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_extracted = nullptr;
  std::vector<cudaEvent_t> tick_ev;      // 2 per tick when tick_timing
  std::vector<cudaEvent_t> mid_ev;       // after the tick kernel (multi-GPU breakdown, SERFSIM_XTIMING=1)
};

namespace {

int slot_of(const serfsim* h, u32 node) {
  for (u32 s = 0; s < h->R; ++s) if (h->subj[s] == node) return (int)s;
  return -1;
}

int ensure_trace(serfsim* h, u32 need) {
  if (need <= h->trace_cap) return 0;
  u32 cap = std::max<u32>(1024, h->trace_cap);
  while (cap < need) cap *= 2;
  u64* nt = nullptr; u32* nk = nullptr; u64* ng = nullptr;
  const bool sharded = h->cfg.world_size > 1;
  CU(cudaMalloc(&nt, (size_t)cap * 8 * sizeof(u64)));
  CU(cudaMalloc(&nk, ((size_t)cap + 1) * 4 * sizeof(u32)));
  CU(cudaMemsetAsync(nt, 0, (size_t)cap * 8 * sizeof(u64), h->stream));
  CU(cudaMemsetAsync(nk, 0, ((size_t)cap + 1) * 4 * sizeof(u32), h->stream));
  if (sharded) { CU(cudaMalloc(&ng, (size_t)cap * 8 * sizeof(u64))); CU(cudaMemsetAsync(ng, 0, (size_t)cap * 8 * sizeof(u64), h->stream)); }
  if (h->d_trace) {
    CU(cudaMemcpyAsync(nt, h->d_trace, (size_t)h->trace_cap * 8 * sizeof(u64), cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(nk, h->d_kinds, ((size_t)h->trace_cap + 1) * 4 * sizeof(u32), cudaMemcpyDeviceToDevice, h->stream));
    if (sharded) CU(cudaMemcpyAsync(ng, h->d_grow, (size_t)h->trace_cap * 8 * sizeof(u64), cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(h->d_trace); cudaFree(h->d_kinds); cudaFree(h->d_grow);
  }
  h->d_trace = nt; h->d_kinds = nk; h->d_grow = ng; h->trace_cap = cap;
  return 0;
}

int upload_ops(serfsim* h) {
  if (!h->ops_dirty) return 0;
  std::stable_sort(h->ops.begin(), h->ops.end(), [](const HostOp& a, const HostOp& b) { return a.tick != b.tick ? a.tick < b.tick : a.seq < b.seq; });
  const size_t n = h->ops.size();
  if (n > h->ev_cap) {
    size_t cap = std::max<size_t>(1024, h->ev_cap);
    while (cap < n) cap *= 2;
    if (h->d_ev_node) { cudaFree(h->d_ev_node); cudaFree(h->d_ev_op); cudaFree(h->d_ev_slot); }
    CU(cudaMalloc(&h->d_ev_node, cap * 4)); CU(cudaMalloc(&h->d_ev_op, cap * 4)); CU(cudaMalloc(&h->d_ev_slot, cap * 4));
    h->ev_cap = cap;
  }
  if (n) {
    std::vector<u32> a(n), b(n), c(n);
    for (size_t i = 0; i < n; ++i) { a[i] = h->ops[i].node; b[i] = h->ops[i].op; c[i] = h->ops[i].slot; }
    CU(cudaMemcpyAsync(h->d_ev_node, a.data(), n * 4, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_ev_op, b.data(), n * 4, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_ev_slot, c.data(), n * 4, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));     // staging vectors die here
  }
  h->ops_dirty = false;
  return 0;
}

bool future_ops(const serfsim* h, u32 after_tick) {       // any op scheduled at tick > after_tick
  return !h->ops.empty() && h->ops.back().tick > after_tick;
}

// Launch n ticks on the stream (no synchronisation).
int launch_ticks(serfsim* h, u32 n) {
  if (!h->has_topo) return fail(SERFSIM_E_INVAL, "serfsim_step: no topology set");
  if (h->cfg.world_size > 1 && !h->connected) return fail(SERFSIM_E_COMM, "serfsim_step: world_size > 1 but serfsim_comm_connect was not called");
  int rc = upload_ops(h);
  if (rc) return rc;
  rc = ensure_trace(h, h->tick + n + 1);
  if (rc) return rc;
  if (!h->timing_open) { CU(cudaEventRecord(h->ev0, h->stream)); h->timing_open = true; h->last_launches = 0; h->launch_log.clear(); h->launch_log_first = h->tick; }
  const bool sharded = h->cfg.world_size > 1;
  const u64* grow = sharded ? h->d_grow : h->d_trace;            // global rows: the device sums them when sharded
  for (u32 i = 0; i < n; ++i) {
    const u32 t = h->tick;
    const u64 launches_before = h->last_launches;
    auto lo = std::lower_bound(h->ops.begin(), h->ops.end(), t, [](const HostOp& o, u32 tt) { return o.tick < tt; });
    auto hi = std::upper_bound(h->ops.begin(), h->ops.end(), t, [](u32 tt, const HostOp& o) { return tt < o.tick; });
    const u32 eb = (u32)(lo - h->ops.begin()), ee = (u32)(hi - h->ops.begin());
    for (auto it = lo; it != hi; ++it) {          // ground truth the SWIM probe observes (after this tick's ops)
      const int s = slot_of(h, it->node);
      if (s >= 0) { if (it->op == SERFSIM_OP_FAIL) h->up_mask &= ~(1u << s); if (it->op == SERFSIM_OP_REJOIN) h->up_mask |= (1u << s); }
    }
    if (ee > eb) { launch_mark_events(h->d_busy, h->d_hot[(t & 1) ^ 1], h->d_ev_node, eb, ee, h->first, h->count, h->stream); h->last_launches++; }
    TickParams p{};
    p.n_local = h->count; p.first = h->first; p.n_global = h->N; p.R = h->R;
    p.fanout = h->cfg.fanout; p.probe_every = h->cfg.probe_interval_ticks; p.tick = t;
    p.down_mask = (~h->up_mask) & ((1u << h->R) - 1);
    h->ever_down |= p.down_mask;
    p.seed_lo = (u32)h->cfg.seed; p.seed_hi = (u32)(h->cfg.seed >> 32); p.ev_begin = eb; p.ev_end = ee;
    p.rules = h->rules;
    for (u32 s = 0; s < h->R; ++s) p.subj[s] = h->subj[s];
    p.rec = h->d_rec; p.qword = h->d_qword; p.inbox_rd = h->d_inbox[(t & 1) ^ 1]; p.inbox_wr = h->d_inbox[t & 1];
    p.node_state = h->d_node; p.busy = h->d_busy; p.watch = h->d_watch; p.row_ptr = h->d_rowptr; p.col = h->d_col;
    p.ev_node = h->d_ev_node; p.ev_op = h->d_ev_op; p.ev_slot = h->d_ev_slot;
    p.row = h->d_trace + (size_t)t * 8;
    p.kinds_prev = h->d_kinds + (size_t)t * 4;
    p.kinds_cur = h->d_kinds + ((size_t)t + 1) * 4;
    p.overflow = h->d_overflow;
    p.hot_rd = h->d_hot[(t & 1) ^ 1]; p.hot_wr = h->d_hot[t & 1];
    p.reap_now = (h->cfg.reap_interval_ticks && ((t + 1) % h->cfg.reap_interval_ticks) == 0) ? 1u : 0u;
    p.tombstone_ticks = h->cfg.tombstone_timeout_ticks; p.reconnect_ticks = h->cfg.reconnect_timeout_ticks; p.intent_ticks = h->cfg.recent_intent_timeout_ticks;
    p.stride = h->stride; p.n_tiles = h->n_tiles; p.tiles_per_cta = (h->n_tiles + h->grid - 1) / h->grid;
    p.force_all = (h->cfg.trace != 0) || h->no_skip || p.reap_now;
    p.compact = h->compact ? 1u : 0u;
    p.udeg = h->udeg; p.ahead = h->ahead;
    p.tile_due = h->d_tile_due; p.node_due = h->d_node_due; p.hot_static = h->d_hot_static; p.sched = h->d_sched;
    p.sleep_on = (h->no_skip || h->byz_on) ? 0u : 1u;          // injectors send every tick: the cluster never sleeps
    p.pp_every = (u32)std::max(0, h->cfg.push_pull_interval_ticks); p.reap_every = h->cfg.reap_interval_ticks;
    p.host_idle_until = h->d_pin_ctl + 2;
    const u32 xpar = h->xepoch & 1;
    p.world = (u32)h->cfg.world_size; p.rank = (u32)h->cfg.rank; p.shard_size = h->shard_size; p.win_cap = h->win_cap;
    p.win_data = h->d_peer_data[xpar]; p.send_count = h->d_send_count;
    p.peer_ctrl = h->d_peer_ctrl; p.stamp = h->xepoch + 1; p.xpar = xpar; p.loopback = h->loopback ? 1u : 0u;
    p.fuse_publish = (sharded && !h->byz_on && !getenv("SERFSIM_NO_FUSE")) ? 1u : 0u;
    p.shard_inv = (u32)(0x100000000ull / h->shard_size); p.xcap = p.world > 1 ? 392u / (p.world - 1) : 0u;     // XW_TOTAL = 392 (tick_kernel.cu)
    Gate gate{};                                   // convergence gate: the first kernel of the tick evaluates the row of tick t-1
    if (h->gate_on) {
      gate.ctl = h->d_runctl; gate.host_ctl = h->d_pin_ctl; gate.prev_row = t > h->gate_first ? grow + (size_t)(t - 1) * 8 : nullptr; gate.tick = t;
      gate.future_ops = (t > 0 && future_ops(h, t - 1)) ? 1u : 0u;
      gate.pp = (u32)std::max(0, h->cfg.push_pull_interval_ticks); gate.byz_on = h->byz_on ? 1u : 0u;
    }
    const u32* gate_word = h->gate_on ? h->d_runctl : nullptr;
    p.gate = gate; p.gate.evaluate = h->ue_table.n ? 0u : 1u;
    if (h->tick_timing) {
      while (h->tick_ev.size() < 2 * ((size_t)t + 1)) { cudaEvent_t e; CU(cudaEventCreate(&e)); h->tick_ev.push_back(e); }
      CU(cudaEventRecord(h->tick_ev[2 * (size_t)t], h->stream));
    }
    if (h->ue_table.n) {                       // user-event tick: needs the pre-operation up flags and op bits, so it runs first
      UeParams u{};
      u.n_local = h->count; u.first = h->first; u.n_global = h->N; u.R = h->R; u.fanout = h->cfg.fanout; u.tick = t;
      u.seed_lo = p.seed_lo; u.seed_hi = p.seed_hi; u.limit = h->rules.limit; u.ev_begin = eb; u.ev_end = ee;
      u.table = h->ue_table; u.state = h->d_ue_state; u.inbox_rd = h->d_ue_inbox[(t & 1) ^ 1]; u.inbox_wr = h->d_ue_inbox[t & 1];
      u.ltime = h->d_ue_ltime; u.node_state = h->d_node; u.busy = h->d_busy; u.row_ptr = h->d_rowptr; u.col = h->d_col;
      u.ev_node = h->d_ev_node; u.ev_op = h->d_ev_op; u.ev_slot = h->d_ev_slot;
      u.row = p.row; u.totals = h->d_ue_totals; u.overflow = h->d_overflow; u.sched = h->d_sched;
      u.world = (u32)h->cfg.world_size; u.rank = (u32)h->cfg.rank; u.shard_size = h->shard_size; u.win_cap = h->win_cap;
      u.win_data = h->d_peer_data[h->xepoch & 1]; u.send_count = h->d_send_count;
      u.gate = gate; u.gate.evaluate = 1u;
      launch_uevent(u, h->cfg.trace != 0, h->stream);
      h->last_launches++;
    }
    // Multi-slot runs in production mode: the general kernel and the single-view kernel are both launched, the device decides (SV_*)
    const bool sv_ok = h->sv && h->R > 1 && h->R < 32 && !h->cfg.trace && p.sleep_on && !h->byz_on && __builtin_popcount(h->ever_down) == 1;
    if (sv_ok) {
      const bool all = ee > eb || p.reap_now;                 // a host operation or a reaper round visits every view
      p.views_host = all ? 0xffffffffu : h->ever_down;
      p.sv_mode = h->sv == 2 ? SV_CHECK : SV_GENERAL;
      p.sv_slot = (u32)__builtin_ctz(h->ever_down); p.sv_R = h->R;
    }
    launch_tick(p, h->cfg.trace != 0, h->grid, h->stream);
    h->last_launches++;
    if (sv_ok && h->sv == 1) {
      TickParams q = p;                                    // the planes as the single-slot kernel sees them: they start at view sv_slot
      const u32 s0 = p.sv_slot;
      q.sv_mode = SV_SINGLE; q.gate.evaluate = 0u; q.sv_wshift = s0;
      q.rec = p.rec + 2 * (size_t)s0 * h->stride; q.qword = p.qword + (size_t)s0 * h->stride;
      q.inbox_rd = p.inbox_rd + (size_t)s0 * h->stride; q.inbox_wr = p.inbox_wr + (size_t)s0 * h->stride;
      q.subj[0] = p.subj[s0]; q.down_mask = (p.down_mask >> s0) & 1u;
      q.tiles_per_cta = (h->n_tiles + h->grid_sv - 1) / h->grid_sv;
      launch_tick_single_view(q, h->grid_sv, h->stream);
      h->last_launches++;
    }
    if (h->byz_n) {                            // stale entries of this shard's injectors (before the exchange: peers in other shards get window entries)
      ByzParams b{};
      b.n_byz = h->byz_n; b.first = h->first; b.R = h->R; b.stride = h->stride; b.fanout = h->cfg.fanout; b.tick = t;
      b.seed_lo = p.seed_lo; b.seed_hi = p.seed_hi; b.delta = h->byz_delta; b.ids = h->d_byz_ids; b.rec = h->d_rec; b.node_state = h->d_node;
      b.row_ptr = h->d_rowptr; b.col = h->d_col; b.inbox_wr = h->d_inbox[t & 1]; b.hot_wr = h->d_hot[t & 1]; b.kinds_cur = p.kinds_cur;
      b.anomaly = h->d_anomaly; b.totals = h->d_byz_totals;
      b.n_local = h->count; b.world = p.world; b.rank = p.rank; b.shard_size = h->shard_size; b.win_cap = h->win_cap;
      b.win_data = p.win_data; b.send_count = h->d_send_count; b.overflow = h->d_overflow; b.gate = gate_word;
      launch_byz(b, h->stream);
      h->last_launches++;
    }
    if (h->tick_timing && h->cfg.world_size > 1) {
      while (h->mid_ev.size() < (size_t)t + 1) { cudaEvent_t e; CU(cudaEventCreate(&e)); h->mid_ev.push_back(e); }
      CU(cudaEventRecord(h->mid_ev[t], h->stream));
    }
    if (h->cfg.world_size > 1) {
      // No host round trip: publish (counts + flag into every peer's control block) and drain (waits for the
      // peers' flags of this exchange) are ordinary kernels on the same stream.
      const u32 stamp = h->xepoch + 1;
      PublishParams pb{};
      pb.world = p.world; pb.rank = p.rank; pb.stamp = stamp; pb.xpar = xpar; pb.send_count = h->d_send_count; pb.peer_ctrl = h->d_peer_ctrl;
      pb.row = p.row; pb.gate = gate_word; pb.sched = h->d_sched; pb.loopback = h->loopback ? 1u : 0u;
      if (!p.fuse_publish) { launch_publish(pb, h->stream); h->last_launches++; }
      DrainParams d{};
      d.n_local = h->count; d.stride = h->stride; d.R = h->R; d.world = p.world; d.rank = p.rank; d.win_cap = h->win_cap; d.stamp = stamp; d.n_tiles = h->n_tiles; d.kinds_prev = p.kinds_prev;
      d.win_data = h->d_win_data[xpar]; d.ctrl = h->d_ctrl + xpar * 16; d.inbox_wr = h->d_inbox[t & 1]; d.hot_wr = h->d_hot[t & 1]; d.kinds_cur = h->d_kinds + ((size_t)t + 1) * 4; d.overflow = h->d_overflow;
      d.byz_on = h->byz_on ? 1u : 0u; d.byz_delta = h->byz_delta; d.shard_size = h->shard_size; d.rec = h->d_rec; d.node_state = h->d_node; d.peer_anomaly = h->d_peer_anomaly;
      d.ue_n = h->ue_table.n; d.ue_inbox_wr = h->ue_table.n ? h->d_ue_inbox[t & 1] : nullptr; d.ue_ltime = h->d_ue_ltime;
      d.my_row = p.row; d.grow = h->d_grow + (size_t)t * 8; d.gate = gate_word;
      d.sums = reinterpret_cast<const u64*>(reinterpret_cast<const unsigned char*>(h->d_ctrl) + CTRL_SUMS_OFF) + (size_t)xpar * 8 * CTRL_FIELDS;
      d.sched = h->d_sched; d.sched_rw = h->d_sched; d.host_idle_until = h->d_pin_ctl + 2; d.tick = t; d.sleep_on = p.sleep_on;
      launch_drain(d, h->stream);
      h->last_launches += 1;
      h->xepoch++;
    }
    const u32 pp = (u32)std::max(0, h->cfg.push_pull_interval_ticks);
    if (pp && (t + 1) % pp == 0) {
      // anti-entropy round on a snapshot of the end-of-tick state (only this node's own records are written)
      const size_t rb = (size_t)h->R * h->stride * 32, nb = (size_t)h->stride * 8;
      if (!h->d_snap_rec) { CU(cudaMalloc(&h->d_snap_rec, rb)); CU(cudaMalloc(&h->d_snap_node, nb)); }
      CU(cudaMemcpyAsync(h->d_snap_rec, h->d_rec, rb, cudaMemcpyDeviceToDevice, h->stream));
      CU(cudaMemcpyAsync(h->d_snap_node, h->d_node, nb, cudaMemcpyDeviceToDevice, h->stream));
      if (h->ue_table.n) {
        CU(cudaMemcpyAsync(h->d_ue_snap, h->d_ue_state, (size_t)h->stride * 16, cudaMemcpyDeviceToDevice, h->stream));
        p.ue_table = h->ue_table; p.ue_state = h->d_ue_state; p.ue_snap = h->d_ue_snap; p.ue_snap_peer = h->d_peer_ue_snap;
        p.ue_ltime = h->d_ue_ltime; p.ue_totals = h->d_ue_totals;
      }
      if (h->cfg.world_size > 1) {
        // partners may live on other GPUs: their snapshots are read through the peer mappings.  Rounds are rare (every
        // push_pull_interval ticks) and always the first tick of a convergence chunk, so two host barriers are affordable:
        // every rank has taken its snapshot before anyone reads, everyone has read before anyone moves on.
        p.snap_rec_peer = h->d_peer_snap_rec; p.snap_node_peer = h->d_peer_snap_node;
        CU(cudaStreamSynchronize(h->stream));
        h->barrier(h->comm_user);
        if (h->ue_table.n) {
          // A partner in another shard may hold events this shard has never received, so their Lamport times are not in the
          // local table yet (a shard learns them from the first window entry of the event).  The replay needs them: the
          // origin's shard contributes its stamp, the others 0, and every rank installs the sum before the round.
          u32 lt[MAX_UEVENTS];
          u64 v[MAX_UEVENTS];
          CU(cudaMemcpy(lt, h->d_ue_ltime, sizeof(lt), cudaMemcpyDeviceToHost));
          for (u32 e = 0; e < MAX_UEVENTS; ++e) v[e] = (((h->ue_injected >> e) & 1u) && h->ue_origin[e] - h->first < h->count) ? lt[e] : 0;
          h->allreduce(h->comm_user, v, MAX_UEVENTS);
          for (u32 e = 0; e < MAX_UEVENTS; ++e) lt[e] = (u32)v[e];
          CU(cudaMemcpy(h->d_ue_ltime, lt, sizeof(lt), cudaMemcpyHostToDevice));
        }
        launch_pushpull(p, h->d_snap_rec, h->d_snap_node, h->cfg.trace != 0, h->stream);
        CU(cudaStreamSynchronize(h->stream));
        h->barrier(h->comm_user);
        // the round changed this rank's row (changed / pending / hash) after the drain kernel summed the rows: redo the sum through
        // the host hook — the host is in the loop here anyway (two barriers), and rounds are rare
        u64 row[8];
        CU(cudaMemcpy(row, h->d_trace + (size_t)t * 8, sizeof(row), cudaMemcpyDeviceToHost));
        h->allreduce(h->comm_user, row, 8);
        CU(cudaMemcpy(h->d_grow + (size_t)t * 8, row, sizeof(row), cudaMemcpyHostToDevice));
      } else {
        launch_pushpull(p, h->d_snap_rec, h->d_snap_node, h->cfg.trace != 0, h->stream);
      }
      h->last_launches++;
    }
    if (h->tick_timing) CU(cudaEventRecord(h->tick_ev[2 * (size_t)t + 1], h->stream));
    h->launch_log.push_back((u32)(h->last_launches - launches_before));
    h->tick++;
  }
  CU(cudaGetLastError());
  return 0;
}

int finish_timing(serfsim* h) {
  if (!h->timing_open) return 0;
  CU(cudaEventRecord(h->ev1, h->stream));
  CU(cudaEventSynchronize(h->ev1));
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->last_ms = ms; h->timing_open = false; h->launches += h->last_launches;
  return 0;
}

int check_overflow(serfsim* h) {
  if (h->ue_table.n) {
    // Cluster runs need one Lamport time per ring slot: the packed event record derives a slot's ltime from the events in it.
    // (Two tracked events 512·k apart would alias — the quirk itself is kept in ue_handle and pinned by the handler tests.)
    u32 lt[MAX_UEVENTS];
    CU(cudaMemcpy(lt, h->d_ue_ltime, sizeof(lt), cudaMemcpyDeviceToHost));
    if (h->cfg.world_size > 1 && h->allreduce) {           // the origin's shard holds the stamp; the others may not have seen it yet
      u64 v[MAX_UEVENTS];
      for (u32 e = 0; e < MAX_UEVENTS; ++e) v[e] = (((h->ue_injected >> e) & 1u) && h->ue_origin[e] - h->first < h->count) ? lt[e] : 0;
      h->allreduce(h->comm_user, v, MAX_UEVENTS);
      for (u32 e = 0; e < MAX_UEVENTS; ++e) lt[e] = (u32)v[e];
    }
    for (u32 a = 0; a < h->ue_table.n; ++a)
      for (u32 b = a + 1; b < h->ue_table.n; ++b) {
        const bool fa = ((h->ue_injected >> a) & 1u) && h->ue_fire_tick[a] < h->tick, fb = ((h->ue_injected >> b) & 1u) && h->ue_fire_tick[b] < h->tick;
        if (fa && fb && lt[a] % UE_RING == lt[b] % UE_RING && lt[a] != lt[b])
          return fail(SERFSIM_E_INVAL, "user events: two tracked events share a ring slot with different Lamport times (not supported in cluster runs)");
      }
  }
  CU(cudaStreamSynchronize(h->stream));
  const u32 ov = *(volatile u32*)h->pin_overflow;
  if (ov == 1) return fail(SERFSIM_E_OVERFLOW, "a Lamport time or incarnation left the 32-bit device range");
  if (ov == 2) return fail(SERFSIM_E_COMM, "cross-shard window overflow (raise SERFSIM_WIN_FACTOR)");
  if (ov == 4) return fail(SERFSIM_E_INVAL, "single-view check (SERFSIM_SV=2): a view outside the set of views with business had business");
  if (ov) return fail(SERFSIM_E_COMM, "corrupt cross-shard window entry");
  return 0;
}

int pull_rows(serfsim* h) {                     // bring rows [rows.size(), tick) to the host (global sums when sharded)
  const u32 have = (u32)h->rows.size();
  if (have >= h->tick) return 0;
  const u32 n = h->tick - have;
  h->rows.resize(h->tick);
  // sharded runs: the drain kernel of every tick has already summed the ranks' rows on the device (d_grow), no host collective
  const u64* src = h->cfg.world_size > 1 ? h->d_grow : h->d_trace;
  CU(cudaMemcpy(h->rows.data() + have, src + (size_t)have * 8, (size_t)n * sizeof(serfsim_tick_row_t), cudaMemcpyDeviceToHost));
  return 0;
}

int fire_events(serfsim* h) {
  if (!h->cb) return 0;
  const u32 nout = 2 + 2 * h->R;
  std::vector<u64> init(nout, 0), out(nout);
  for (u32 s = 0; s < h->R; ++s) init[2 + 2 * s] = ~0ull;
  CU(cudaMemcpyAsync(h->d_scratch, init.data(), nout * 8, cudaMemcpyHostToDevice, h->stream));
  launch_summary(h->d_rec, h->d_qword, h->d_node, h->count, h->stride, h->first, h->R, h->d_subj, h->d_scratch, h->stream);
  CU(cudaMemcpyAsync(out.data(), h->d_scratch, nout * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (u32 type = 0; type < 3; ++type) {
    std::vector<u32> ids;
    for (u32 s = 0; s < h->R; ++s) {
      if (out[2 + 2 * s] != out[3 + 2 * s]) continue;                 // views still disagree
      const u8 status = (u8)((out[2 + 2 * s] >> 4) & 0xf);
      const u32 ty = status == ST_ALIVE ? SERFSIM_EVENT_JOIN : status == ST_FAILED ? SERFSIM_EVENT_FAILED : SERFSIM_EVENT_LEAVE;
      if (ty == type && h->reported[s] != status) ids.push_back(h->subj[s]);
    }
    if (!ids.empty()) h->cb(h->cb_user, h->tick, type, ids.data(), (u32)ids.size());
  }
  for (u32 s = 0; s < h->R; ++s) if (out[2 + 2 * s] == out[3 + 2 * s]) h->reported[s] = (u8)((out[2 + 2 * s] >> 4) & 0xf);
  return 0;
}

// Watcher masks depend on topology and subjects; the busy bit / hot tiles of the watchers are re-applied after every reset.
int refresh_watchers(serfsim* h) {
  if (!h->has_topo) return 0;
  if (h->watch_dirty) {
    launch_compute_watch(h->d_rowptr, h->d_col, h->d_subj, h->R, h->first, h->count, h->d_watch, h->stream);
    h->watch_dirty = false;
  }
  CU(cudaMemsetAsync(h->d_hot_static, 0, h->n_tiles, h->stream));
  launch_apply_watch(h->d_watch, h->count, h->d_busy, h->d_hot_static, h->stream);
  CU(cudaGetLastError());
  return 0;
}

int ue_reset(serfsim* h) {                      // bootstrap event state: clock 1, nothing seen, nothing queued
  h->ue_injected = 0;
  if (!h->ue_table.n) return 0;
  launch_ue_init(h->d_ue_state, h->count, h->stream);
  CU(cudaMemsetAsync(h->d_ue_inbox[0], 0, (size_t)h->stride * 4, h->stream));
  CU(cudaMemsetAsync(h->d_ue_inbox[1], 0, (size_t)h->stride * 4, h->stream));
  CU(cudaMemsetAsync(h->d_ue_ltime, 0, MAX_UEVENTS * 4, h->stream));
  CU(cudaMemsetAsync(h->d_ue_totals, 0, 8 * 8, h->stream));
  CU(cudaGetLastError());
  return 0;
}

int do_reset(serfsim* h, u64 seed) {
  h->cfg.seed = seed; h->tick = 0; h->ops.clear(); h->op_keys.clear(); h->ops_dirty = false; h->rows.clear();
  h->up_mask = (h->R >= 32) ? 0xffffffffu : ((1u << h->R) - 1);
  h->ever_down = 0;
  h->reported.assign(h->R, (u8)ST_ALIVE);
  const size_t inbox_bytes = (size_t)3 * h->R * h->stride * sizeof(u32);
  launch_init_state(h->d_rec, h->d_node, h->count, h->stride, h->R, h->cfg.init_status_ltime, h->cfg.init_clock, h->stream);
  CU(cudaMemsetAsync(h->d_inbox[0], 0, inbox_bytes, h->stream));
  CU(cudaMemsetAsync(h->d_inbox[1], 0, inbox_bytes, h->stream));
  CU(cudaStreamSynchronize(h->stream));                   // no kernel of an earlier run is still writing the error word
  *(volatile u32*)h->pin_overflow = 0;
  ((volatile u32*)h->pin_ctl)[2] = 0;                     // the scheduler's "sleep until" word (mirrors d_sched, cleared below)
  CU(cudaMemsetAsync(h->d_busy, 0, h->stride, h->stream));
  CU(cudaMemsetAsync(h->d_qword, 0, (size_t)h->R * h->stride * 4, h->stream));
  CU(cudaMemsetAsync(h->d_hot[0], 0, h->n_tiles, h->stream));
  CU(cudaMemsetAsync(h->d_hot[1], 0, h->n_tiles, h->stream));
  CU(cudaMemsetAsync(h->d_tile_due, 0xff, (size_t)h->n_tiles * sizeof(u32), h->stream));      // no timer runs
  CU(cudaMemsetAsync(h->d_node_due, 0xff, (size_t)h->stride * sizeof(u32), h->stream));
  CU(cudaMemsetAsync(h->d_sched, 0, SCHED_WORDS * sizeof(u32), h->stream));
  if (h->d_trace) {
    CU(cudaMemsetAsync(h->d_trace, 0, (size_t)h->trace_cap * 8 * sizeof(u64), h->stream));
    CU(cudaMemsetAsync(h->d_kinds, 0, ((size_t)h->trace_cap + 1) * 4 * sizeof(u32), h->stream));
  }
  if (h->d_grow) CU(cudaMemsetAsync(h->d_grow, 0, (size_t)h->trace_cap * 8 * sizeof(u64), h->stream));
  CU(cudaMemsetAsync(h->d_runctl, 0, 2 * sizeof(u32), h->stream));
  if (h->d_send_count) CU(cudaMemsetAsync(h->d_send_count, 0, sizeof(u32) * 8, h->stream));
  { int rc = ue_reset(h); if (rc) return rc; }
  if (h->d_anomaly) { CU(cudaMemsetAsync(h->d_anomaly, 0, h->stride, h->stream)); CU(cudaMemsetAsync(h->d_byz_totals, 0, 4 * 8, h->stream)); }
  { int rc = refresh_watchers(h); if (rc) return rc; }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

void free_all(serfsim* h) {
  for (void* p : h->ipc_opened) cudaIpcCloseMemHandle(p);
  for (cudaEvent_t e : h->tick_ev) cudaEventDestroy(e);
  cudaFree(h->d_hot_static); cudaFree(h->d_tile_due); cudaFree(h->d_node_due); cudaFree(h->d_sched);
  cudaFree(h->d_hot[0]); cudaFree(h->d_hot[1]); cudaFree(h->d_busy); cudaFree(h->d_watch); cudaFree(h->d_snap_rec); cudaFree(h->d_snap_node); cudaFree(h->d_peer_snap_rec); cudaFree(h->d_peer_snap_node);
  cudaFree(h->d_qword);
  cudaFree(h->d_rec); cudaFree(h->d_inbox[0]); cudaFree(h->d_inbox[1]); cudaFree(h->d_node); cudaFree(h->d_rowptr); cudaFree(h->d_col);
  cudaFree(h->d_ev_node); cudaFree(h->d_ev_op); cudaFree(h->d_ev_slot); cudaFree(h->d_trace); cudaFree(h->d_kinds); cudaFree(h->d_ones);
  if (h->pin_overflow) cudaFreeHost(h->pin_overflow);
  cudaFree(h->d_subj); cudaFree(h->d_scratch); cudaFree(h->d_stage);
  cudaFree(h->d_byz_ids); cudaFree(h->d_anomaly); cudaFree(h->d_byz_totals); cudaFree(h->d_peer_anomaly);
  cudaFree(h->d_ue_snap); cudaFree(h->d_peer_ue_snap);
  cudaFree(h->d_ue_state); cudaFree(h->d_ue_inbox[0]); cudaFree(h->d_ue_inbox[1]); cudaFree(h->d_ue_ltime); cudaFree(h->d_ue_totals);
  for (int par = 0; par < 2; ++par) { cudaFree(h->d_win_data[par]); cudaFree(h->d_peer_data[par]); }
  cudaFree(h->d_ctrl); cudaFree(h->d_send_count); cudaFree(h->d_peer_ctrl);
  for (auto& b : h->res) { cudaFree(b.d); if (b.copied) cudaEventDestroy(b.copied); }
  if (h->ev_extracted) cudaEventDestroy(h->ev_extracted);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->pin_ctl) cudaFreeHost(h->pin_ctl);
  cudaFree(h->d_runctl); cudaFree(h->d_grow);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
}

int getter(serfsim* h, u32 slot, int what, void* out, size_t elem) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  if (what != EXTRACT_CLOCK && what != EXTRACT_CLOCK32 && slot >= h->R) return fail(SERFSIM_E_INVAL, "slot out of range");
  launch_extract(h->d_rec, h->d_node, h->count, h->stride, slot, what, h->d_stage, h->stream);
  CU(cudaMemcpyAsync(out, h->d_stage, (size_t)h->count * elem, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

}  // namespace

// hooks for wire_codec.cu (the other translation unit behind the C ABI)
namespace sfs {
struct WireView { const uint4* rec; const u32* qword; const u64* node_state; const uint4* ue_state; const u32* subj; u32 n_local, stride, R; cudaStream_t stream; };
int serfsim_fail(int code, const char* msg) { return fail(code, msg); }
int serfsim_wire_view(const serfsim* h, WireView* out) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  *out = WireView{h->d_rec, h->d_qword, h->d_node, h->ue_table.n ? h->d_ue_state : nullptr, h->d_subj, h->count, h->stride, h->R, h->stream};
  return 0;
}
}  // namespace sfs

// =====================================================================================
// C ABI
// =====================================================================================
#pragma GCC visibility push(default)
extern "C" {

uint32_t serfsim_abi_version(void) { return SERFSIM_ABI_VERSION; }
const char* serfsim_last_error(void) { return g_err.c_str(); }

void serfsim_default_config(serfsim_config_t* c) {
  if (!c) return;
  memset(c, 0, sizeof(*c));
  c->abi_version = SERFSIM_ABI_VERSION;
  c->n_nodes = 0; c->slots = 1;
  c->fanout = 3;                       // memberlist LAN gossip_nodes
  c->retransmit_mult = 4; c->suspicion_mult = 4; c->suspicion_max_timeout_mult = 6;
  c->probe_interval_ticks = 5;         // 1 s / 200 ms
  c->gossip_interval_ms = 200;
  c->init_status_ltime = 1; c->init_clock = 2;
  c->trace = 0; c->seed = 1; c->device = -1; c->rank = 0; c->world_size = 1;
  c->push_pull_interval_ticks = 0;     // LAN: 30 s = 150 ticks × pushPullScale(n); off unless asked for
  c->reap_interval_ticks = 0;          // options.rs:506: 15 s = 75 ticks; off unless asked for
  c->tombstone_timeout_ticks = 432000; c->reconnect_timeout_ticks = 432000;   // 24 h (options.rs:508-509)
  c->recent_intent_timeout_ticks = 1500;                                     // 5 min (options.rs:515)
}

int serfsim_create(const serfsim_config_t* cfg, serfsim_t** out) {
  if (!cfg || !out) return fail(SERFSIM_E_INVAL, "null argument");
  *out = nullptr;
  if (cfg->abi_version != SERFSIM_ABI_VERSION) return fail(SERFSIM_E_INVAL, "abi_version mismatch");
  if (cfg->n_nodes < 2 || cfg->slots < 1 || cfg->slots > MAX_SLOTS || cfg->fanout < 1 || cfg->fanout > MAX_FANOUT)
    return fail(SERFSIM_E_INVAL, "bad n_nodes / slots (1..16) / fanout (1..8)");
  if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size) return fail(SERFSIM_E_INVAL, "bad rank / world_size");
  if (cfg->gossip_interval_ms == 0) return fail(SERFSIM_E_INVAL, "gossip_interval_ms must be > 0");
  if (cfg->push_pull_interval_ticks < 0) return fail(SERFSIM_E_INVAL, "push_pull_interval_ticks must be >= 0");
  if (cfg->suspicion_mult >= 2 && cfg->suspicion_mult - 2 > MAX_K) return fail(SERFSIM_E_INVAL, "suspicion_mult too large");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(SERFSIM_E_NO_DEVICE, "no CUDA device: serfsim has no CPU execution path");
  if (cfg->device >= 0) { if (cfg->device >= ndev) return fail(SERFSIM_E_NO_DEVICE, "device ordinal out of range"); CU(cudaSetDevice(cfg->device)); }
  int dev = 0, major = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return fail(SERFSIM_E_NO_DEVICE, "kernels are built for sm_100a only (B200)");

  serfsim* h = new serfsim();
  h->cfg = *cfg; h->N = cfg->n_nodes; h->R = cfg->slots;
  h->shard_size = (h->N + cfg->world_size - 1) / cfg->world_size;
  h->first = std::min<u64>((u64)h->shard_size * cfg->rank, h->N);
  h->count = (u32)std::min<u64>(h->shard_size, (u64)h->N - h->first);
  if (h->count == 0) { delete h; return fail(SERFSIM_E_INVAL, "empty shard"); }
  if (h->shard_size >= (1u << 26)) { delete h; return fail(SERFSIM_E_INVAL, "shard larger than 2^26 nodes"); }
  h->rules.limit = retransmit_limit(cfg->retransmit_mult, h->N);
  if (h->rules.limit == 0 || h->rules.limit > 255) { delete h; return fail(SERFSIM_E_INVAL, "retransmit limit must be 1..255"); }
  auto tab = suspicion_table(cfg->suspicion_mult, cfg->suspicion_max_timeout_mult, cfg->probe_interval_ticks ? cfg->probe_interval_ticks : 1, cfg->gossip_interval_ms, h->N);
  h->rules.k = (u32)tab.size() - 1;
  for (size_t i = 0; i < tab.size(); ++i) h->rules.timeout[i] = tab[i];
  h->subj.resize(h->R);
  for (u32 s = 0; s < h->R; ++s) h->subj[s] = s;

  auto bail = [&](int rc) { free_all(h); delete h; return rc; };
#define CUB(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return bail(fail(e_ == cudaErrorMemoryAllocation ? SERFSIM_E_NOMEM : SERFSIM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_))); } while (0)
  CUB(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CUB(cudaEventCreate(&h->ev0)); CUB(cudaEventCreate(&h->ev1));
  h->stride = ((h->count + 255) / 256) * 256;
  const size_t inbox_bytes = (size_t)3 * h->R * h->stride * sizeof(u32);
  CUB(cudaMalloc(&h->d_rec, (size_t)h->R * h->stride * 32));
  CUB(cudaMemset(h->d_rec, 0, (size_t)h->R * h->stride * 32));
  CUB(cudaMalloc(&h->d_qword, (size_t)h->R * h->stride * 4));
  CUB(cudaMemset(h->d_qword, 0, (size_t)h->R * h->stride * 4));
  CUB(cudaMalloc(&h->d_inbox[0], inbox_bytes)); CUB(cudaMalloc(&h->d_inbox[1], inbox_bytes));
  CUB(cudaMalloc(&h->d_node, (size_t)h->stride * 8));
  CUB(cudaMemset(h->d_node, 0, (size_t)h->stride * 8));
  h->n_tiles = (h->count + 255) / 256;
  CUB(cudaMalloc(&h->d_busy, h->stride));
  CUB(cudaMalloc(&h->d_watch, (size_t)h->stride * 2));
  CUB(cudaMemset(h->d_watch, 0, (size_t)h->stride * 2));
  CUB(cudaMalloc(&h->d_hot[0], h->n_tiles)); CUB(cudaMalloc(&h->d_hot[1], h->n_tiles));
  CUB(cudaMalloc(&h->d_hot_static, h->n_tiles)); CUB(cudaMalloc(&h->d_tile_due, (size_t)h->n_tiles * sizeof(u32))); CUB(cudaMalloc(&h->d_node_due, (size_t)h->stride * sizeof(u32))); CUB(cudaMalloc(&h->d_sched, SCHED_WORDS * sizeof(u32)));
  CUB(cudaMemset(h->d_hot_static, 0, h->n_tiles));
  CUB(cudaHostAlloc(&h->pin_overflow, sizeof(u32), cudaHostAllocMapped));
  CUB(cudaHostGetDevicePointer(&h->d_overflow, h->pin_overflow, 0));
  *h->pin_overflow = 0;
  CUB(cudaMalloc(&h->d_subj, MAX_SLOTS * 4)); CUB(cudaMalloc(&h->d_scratch, 64 * 8));
  CUB(cudaMalloc(&h->d_stage, (size_t)h->count * 8));
  CUB(cudaMalloc(&h->d_runctl, 2 * sizeof(u32)));
  CUB(cudaMemset(h->d_runctl, 0, 2 * sizeof(u32)));
  CUB(cudaHostAlloc(&h->pin_ctl, 4 * sizeof(u32), cudaHostAllocMapped));
  CUB(cudaHostGetDevicePointer(&h->d_pin_ctl, h->pin_ctl, 0));
  h->pin_ctl[0] = h->pin_ctl[1] = h->pin_ctl[2] = h->pin_ctl[3] = 0;
  CUB(cudaMalloc(&h->d_ones, 16));
  const u32 ones[4] = {0x40000000u, 0x40000000u, 0x40000000u, 1u};   // multi-GPU: every inbox plane may hold entries, every tick is dense
  CUB(cudaMemcpy(h->d_ones, ones, 16, cudaMemcpyHostToDevice));
  CUB(cudaMemcpy(h->d_subj, h->subj.data(), h->R * 4, cudaMemcpyHostToDevice));
  h->ctas_per_sm = (h->R == 1) ? (cfg->world_size > 1 ? tick_ctas_per_sm_r1s() : tick_ctas_per_sm_r1()) : tick_ctas_per_sm_rn();
  h->grid = tick_grid_size(h->count, h->ctas_per_sm);
  h->grid_sv = tick_grid_size(h->count, cfg->world_size > 1 ? tick_ctas_per_sm_r1s() : tick_ctas_per_sm_r1());
  if (const char* e = getenv("SERFSIM_NO_SKIP")) h->no_skip = atoi(e) != 0;
  if (const char* e = getenv("SERFSIM_COMPACT")) h->compact = atoi(e) != 0;
  if (const char* e = getenv("SERFSIM_AHEAD")) h->ahead = (u32)std::min(2, std::max(0, atoi(e)));
  if (const char* e = getenv("SERFSIM_SV")) h->sv = (u32)std::min(2, std::max(0, atoi(e)));
  if (cfg->world_size > 1) {
    // receive windows: one segment per peer; expected entries per tick and pair ≈ shard · fanout · R · kinds / world
    if (cfg->world_size > 8) return bail(fail(SERFSIM_E_INVAL, "world_size > 8"));
    double factor = 1.25;
    if (const char* e = getenv("SERFSIM_WIN_FACTOR")) factor = atof(e);
    // … plus the entries the warps of the tick kernel reserve ahead and do not fill (flush_xwarp: at most XW_RESERVE_MAX = 128 per warp and peer)
    const double pad = (double)std::max(tick_grid_size(h->count, h->ctas_per_sm), h->grid_sv) * 8.0 * 160.0;   // (the single-view kernel of a multi-slot run has the larger grid)
    double cap = (double)h->shard_size * cfg->fanout * h->R * 3.0 * factor / cfg->world_size + 4096.0 + pad;
    h->win_cap = (u32)std::min(cap, 4.0e9);
    h->win_cap_base = h->win_cap;
    for (int par = 0; par < 2; ++par) {
      CUB(cudaMalloc(&h->d_win_data[par], (size_t)cfg->world_size * h->win_cap * 8));
      CUB(cudaMemset(h->d_win_data[par], 0, (size_t)cfg->world_size * h->win_cap * 8));      // windows read as zeros wherever nothing was written
      CUB(cudaMalloc(&h->d_peer_data[par], sizeof(u64*) * 8));
    }
    CUB(cudaMalloc(&h->d_ctrl, CTRL_BYTES));
    CUB(cudaMemset(h->d_ctrl, 0, CTRL_BYTES));
    CUB(cudaMalloc(&h->d_send_count, 8 * sizeof(u32)));
    CUB(cudaMemset(h->d_send_count, 0, 8 * sizeof(u32)));
    CUB(cudaMalloc(&h->d_peer_ctrl, sizeof(u32*) * 8));
    CUB(cudaMalloc(&h->d_anomaly, h->stride)); CUB(cudaMemset(h->d_anomaly, 0, h->stride));   // byzantine sender flags: peers' drain kernels raise them
    CUB(cudaMalloc(&h->d_byz_totals, 4 * 8)); CUB(cudaMemset(h->d_byz_totals, 0, 4 * 8));
    CUB(cudaMalloc(&h->d_peer_anomaly, sizeof(void*) * 8));
    if (cfg->push_pull_interval_ticks > 0) {      // the snapshots partners on other GPUs read: allocated now so that they can be exported
      CUB(cudaMalloc(&h->d_snap_rec, (size_t)h->R * h->stride * 32));
      CUB(cudaMalloc(&h->d_snap_node, (size_t)h->stride * 8));
      CUB(cudaMalloc(&h->d_peer_snap_rec, sizeof(void*) * 8));
      CUB(cudaMalloc(&h->d_peer_snap_node, sizeof(void*) * 8));
    }
  }
  {
    int rc = ensure_trace(h, 1024);
    if (rc) return bail(rc);
    rc = do_reset(h, cfg->seed);
    if (rc) return bail(rc);
  }
#undef CUB
  *out = h;
  return 0;
}

void serfsim_destroy(serfsim_t* h) {
  if (!h) return;
  cudaStreamSynchronize(h->stream);
  if (getenv("SERFSIM_XTIMING") && !h->mid_ev.empty()) {
    double a = 0, b = 0; size_t n = std::min(h->mid_ev.size(), h->tick_ev.size() / 2);
    for (size_t t = 0; t < n; ++t) {
      float x = 0, y = 0;
      if (cudaEventElapsedTime(&x, h->tick_ev[2 * t], h->mid_ev[t]) == cudaSuccess && cudaEventElapsedTime(&y, h->mid_ev[t], h->tick_ev[2 * t + 1]) == cudaSuccess) {
        a += x; b += y;
        if (t >= 12 && t <= 15) fprintf(stderr, "rank %d tick %zu: tick kernel %.1f us, publish+drain %.1f us\n", h->cfg.rank, t, x * 1e3, y * 1e3);
      }
    }
    fprintf(stderr, "rank %d: tick kernels %.3f ms, publish+drain %.3f ms over %zu ticks\n", h->cfg.rank, a, b, n);
  }
  free_all(h);
  delete h;
}

int serfsim_set_topology_csr(serfsim_t* h, const uint64_t* row_ptr, const uint32_t* col_idx) {
  if (!h || !row_ptr || !col_idx) return fail(SERFSIM_E_INVAL, "null argument");
  if (row_ptr[0] != 0) return fail(SERFSIM_E_INVAL, "row_ptr[0] must be 0");
  const u64 e0 = row_ptr[h->first], e1 = row_ptr[h->first + h->count];
  if (e1 < e0 || e1 - e0 >= 0xffffffffull) return fail(SERFSIM_E_INVAL, "shard has too many edges (u32 offsets)");
  std::vector<u32> rp((size_t)h->stride + 8);
  for (u32 i = 0; i <= h->count; ++i) {
    const u64 r = row_ptr[h->first + i];
    if (r < e0 || (i && r < row_ptr[h->first + i - 1])) return fail(SERFSIM_E_INVAL, "row_ptr not monotone");
    if (i && r - row_ptr[h->first + i - 1] > 65535) return fail(SERFSIM_E_INVAL, "node degree > 65535 (peer draws are 16-bit)");
    rp[i] = (u32)(r - e0);
  }
  const u64 ne = e1 - e0;
  h->udeg = (h->count && ne % h->count == 0) ? (u32)(ne / h->count) : 0u;
  for (u32 i = 0; i <= h->count && h->udeg; ++i) if (rp[i] != (u64)i * h->udeg) h->udeg = 0;
  for (size_t i = h->count + 1; i < rp.size(); ++i) rp[i] = (u32)ne;      // padding rows: degree 0
  for (u64 i = 0; i < ne; ++i) if (col_idx[e0 + i] >= h->N) return fail(SERFSIM_E_INVAL, "col_idx out of range");
  cudaFree(h->d_rowptr); cudaFree(h->d_col); h->d_rowptr = nullptr; h->d_col = nullptr;
  CU(cudaMalloc(&h->d_rowptr, rp.size() * 4));
  CU(cudaMalloc(&h->d_col, (ne + 8) * 4));
  CU(cudaMemset(h->d_col, 0, (ne + 8) * 4));
  CU(cudaMemcpy(h->d_rowptr, rp.data(), rp.size() * 4, cudaMemcpyHostToDevice));
  if (ne) CU(cudaMemcpy(h->d_col, col_idx + e0, ne * 4, cudaMemcpyHostToDevice));
  if (getenv("SERFSIM_VERBOSE")) fprintf(stderr, "serfsim: tick kernel = tick_kernel (grid %d)\n", h->grid);
  h->has_topo = true;
  h->watch_dirty = true;
  return refresh_watchers(h);
}

int serfsim_set_subjects(serfsim_t* h, const uint32_t* subjects) {
  if (!h || !subjects) return fail(SERFSIM_E_INVAL, "null argument");
  if (h->tick != 0) return fail(SERFSIM_E_INVAL, "subjects can only change at tick 0");
  for (u32 i = 0; i < h->R; ++i) {
    if (subjects[i] >= h->N) return fail(SERFSIM_E_INVAL, "subject id out of range");
    for (u32 j = 0; j < i; ++j) if (subjects[j] == subjects[i]) return fail(SERFSIM_E_INVAL, "subjects must be distinct");
  }
  h->subj.assign(subjects, subjects + h->R);
  CU(cudaMemcpy(h->d_subj, h->subj.data(), h->R * 4, cudaMemcpyHostToDevice));
  h->watch_dirty = true;
  // tick 0 with a clean state: re-derive the watchers' busy bits / hot tiles for the new subjects
  CU(cudaMemsetAsync(h->d_busy, 0, h->stride, h->stream));
  CU(cudaMemsetAsync(h->d_hot[0], 0, h->n_tiles, h->stream));
  CU(cudaMemsetAsync(h->d_hot[1], 0, h->n_tiles, h->stream));
  return refresh_watchers(h);
}

int serfsim_reset(serfsim_t* h, uint64_t seed) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  return do_reset(h, seed);
}

int serfsim_inject(serfsim_t* h, uint32_t tick, uint32_t op, uint32_t node, uint32_t slot) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  if (tick < h->tick) return fail(SERFSIM_E_INVAL, "cannot schedule an operation in the past");
  if (node >= h->N || op < SERFSIM_OP_JOIN || op > SERFSIM_OP_FORCE_LEAVE_PRUNE) return fail(SERFSIM_E_INVAL, "bad node / op");
  if (op == SERFSIM_OP_USER_EVENT) {
    if (slot >= h->ue_table.n) return fail(SERFSIM_E_INVAL, "user event index out of range (serfsim_set_user_events)");
    if ((h->ue_injected >> slot) & 1u) return fail(SERFSIM_E_INVAL, "a tracked user event can be injected once");
  }
  if (op == SERFSIM_OP_FORCE_LEAVE || op == SERFSIM_OP_FORCE_LEAVE_PRUNE) { if (slot >= h->R) return fail(SERFSIM_E_INVAL, "slot out of range"); }
  else if ((op == SERFSIM_OP_JOIN || op == SERFSIM_OP_LEAVE) && slot_of(h, node) < 0)
    return fail(SERFSIM_E_INVAL, "join/leave origin must be a tracked subject");
  if (!h->op_keys.insert(((u64)tick << 32) | node).second) return fail(SERFSIM_E_INVAL, "one operation per node per tick");
  if (op == SERFSIM_OP_USER_EVENT) { h->ue_injected |= 1u << slot; h->ue_origin[slot] = node; h->ue_fire_tick[slot] = tick; }
  h->ops.push_back(HostOp{tick, op, node, slot, h->op_seq++});
  h->ops_dirty = true;
  return 0;
}

int serfsim_step(serfsim_t* h, uint32_t n_ticks) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  int rc = launch_ticks(h, n_ticks);
  if (rc) return rc;
  rc = finish_timing(h);
  if (rc) return rc;
  rc = check_overflow(h);
  if (rc) return rc;
  return fire_events(h);
}

int serfsim_run_until_converged(serfsim_t* h, uint32_t max_ticks, uint32_t* ticks_out) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  // Ticks are launched in chunks WITHOUT looking at their rows: the first kernel of every tick evaluates the quiescence rule
  // on the previous tick's (global) row on the device and, once the run is over, it and every later kernel return at once
  // (tick_kernel.cuh: Gate).  The host reads two words per chunk; ranks of a sharded run reach the same verdict from the same
  // device-summed rows, so there is no host collective in the loop.  Ticks launched past the first quiescent one never
  // execute: nothing to rewind on the device, the logical clock (and the exchange epoch) is simply set back.
  // Chunks start small and grow (8, 16, 32) — and start small again after every jump over a sleeping stretch: a tick launched into a
  // cluster that has just gone to sleep (or has just finished) still costs its launches (5 – 11 µs: two kernels per tick in multi-slot
  // runs; in sharded runs it even executes), a synchronisation costs less than two of them.  The leave + fail study (877 ticks, ≈ 70 of
  // them busy) launched 382 ticks per run with chunks of up to 128.
  u32 chunk = 8, chunk_max = 32;
  if (const char* e = getenv("SERFSIM_CHUNK")) chunk = chunk_max = (u32)std::max(1, atoi(e));
  const bool host_jump = !getenv("SERFSIM_NO_JUMP");
  const u32 pp = (u32)std::max(0, h->cfg.push_pull_interval_ticks);
  const u32 start = h->tick;
  int rc = 0;
  CU(cudaMemsetAsync(h->d_runctl, 0, 2 * sizeof(u32), h->stream));
  h->pin_ctl[0] = h->pin_ctl[1] = 0;                   // nothing of an earlier call is in flight: every call ends synchronised
  h->gate_on = true; h->gate_first = start;
  struct GateOff { serfsim* h; ~GateOff() { h->gate_on = false; } } gate_off{h};
  auto finish = [&](u32 converged_at, bool converged) -> int {
    if ((rc = finish_timing(h))) return rc;
    if ((rc = check_overflow(h))) return rc;
    if (ticks_out) *ticks_out = converged_at;
    if ((rc = fire_events(h))) return rc;
    return converged ? 0 : 1;
  };
  auto stop_at = [&](u32 t) {                         // tick t is the first quiescent one: later launches did not execute
    const u32 skipped = h->tick - (t + 1);
    if (h->cfg.world_size > 1) h->xepoch -= skipped;   // skipped ticks exchanged nothing
    h->tick = t + 1;
    if (h->rows.size() > h->tick) h->rows.resize(h->tick);
    u64 executed = 0;                                  // kernels of the ticks that did run (launch_log starts at launch_log_first)
    for (u32 k = 0; k < h->launch_log.size() && h->launch_log_first + k <= t; ++k) executed += h->launch_log[k];
    h->last_launches = executed;
  };
  bool probe = false;                                  // the next launch is the single tick whose gate judges the row the jump starts from
  while (h->tick - start < max_ticks) {
    const u32 n = probe ? 1u : std::min(chunk, max_ticks - (h->tick - start));
    if ((rc = launch_ticks(h, n))) return rc;
    CU(cudaStreamSynchronize(h->stream));
    if (getenv("SERFSIM_DEBUG_LOOP")) fprintf(stderr, "loop: launched %u ticks -> tick %u, ctl %u %u until %u probe %d chunk %u\n", n, h->tick, h->pin_ctl[0], h->pin_ctl[1], h->pin_ctl[2], (int)probe, chunk);
    if (*(volatile u32*)h->pin_ctl) {
      const u32 t = ((volatile u32*)h->pin_ctl)[1];
      stop_at(t);
      return finish(t, true);
    }
    if (!probe) chunk = std::min(chunk * 2, chunk_max);
    // The last executed tick proved that nothing can happen before tick `until` (tick_kernel.cu: finish_tick): the ticks up to
    // there — and up to the next host operation — are not even launched; one small kernel writes their rows.  The rows a jump
    // produces equal the row before it, and that one must have been judged "not quiescent" by a gate first: a jump is
    // preceded by one single-tick launch (`probe`).
    const u32 until = ((volatile u32*)h->pin_ctl)[2];
    const bool sleeping = host_jump && until > h->tick && h->tick - start < max_ticks;      // sharded runs: every rank reads the same word
    // … and the probe tick itself must have been an idle one: with a host operation in it (which may well change nothing) its row is a new
    // one that no gate has judged yet — the next launch is another single tick (found by fuzz scenario 16 once the launch chunks ended
    // on the tick before a no-op operation: the run was reported quiescent at the end of the jump instead of at the operation's tick)
    bool probe_was_idle = true;
    if (probe && h->tick > 0) {
      auto it = std::lower_bound(h->ops.begin(), h->ops.end(), h->tick - 1, [](const HostOp& o, u32 tt) { return o.tick < tt; });
      probe_was_idle = it == h->ops.end() || it->tick != h->tick - 1;
    }
    if (sleeping && probe && probe_was_idle) {
      u32 stop = until;
      auto nxt = std::lower_bound(h->ops.begin(), h->ops.end(), h->tick, [](const HostOp& o, u32 tt) { return o.tick < tt; });
      if (nxt != h->ops.end()) stop = std::min(stop, nxt->tick);
      const u32 n_skip = std::min(stop > h->tick ? stop - h->tick : 0u, max_ticks - (h->tick - start));
      if (n_skip) {
        if ((rc = ensure_trace(h, h->tick + n_skip + 1))) return rc;
        launch_fill_idle_rows(h->d_trace + (size_t)h->tick * 8, h->cfg.world_size > 1 ? h->d_grow + (size_t)h->tick * 8 : nullptr, n_skip, h->d_sched, h->cfg.trace != 0, h->stream);
        h->last_launches++;
        SFS_COUNT(17, n_skip);                           // ticks the host jumped over
        for (u32 k = 0; k < n_skip; ++k) {
          if (h->tick_timing) {
            const u32 t = h->tick + k;
            while (h->tick_ev.size() < 2 * ((size_t)t + 1)) { cudaEvent_t e; CU(cudaEventCreate(&e)); h->tick_ev.push_back(e); }
            CU(cudaEventRecord(h->tick_ev[2 * (size_t)t], h->stream)); CU(cudaEventRecord(h->tick_ev[2 * (size_t)t + 1], h->stream));
          }
          h->launch_log.push_back(k == 0 ? 1u : 0u);
        }
        h->tick += n_skip;
        if (!getenv("SERFSIM_CHUNK")) chunk = 8;            // the busy stretch after a sleep is short as a rule
      }
      probe = false;
    } else {
      probe = sleeping;
    }
  }
  // max_ticks reached: the last tick's row has not been judged by any kernel yet — apply the same rule here
  if (h->tick > start) {
    if ((rc = pull_rows(h))) return rc;
    const u32 t = h->tick - 1;
    if (quiescent_row((const u64*)&h->rows[t], t, future_ops(h, t), pp, h->byz_on)) return finish(t, true);
  }
  return finish(h->tick, false);
}

int serfsim_shard_range(serfsim_t* h, uint32_t* first, uint32_t* count) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  if (first) *first = h->first;
  if (count) *count = h->count;
  return 0;
}
int serfsim_member_status(serfsim_t* h, uint32_t slot, uint8_t* out) { return getter(h, slot, EXTRACT_STATUS, out, 1); }
int serfsim_status_ltime(serfsim_t* h, uint32_t slot, uint64_t* out) { return getter(h, slot, EXTRACT_STATUS_LTIME, out, 8); }
int serfsim_lamport_time(serfsim_t* h, uint64_t* out) { return getter(h, 0, EXTRACT_CLOCK, out, 8); }
// compact variants: the device keeps Lamport times in 32 bits (a run that would leave that range fails with SERFSIM_E_OVERFLOW), so
// the same values can cross PCIe at half the size
int serfsim_status_ltime_u32(serfsim_t* h, uint32_t slot, uint32_t* out) { return getter(h, slot, EXTRACT_STATUS_LTIME32, out, 4); }
int serfsim_lamport_time_u32(serfsim_t* h, uint32_t* out) { return getter(h, 0, EXTRACT_CLOCK32, out, 4); }
int serfsim_incarnation(serfsim_t* h, uint32_t slot, uint32_t* out) { return getter(h, slot, EXTRACT_INC, out, 4); }
int serfsim_ml_state(serfsim_t* h, uint32_t slot, uint8_t* out) { return getter(h, slot, EXTRACT_ML, out, 1); }

// The step's result vectors without stalling the launch stream: the three extractions run on the launch stream (in order after
// the ticks), the device→host copies on a second stream.  The caller may start its next step at once; the copies overlap its
// ticks.  Host buffers must stay valid (and should be pinned) until serfsim_results_wait returns.
int serfsim_results_async(serfsim_t* h, uint32_t slot, uint8_t* status, uint32_t* status_ltime, uint32_t* lamport) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  if (slot >= h->R) return fail(SERFSIM_E_INVAL, "slot out of range");
  if (!h->copy_stream) { CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking)); CU(cudaEventCreate(&h->ev_extracted)); }
  serfsim::ResBuf& b = h->res[h->res_next++ & 3u];
  const size_t n = h->count, n4 = ((n * 4 + 255) / 256) * 256;
  if (!b.d) { CU(cudaMalloc(&b.d, 2 * n4 + n)); CU(cudaEventCreate(&b.copied)); }
  if (b.used) CU(cudaStreamWaitEvent(h->stream, b.copied, 0));            // the copy that last read this staging buffer has finished
  if (status_ltime) launch_extract(h->d_rec, h->d_node, h->count, h->stride, slot, EXTRACT_STATUS_LTIME32, b.d, h->stream);
  if (lamport) launch_extract(h->d_rec, h->d_node, h->count, h->stride, slot, EXTRACT_CLOCK32, b.d + n4, h->stream);
  if (status) launch_extract(h->d_rec, h->d_node, h->count, h->stride, slot, EXTRACT_STATUS, b.d + 2 * n4, h->stream);
  CU(cudaEventRecord(h->ev_extracted, h->stream));
  CU(cudaStreamWaitEvent(h->copy_stream, h->ev_extracted, 0));
  if (status_ltime) CU(cudaMemcpyAsync(status_ltime, b.d, n * 4, cudaMemcpyDeviceToHost, h->copy_stream));
  if (lamport) CU(cudaMemcpyAsync(lamport, b.d + n4, n * 4, cudaMemcpyDeviceToHost, h->copy_stream));
  if (status) CU(cudaMemcpyAsync(status, b.d + 2 * n4, n, cudaMemcpyDeviceToHost, h->copy_stream));
  CU(cudaEventRecord(b.copied, h->copy_stream));
  b.used = true;
  return 0;
}
int serfsim_results_wait(serfsim_t* h) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  if (h->copy_stream) CU(cudaStreamSynchronize(h->copy_stream));
  return 0;
}

int serfsim_records(serfsim_t* h, uint32_t slot, void* out) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  if (slot >= h->R) return fail(SERFSIM_E_INVAL, "slot out of range");
  uint4* tmp = nullptr;                          // merged image: record | transmit budgets of the queue word
  CU(cudaMalloc(&tmp, (size_t)h->count * 32));
  launch_compose_records(h->d_rec, h->d_qword, h->count, h->stride, slot, tmp, h->stream);
  cudaError_t e = cudaMemcpyAsync(out, tmp, (size_t)h->count * 32, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(tmp);
  if (e != cudaSuccess) return fail(SERFSIM_E_CUDA, cudaGetErrorString(e));
  return 0;
}

int serfsim_tick_trace(serfsim_t* h, uint32_t first_tick, uint32_t n, serfsim_tick_row_t* out) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  if ((u64)first_tick + n > h->tick) return fail(SERFSIM_E_INVAL, "trace range beyond the executed ticks");
  CU(cudaStreamSynchronize(h->stream));
  int rc = pull_rows(h);
  if (rc) return rc;
  memcpy(out, h->rows.data() + first_tick, (size_t)n * sizeof(serfsim_tick_row_t));
  return 0;
}

int serfsim_state_hash(serfsim_t* h, uint64_t* out) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  CU(cudaMemsetAsync(h->d_scratch, 0, 4 * 8, h->stream));
  launch_state_hash(h->d_rec, h->d_qword, h->d_node, h->count, h->stride, h->first, h->N, h->R, h->d_scratch, h->stream);
  if (h->ue_table.n) launch_ue_summary(h->d_ue_state, h->count, h->first, h->N, h->R, h->ue_table.n, h->d_scratch + 1, h->stream);
  u64 parts[4] = {0, 0, 0, 0};
  CU(cudaMemcpyAsync(parts, h->d_scratch, 4 * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  *out = parts[0] + parts[3];                    // records + node words, plus the event records when user events are on
  if (h->cfg.world_size > 1) {
    if (!h->allreduce) return fail(SERFSIM_E_COMM, "world_size > 1: serfsim_comm_set_hooks was not called");
    h->allreduce(h->comm_user, out, 1);
  }
  return 0;
}

int serfsim_stats(serfsim_t* h, serfsim_stats_t* o) {
  if (!h || !o) return fail(SERFSIM_E_INVAL, "null argument");
  memset(o, 0, sizeof(*o));
  CU(cudaStreamSynchronize(h->stream));
  int rc = pull_rows(h);
  if (rc) return rc;
  o->tick = h->tick; o->members = h->N;
  for (size_t i = 0; i < h->rows.size(); ++i) {
    const auto& r = h->rows[i];
    o->packets += r.packets; o->edge_updates += r.edge_updates; o->messages += r.messages; o->changed += r.changed; o->events += r.events;
    if (r.pending || r.edge_updates || r.events) o->last_active_tick = i;
  }
  if (!h->rows.empty()) o->pending = h->rows.back().pending;
  const u32 nout = 2 + 2 * h->R;
  std::vector<u64> init(nout, 0), out(nout);
  for (u32 s = 0; s < h->R; ++s) init[2 + 2 * s] = ~0ull;
  CU(cudaMemcpyAsync(h->d_scratch, init.data(), nout * 8, cudaMemcpyHostToDevice, h->stream));
  launch_summary(h->d_rec, h->d_qword, h->d_node, h->count, h->stride, h->first, h->R, h->d_subj, h->d_scratch, h->stream);
  CU(cudaMemcpyAsync(out.data(), h->d_scratch, nout * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  o->member_time = out[0]; o->intent_queue = out[1];
  for (u32 s = 0; s < h->R; ++s) if (out[2 + 2 * s] != ~0ull && out[2 + 2 * s] != out[3 + 2 * s]) o->disagree_slots++;
  return 0;
}

// ---- byzantine injectors (BASELINE configs[4]; model in byz.cuh) ----
int serfsim_set_byzantine(serfsim_t* h, uint32_t n, const uint32_t* ids, uint32_t delta) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  if (n && !ids) return fail(SERFSIM_E_INVAL, "null ids");
  if (h->tick != 0 || !h->ops.empty()) return fail(SERFSIM_E_INVAL, "serfsim_set_byzantine: call before any operation is scheduled (or after serfsim_reset)");
  if (n && h->cfg.world_size > 1 && h->shard_size >= BYZ_FLAG) return fail(SERFSIM_E_INVAL, "byzantine injectors: shards must hold fewer than 2^25 nodes");
  std::vector<u32> v(ids, ids + n);
  std::sort(v.begin(), v.end());
  for (u32 i = 0; i < n; ++i) if (v[i] >= h->N || (i && v[i] == v[i - 1])) return fail(SERFSIM_E_INVAL, "byzantine ids must be distinct node ids");
  std::vector<u32> mine;                           // every rank is given the global list and keeps the injectors of its shard
  for (u32 id : v) if (id - h->first < h->count) mine.push_back(id);
  cudaFree(h->d_byz_ids); h->d_byz_ids = nullptr;
  h->byz_n = 0; h->byz_delta = delta; h->byz_on = n != 0;
  if (n) {
    if (!h->d_anomaly) { CU(cudaMalloc(&h->d_anomaly, h->stride)); CU(cudaMalloc(&h->d_byz_totals, 4 * 8)); }
    if (!mine.empty()) {
      CU(cudaMalloc(&h->d_byz_ids, mine.size() * 4));
      CU(cudaMemcpy(h->d_byz_ids, mine.data(), mine.size() * 4, cudaMemcpyHostToDevice));
    }
    CU(cudaMemset(h->d_anomaly, 0, h->stride));
    CU(cudaMemset(h->d_byz_totals, 0, 4 * 8));
    h->byz_n = (u32)mine.size();
  }
  return 0;
}

int serfsim_anomaly_flags(serfsim_t* h, uint8_t* out) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  if (!h->byz_on) return fail(SERFSIM_E_INVAL, "no byzantine injectors set (serfsim_set_byzantine)");
  CU(cudaStreamSynchronize(h->stream));
  if (h->cfg.world_size > 1) {                     // peers' drain kernels raise flags in this array: wait until every rank has drained
    if (!h->barrier) return fail(SERFSIM_E_COMM, "world_size > 1: serfsim_comm_set_hooks was not called");
    h->barrier(h->comm_user);
  }
  CU(cudaMemcpy(out, h->d_anomaly, h->count, cudaMemcpyDeviceToHost));
  return 0;
}

int serfsim_byzantine_stats(serfsim_t* h, serfsim_byz_stats_t* o) {
  if (!h || !o) return fail(SERFSIM_E_INVAL, "null argument");
  if (!h->byz_on) return fail(SERFSIM_E_INVAL, "no byzantine injectors set (serfsim_set_byzantine)");
  u64 t[4] = {0, 0, 0, 0};
  CU(cudaStreamSynchronize(h->stream));
  if (h->cfg.world_size > 1) {
    if (!h->barrier || !h->allreduce) return fail(SERFSIM_E_COMM, "world_size > 1: serfsim_comm_set_hooks was not called");
    h->barrier(h->comm_user);                      // see serfsim_anomaly_flags
  }
  CU(cudaMemcpy(t, h->d_byz_totals, 4 * 8, cudaMemcpyDeviceToHost));
  std::vector<u8> flags(h->count);
  CU(cudaMemcpy(flags.data(), h->d_anomaly, h->count, cudaMemcpyDeviceToHost));
  u64 v[3] = {t[0], t[1], 0};
  for (u8 f : flags) v[2] += f ? 1 : 0;
  if (h->cfg.world_size > 1) h->allreduce(h->comm_user, v, 3);
  o->messages = v[0]; o->edge_updates = v[1]; o->flagged = v[2];
  return 0;
}

// ---- user events (SURVEY §8f row 3; rules in uevent.cuh) ----
int serfsim_set_user_events(serfsim_t* h, uint32_t n_events, const uint32_t* content_ids) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  if (n_events > MAX_UEVENTS) return fail(SERFSIM_E_INVAL, "at most SERFSIM_MAX_USER_EVENTS tracked user events");
  if (n_events && !content_ids) return fail(SERFSIM_E_INVAL, "null content ids");
  if (h->tick != 0 || !h->ops.empty()) return fail(SERFSIM_E_INVAL, "serfsim_set_user_events: call before any operation is scheduled (or after serfsim_reset)");
  if (h->cfg.world_size > 1) {
    // every event bit bound for another shard is one window entry: up to fanout · n_events per node and tick on top of the
    // membership entries the windows were sized for.  The windows are exported by serfsim_comm_export, so this must come first.
    double factor = 1.25;
    if (const char* e = getenv("SERFSIM_WIN_FACTOR")) factor = atof(e);
    const double cap = (double)h->win_cap_base + (double)h->shard_size * h->cfg.fanout * n_events * factor / h->cfg.world_size;
    const u32 want = (u32)std::min(cap, 4.0e9);
    if (want != h->win_cap) {
      if (h->connected) return fail(SERFSIM_E_INVAL, "serfsim_set_user_events: in sharded runs call it before serfsim_comm_export / serfsim_comm_connect (it resizes the receive windows)");
      for (int par = 0; par < 2; ++par) {
        cudaFree(h->d_win_data[par]); h->d_win_data[par] = nullptr;
        CU(cudaMalloc(&h->d_win_data[par], (size_t)h->cfg.world_size * want * 8));
        CU(cudaMemset(h->d_win_data[par], 0, (size_t)h->cfg.world_size * want * 8));
      }
      h->win_cap = want;
    }
  }
  if (n_events && !h->d_ue_state) {
    CU(cudaMalloc(&h->d_ue_state, (size_t)h->stride * 16));
    CU(cudaMalloc(&h->d_ue_inbox[0], (size_t)h->stride * 4));
    CU(cudaMalloc(&h->d_ue_inbox[1], (size_t)h->stride * 4));
    CU(cudaMalloc(&h->d_ue_ltime, MAX_UEVENTS * 4));
    CU(cudaMalloc(&h->d_ue_totals, 8 * 8));
  }
  if (n_events && h->cfg.push_pull_interval_ticks > 0 && !h->d_ue_snap) {
    if (h->connected) return fail(SERFSIM_E_INVAL, "serfsim_set_user_events: in sharded runs with push-pull rounds call it before serfsim_comm_export (the event snapshot is exported)");
    CU(cudaMalloc(&h->d_ue_snap, (size_t)h->stride * 16));
    CU(cudaMalloc(&h->d_peer_ue_snap, sizeof(void*) * 8));
  }
  h->ue_table = UeTable{};
  h->ue_table.n = n_events;
  for (u32 e = 0; e < n_events; ++e) h->ue_table.content[e] = content_ids[e];
  int rc = ue_reset(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int serfsim_event_time(serfsim_t* h, uint64_t* out) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  if (!h->ue_table.n) return fail(SERFSIM_E_INVAL, "user events are off (serfsim_set_user_events)");
  launch_ue_extract(h->d_ue_state, h->count, 0, 0, h->d_stage, h->stream);
  CU(cudaMemcpyAsync(out, h->d_stage, (size_t)h->count * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int serfsim_user_event_seen(serfsim_t* h, uint32_t event, uint8_t* out) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  if (event >= h->ue_table.n) return fail(SERFSIM_E_INVAL, "user event index out of range");
  launch_ue_extract(h->d_ue_state, h->count, 1, event, h->d_stage, h->stream);
  CU(cudaMemcpyAsync(out, h->d_stage, (size_t)h->count, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int serfsim_user_event_ltime(serfsim_t* h, uint32_t event, uint64_t* ltime) {
  if (!h || !ltime) return fail(SERFSIM_E_INVAL, "null argument");
  if (event >= h->ue_table.n) return fail(SERFSIM_E_INVAL, "user event index out of range");
  u32 v = 0;
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpy(&v, h->d_ue_ltime + event, 4, cudaMemcpyDeviceToHost));
  *ltime = v;
  if (h->cfg.world_size > 1) {                      // the origin's shard stamped it; the others contribute 0 to the sum
    if (!h->allreduce) return fail(SERFSIM_E_COMM, "world_size > 1: serfsim_comm_set_hooks was not called");
    const bool scheduled = (h->ue_injected >> event) & 1u;
    if (!scheduled || h->ue_origin[event] - h->first >= h->count) *ltime = 0;
    h->allreduce(h->comm_user, ltime, 1);
  }
  return 0;
}

int serfsim_user_event_records(serfsim_t* h, void* out) {
  if (!h || !out) return fail(SERFSIM_E_INVAL, "null argument");
  if (!h->ue_table.n) return fail(SERFSIM_E_INVAL, "user events are off (serfsim_set_user_events)");
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpy(out, h->d_ue_state, (size_t)h->count * 16, cudaMemcpyDeviceToHost));
  return 0;
}

int serfsim_user_event_stats(serfsim_t* h, serfsim_uevent_stats_t* o) {
  if (!h || !o) return fail(SERFSIM_E_INVAL, "null argument");
  memset(o, 0, sizeof(*o));
  if (!h->ue_table.n) return fail(SERFSIM_E_INVAL, "user events are off (serfsim_set_user_events)");
  u64 tot[8] = {0}, sum[3] = {0, 0, 0};
  CU(cudaMemsetAsync(h->d_scratch, 0, 3 * 8, h->stream));
  launch_ue_summary(h->d_ue_state, h->count, h->first, h->N, h->R, h->ue_table.n, h->d_scratch, h->stream);
  CU(cudaMemcpyAsync(sum, h->d_scratch, 3 * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(tot, h->d_ue_totals, 8 * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  u64 v[6] = {tot[0], tot[1], tot[2], tot[3], tot[4], sum[0]};
  if (h->cfg.world_size > 1) {                      // counters are sums over shards; event_time (a maximum) stays shard-local
    if (!h->allreduce) return fail(SERFSIM_E_COMM, "world_size > 1: serfsim_comm_set_hooks was not called");
    h->allreduce(h->comm_user, v, 6);
  }
  o->messages = v[0]; o->edge_updates = v[1]; o->delivered = v[2]; o->duplicates = v[3]; o->too_old = v[4];
  o->event_queue = v[5]; o->event_time = sum[1];
  return 0;
}

int serfsim_set_event_cb(serfsim_t* h, serfsim_event_cb cb, void* user) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  h->cb = cb; h->cb_user = user;
  return 0;
}

int serfsim_last_step_device_ms(serfsim_t* h, double* ms, uint64_t* kernel_launches) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  if (ms) *ms = h->last_ms;
  if (kernel_launches) *kernel_launches = h->last_launches;
  return 0;
}

int serfsim_set_tick_timing(serfsim_t* h, int enabled) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  h->tick_timing = enabled != 0;
  return 0;
}

int serfsim_tick_times(serfsim_t* h, uint32_t first_tick, uint32_t n, float* ms_out) {
  if (!h || !ms_out) return fail(SERFSIM_E_INVAL, "null argument");
  if (((size_t)first_tick + n) * 2 > h->tick_ev.size()) return fail(SERFSIM_E_INVAL, "tick timing was not enabled for that range");
  CU(cudaStreamSynchronize(h->stream));
  for (u32 i = 0; i < n; ++i) CU(cudaEventElapsedTime(ms_out + i, h->tick_ev[2 * ((size_t)first_tick + i)], h->tick_ev[2 * ((size_t)first_tick + i) + 1]));
  return 0;
}

// ---- multi-GPU: CUDA IPC windows ----------------------------------------------------------
struct comm_blob { cudaIpcMemHandle_t data[2]; cudaIpcMemHandle_t ctrl; cudaIpcMemHandle_t snap_rec, snap_node, anomaly, ue_snap; u32 win_cap; u32 rank; u32 has_snap; u32 has_ue_snap; unsigned char dev_uuid[16]; };

size_t serfsim_comm_blob_size(void) { return sizeof(comm_blob); }

int serfsim_comm_export(serfsim_t* h, void* blob) {
  if (!h || !blob) return fail(SERFSIM_E_INVAL, "null argument");
  if (h->cfg.world_size < 2) return fail(SERFSIM_E_INVAL, "world_size == 1: nothing to export");
  comm_blob b{};
  for (int par = 0; par < 2; ++par) CU(cudaIpcGetMemHandle(&b.data[par], h->d_win_data[par]));
  CU(cudaIpcGetMemHandle(&b.ctrl, h->d_ctrl));
  CU(cudaIpcGetMemHandle(&b.anomaly, h->d_anomaly));
  if (h->d_ue_snap) { CU(cudaIpcGetMemHandle(&b.ue_snap, h->d_ue_snap)); b.has_ue_snap = 1; }
  b.win_cap = h->win_cap; b.rank = (u32)h->cfg.rank;
#ifndef SERFSIM_EMU
  { int dev = 0; cudaDeviceProp pr{}; CU(cudaGetDevice(&dev)); CU(cudaGetDeviceProperties(&pr, dev)); memcpy(b.dev_uuid, pr.uuid.bytes, 16); }
#endif
  if (h->d_snap_rec) {                              // push-pull rounds are on: partners on other GPUs read these
    CU(cudaIpcGetMemHandle(&b.snap_rec, h->d_snap_rec)); CU(cudaIpcGetMemHandle(&b.snap_node, h->d_snap_node));
    b.has_snap = 1;
  }
  memcpy(blob, &b, sizeof(b));
  return 0;
}

int serfsim_comm_connect(serfsim_t* h, const void* blobs) {
  if (!h || !blobs) return fail(SERFSIM_E_INVAL, "null argument");
  const int W = h->cfg.world_size;
  if (W < 2) return fail(SERFSIM_E_INVAL, "world_size == 1");
  if (!h->barrier || !h->allreduce) return fail(SERFSIM_E_COMM, "serfsim_comm_set_hooks must be called first");
  const comm_blob* bs = (const comm_blob*)blobs;
  std::vector<u32*> pc(8, nullptr);
  std::vector<std::vector<u64*>> pd(2, std::vector<u64*>(8, nullptr));
  std::vector<const uint4*> psr(8, nullptr);
  std::vector<const u64*> psn(8, nullptr);
  std::vector<u8*> pan(8, nullptr);
  std::vector<const uint4*> pus(8, nullptr);
  for (int r = 0; r < W; ++r) {
    if (bs[r].rank != (u32)r || bs[r].win_cap != h->win_cap) return fail(SERFSIM_E_COMM, "blob order / window size mismatch");
#ifndef SERFSIM_EMU
    // one rank per GPU: the drain kernel spins on its peers' flags, and a peer that shares this GPU may never get an SM to raise them
    for (int r2 = 0; r2 < r; ++r2) if (!h->loopback && memcmp(bs[r].dev_uuid, bs[r2].dev_uuid, 16) == 0) return fail(SERFSIM_E_COMM, "two ranks share one GPU (one process per GPU is required)");
#endif
    if ((bs[r].has_snap != 0) != (h->d_snap_rec != nullptr)) return fail(SERFSIM_E_COMM, "push_pull_interval_ticks differs between ranks");
    if (r == h->cfg.rank) { pd[0][r] = h->d_win_data[0]; pd[1][r] = h->d_win_data[1]; pc[r] = h->d_ctrl; psr[r] = h->d_snap_rec; psn[r] = h->d_snap_node; pan[r] = h->d_anomaly; pus[r] = h->d_ue_snap; continue; }
    void* ptr = nullptr;
    if ((bs[r].has_ue_snap != 0) != (h->d_ue_snap != nullptr)) return fail(SERFSIM_E_COMM, "user events / push-pull configuration differs between ranks");
    if (bs[r].has_ue_snap) {
      cudaError_t e = cudaIpcOpenMemHandle(&ptr, bs[r].ue_snap, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) return fail(SERFSIM_E_COMM, std::string("cudaIpcOpenMemHandle(event snapshot): ") + cudaGetErrorString(e));
      h->ipc_opened.push_back(ptr); pus[r] = (const uint4*)ptr;
    }
    {
      cudaError_t e = cudaIpcOpenMemHandle(&ptr, bs[r].anomaly, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) return fail(SERFSIM_E_COMM, std::string("cudaIpcOpenMemHandle(flags): ") + cudaGetErrorString(e));
      h->ipc_opened.push_back(ptr); pan[r] = (u8*)ptr;
    }
    if (bs[r].has_snap) {
      cudaError_t e = cudaIpcOpenMemHandle(&ptr, bs[r].snap_rec, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) return fail(SERFSIM_E_COMM, std::string("cudaIpcOpenMemHandle(snapshot): ") + cudaGetErrorString(e));
      h->ipc_opened.push_back(ptr); psr[r] = (const uint4*)ptr;
      e = cudaIpcOpenMemHandle(&ptr, bs[r].snap_node, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) return fail(SERFSIM_E_COMM, std::string("cudaIpcOpenMemHandle(snapshot): ") + cudaGetErrorString(e));
      h->ipc_opened.push_back(ptr); psn[r] = (const u64*)ptr;
    }
    for (int par = 0; par < 2; ++par) {
      cudaError_t e = cudaIpcOpenMemHandle(&ptr, bs[r].data[par], cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) return fail(SERFSIM_E_COMM, std::string("cudaIpcOpenMemHandle(window): ") + cudaGetErrorString(e));
      h->ipc_opened.push_back(ptr); pd[par][r] = (u64*)ptr;
    }
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, bs[r].ctrl, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(SERFSIM_E_COMM, std::string("cudaIpcOpenMemHandle(ctrl): ") + cudaGetErrorString(e));
    h->ipc_opened.push_back(ptr); pc[r] = (u32*)ptr;
  }
  for (int par = 0; par < 2; ++par) CU(cudaMemcpy(h->d_peer_data[par], pd[par].data(), sizeof(u64*) * 8, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_peer_ctrl, pc.data(), sizeof(u32*) * 8, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_peer_anomaly, pan.data(), sizeof(void*) * 8, cudaMemcpyHostToDevice));
  if (h->d_ue_snap) CU(cudaMemcpy(h->d_peer_ue_snap, pus.data(), sizeof(void*) * 8, cudaMemcpyHostToDevice));
  if (h->d_snap_rec) {
    CU(cudaMemcpy(h->d_peer_snap_rec, psr.data(), sizeof(void*) * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->d_peer_snap_node, psn.data(), sizeof(void*) * 8, cudaMemcpyHostToDevice));
  }
  h->barrier(h->comm_user);          // every rank has mapped every window before the first tick writes into one
  h->connected = true;
  return 0;
}

int serfsim_comm_loopback(serfsim_t* h) {
  if (!h) return fail(SERFSIM_E_INVAL, "null handle");
  const int W = h->cfg.world_size;
  if (W < 2) return fail(SERFSIM_E_INVAL, "world_size == 1");
  if (h->cfg.rank != 0) return fail(SERFSIM_E_INVAL, "loopback: create the handle as rank 0");
  if (h->cfg.push_pull_interval_ticks > 0 || h->byz_on || h->ue_table.n) return fail(SERFSIM_E_INVAL, "loopback profiles the membership path only");
  // entries for shard s are written at win_data[s][rank·win_cap + g]: with rank 0 the window of "peer" s is my own segment s
  std::vector<u32*> pc(8, nullptr);
  std::vector<std::vector<u64*>> pd(2, std::vector<u64*>(8, nullptr));
  std::vector<u8*> pan(8, nullptr);
  for (int r = 0; r < W; ++r) {
    pc[r] = h->d_ctrl; pan[r] = h->d_anomaly;
    for (int par = 0; par < 2; ++par) pd[par][r] = h->d_win_data[par] + (size_t)r * h->win_cap;
  }
  for (int par = 0; par < 2; ++par) CU(cudaMemcpy(h->d_peer_data[par], pd[par].data(), sizeof(u64*) * 8, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_peer_ctrl, pc.data(), sizeof(u32*) * 8, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_peer_anomaly, pan.data(), sizeof(void*) * 8, cudaMemcpyHostToDevice));
  h->barrier = [](void*) {};
  h->allreduce = [](void*, uint64_t*, uint32_t) {};
  h->connected = true; h->loopback = true;
  return 0;
}

int serfsim_comm_set_hooks(serfsim_t* h, serfsim_barrier_fn barrier, serfsim_allreduce_u64_fn allreduce, void* user) {
  if (!h || !barrier || !allreduce) return fail(SERFSIM_E_INVAL, "null argument");
  h->barrier = barrier; h->allreduce = allreduce; h->comm_user = user;
  return 0;
}

}  // extern "C"
#pragma GCC visibility pop
