// tick_kernel.cuh — parameter block and launch interface of the device side.
#pragma once
#include <cuda_runtime.h>

#include "record.cuh"
#include "uevent.cuh"

// Kernel launch in one spelling for nvcc and for the host build of tests/emu (which defines its own SFS_LAUNCH):
//   SFS_LAUNCH(grid, block, dynamic_smem_bytes, stream, kernel<template, args>)(kernel arguments);
#if defined(SERFSIM_EMU) && defined(__CUDACC__)
#error "SERFSIM_EMU is the host-only test build of tests/emu (g++); the product is built by nvcc without it"
#endif
#ifndef SERFSIM_EMU
#define SFS_LAUNCH(grid, block, smem, stream, ...) __VA_ARGS__<<<(grid), (block), (smem), (stream)>>>
constexpr int SFS_SMS = 148;                 // B200: grid-stride helper kernels are sized in multiples of the SM count
#else
constexpr int SFS_SMS = 1;
#endif
// Coverage probes of the host build (tests assert that a code path was actually taken); nothing under nvcc.
#ifdef SERFSIM_EMU
#define SFS_PROBE(i) (emu::probes[i]++)
#define SFS_COUNT(i, n) (emu::probes[i] += (n))
#else
#define SFS_PROBE(i) ((void)0)
#define SFS_COUNT(i, n) ((void)0)
#endif

namespace sfs {

// Device-side convergence gate (serfsim_run_until_converged).  The host launches ticks in large chunks without looking at
// their rows; the FIRST kernel of tick t evaluates the quiescence rule on the (global) row of tick t-1 and, when the run is
// over, sets a sticky word — that kernel and every later kernel of the call then return at once, so ticks launched past the
// first quiescent one cost a few microseconds of launch latency and touch no state at all (no rewind, no consumed tile
// flags, no exchange epoch).  Every rank evaluates the same global row with the same parameters, so all ranks stop at the
// same tick without a host collective.  ctl[0]: done flag, ctl[1]: index of the first quiescent tick.
struct Gate {
  u32* ctl;                   // null: gating off (serfsim_step)
  u32* host_ctl;              // the same two words in mapped pinned host memory: the host reads the verdict without a device→host copy
                              // (a copy would queue behind the result vectors of the previous run on the copy engine)
  const u64* prev_row;        // global trace row of tick-1 (8 × u64); null for the first tick of a call (it always runs)
  u32 tick;                   // this tick
  u32 evaluate;               // 1: this kernel is the first of the tick's launch sequence and evaluates the rule
  u32 future_ops;             // a host operation is scheduled at a tick > tick-1
  u32 pp, byz_on;             // push-pull interval (0 = off), byzantine injectors on
};
// The quiescence rule — one definition for the device gate and the host (max_ticks boundary, serfsim.cu):
// nothing pending, nothing delivered, no operation still to come; with anti-entropy on additionally a push-pull round that
// changed nothing but Lamport times (serf/delegate.rs:495-510: status_time creeps by design); with injectors on nothing merged
// (stale entries stay in flight forever).
__host__ __device__ inline bool quiescent_row(const u64* row, u32 t, bool future_ops, u32 pp, bool byz_on) {
  const u64 edges = row[1], changed = row[3], pending = row[4];
  const bool pp_ok = !pp || (((t + 1) % pp) == 0 && changed == 0);
  const bool byz_ok = !byz_on || changed == 0;
  return pending == 0 && edges == 0 && !future_ops && pp_ok && byz_ok;
}
__device__ __forceinline__ bool gate_closed(const Gate& g, bool leader) {
  if (!g.ctl) return false;
  if (g.ctl[0]) return true;
  if (!g.evaluate || !g.prev_row) return false;
  if (!quiescent_row(g.prev_row, g.tick - 1, g.future_ops != 0, g.pp, g.byz_on != 0)) return false;
  if (leader) {                                            // every CTA of this kernel reaches the same verdict from the row itself
    g.ctl[1] = g.tick - 1; g.ctl[0] = 1;
    if (g.host_ctl) { g.host_ctl[1] = g.tick - 1; g.host_ctl[0] = 1; }   // visible to the host once the kernel has completed
  }
  return true;
}

struct TickParams {
  // geometry / run constants
  u32 n_local, first, n_global, R;
  u32 fanout, probe_every, tick, down_mask;
  u32 seed_lo, seed_hi, ev_begin, ev_end;
  Rules rules;
  u32 subj[MAX_SLOTS];
  // state in HBM
  uint4* rec;                 // [R][stride] records, 2 × uint4 each (transmit-budget bytes kept zero: they live in qword)
  u32* qword;                 // [R][stride] queue words: tx_join | tx_leave << 8 | tx_ml << 16
  u32* inbox_rd;              // [3][R][n_local] reduced inbox filled by the previous tick (value+1, 0 = empty)
  u32* inbox_wr;              // [3][R][n_local] inbox the sends of this tick reduce into
  u64* node_state;            // [n_local]  clock | up | SerfState
  u8* busy;                   // [n_local]  bit 0: pending work (queued transmits, suspicion timer); bit 1: host op this tick; bit 2: watcher (static)
  const u16* watch;           // [n_local]  bit s: subject s is in the node's neighbour list (only such nodes can probe it)
  const u32* row_ptr;         // [n_local+1] CSR offsets into col (shard-local)
  const u32* col;             // neighbour ids (global)
  const u32* ev_node;         // host operations, sorted by tick
  const u32* ev_op;
  const u32* ev_slot;
  u64* row;                   // this tick's trace row (8 × u64, zeroed)
  const u32* kinds_prev;      // [4] messages of each kind sent in the previous tick (skip empty inbox planes)
  u32* kinds_cur;             // [4] same, for this tick
  u32* overflow;              // set when a Lamport time / incarnation nears the device width
  u8* hot_rd;                 // [n_tiles] tile flags set during the previous tick (deliveries, pending work, host ops)
  u8* hot_wr;                 // [n_tiles] tile flags for the next tick
  u32 pad1, reap_now, pad2, pad3;         // reap_now: this tick the reaper runs (every view is visited); pad1 keeps the offsets of the members below
  u32 tombstone_ticks, reconnect_ticks, intent_ticks, pad4;
  u32 n_tiles, tiles_per_cta, force_all, stride;   // stride: plane stride in nodes = n_local rounded up to a whole tile
  // cross-shard exchange (world_size > 1): every rank owns one receive window per peer (mapped into the
  // peers with CUDA IPC); the tick kernel stages cross-shard entries per destination shard in shared memory
  // and writes them into the peer's window with coalesced stores over NVLink.
  u32 world, rank, shard_size, win_cap;
  u64* const* win_data;       // [world] peer windows of this exchange parity; my segment starts at rank·win_cap
  u32* send_count;            // [world] entries written so far into each peer's window (local counters)
  // sharded push-pull rounds: every rank's end-of-tick snapshot, indexed by shard (null when world == 1).  New members go
  // at the end: the tick kernels do not read them and keep their parameter offsets (and their SASS) unchanged.
  const uint4* const* snap_rec_peer; const u64* const* snap_node_peer;
  // push-pull replay of the partner's user-event ring (delegate.rs:469-474, 539-552); ue_table.n == 0: user events off
  UeTable ue_table; uint4* ue_state; const uint4* ue_snap; const uint4* const* ue_snap_peer; const u32* ue_ltime; u64* ue_totals;
  u32 compact;                // 1: unsaturated ticks gather their active nodes across several tiles (SERFSIM_COMPACT=0 switches it off)
  Gate gate;
  u32 udeg;                   // > 0: every node of the shard has this out-degree (row v starts at v·udeg): row offsets are not loaded and senders draw their peers early
  // Sleeping views (the suspicion timer wheel).  A view whose only business is a running suspicion timer is not visited tick after
  // tick: its deadline is registered in tile_due (a lower bound of the earliest deadline of the tile's 256 nodes, reset and
  // re-registered whenever it comes due), its node carries busy bit 3, and the number of such views lives in a persistent counter
  // instead of being recounted every tick.  Ticks in which provably nothing can happen (no mail, no queued transmit, no probe
  // duty, no timer due, no host operation, no anti-entropy / reaper round) return at once (sched[SCHED_IDLE_UNTIL]).
  u32* tile_due;              // [n_tiles]
  u32* node_due;              // [n_local] lower bound of the node's own earliest running deadline (exact after a visit of all its views; meaningful while busy bit 3 is set):
                              // when a tile comes due only the nodes whose own deadline has been reached visit their views, the others re-register this word
  const u8* hot_static;       // [n_tiles] tiles that hold a watcher (static; never consumed)
  u32* sched;                 // scheduler words (SCHED_*), u64 suspect-view counter at sched + SCHED_SUSPECTS
  u32 sleep_on;               // 0: SERFSIM_NO_SKIP — every tile, every view, every tick
  u32 pp_every, reap_every;   // push-pull / reaper periods in ticks (0 = off): such ticks are never skipped
  // sharded runs without injectors: the tick's LAST CTA also publishes (counts, row, verdict, release flag → every peer's control
  // block): one launch less per tick.  With injectors their kernel still writes windows after this one, and publish_kernel follows it.
  u32* const* peer_ctrl; u32 stamp, xpar, loopback, fuse_publish;
  u32 shard_inv, xcap;        // floor(2^32 / shard_size) (a remote target's shard without a division); staged entries per warp and peer
  u32 sv_wshift;              // single-view launch: its view's bit in the watch masks (0 in every other launch)
  u32 sv_mode, views_host, sv_slot, sv_R;    // single-view ticks (SV_*, below): sv_slot = the view the single-view launch works on, sv_R = number of views of the run
  u32 ahead;                  // multi-slot runs: 1 = saturated ticks request node word, peers and the probable first view's record one tile ahead; 2 = every tick (tests); 0 = off (SERFSIM_AHEAD)
  u32* host_idle_until;       // SCHED_IDLE_UNTIL mirrored into mapped pinned host memory: serfsim_run_until_converged does not even launch the ticks the cluster sleeps through
};
constexpr u32 SCHED_TICKET = 0, SCHED_IDLE_UNTIL = 1, SCHED_UE_ACTIVITY = 2, SCHED_AWAKE = 3, SCHED_SUSPECTS = 4 /* u64 */,
              SCHED_LOCAL_QUIET = 6, SCHED_LOCAL_UNTIL = 7 /* sharded runs: this rank's verdict; the drain kernel combines the ranks' */,
              SCHED_VIEWS_NEW = 8 /* single-view ticks: bit s = view s can have business, in the ticks from SCHED_VIEWS_FROM on */, SCHED_VIEWS_NEXT = 9 /* being collected */,
              SCHED_VIEWS_OLD = 10 /* the set of the tick before SCHED_VIEWS_FROM */, SCHED_VIEWS_FROM = 11, SCHED_WORDS = 12;
// Single-view ticks (multi-slot runs).  In long stretches of a study exactly one tracked subject is in motion (the suspicion and dead waves
// of a crash after the leave wave has died down): every node visits the same single view, and the lean single-slot kernel (64 registers,
// 32 warps per SM, every load requested up front) does that tick in half the time of the multi-slot kernel (128 registers, 16 warps).
// Which views can have business in tick t+1 is known at the end of tick t: views that sent mail or keep a queue (collected by the tick
// kernel, the anti-entropy kernel and — across shards — the drain kernel in SCHED_VIEWS_*), plus what the host knows (views_host: every
// subject that has ever been down — only those are probed, suspected and run timers; all views when the tick carries a host operation or a
// reaper round).  While exactly ONE subject has ever been down (sv_slot) the host launches BOTH kernels — the single-view one with a
// parameter block whose planes start at that view and whose subject / down flag are that view's — each looks at the set and one of them
// returns at once.  SV_CHECK (SERFSIM_SV=2) runs the
// general kernel alone and raises error 4 if a view outside a one-element set turns out to have business (the set must be a superset).
constexpr u32 SV_OFF = 0, SV_GENERAL = 1, SV_SINGLE = 2, SV_CHECK = 3;
constexpr u32 NO_DEADLINE = 0xffffffffu;
// A tick is skipped (grid-uniform decision of its first instruction) when the last executed tick proved that nothing can happen
// before SCHED_IDLE_UNTIL and the host scheduled no operation for it.
__device__ __forceinline__ bool tick_is_idle(const u32* sched, u32 tick, u32 ev_begin, u32 ev_end) {
  return sched && ev_begin == ev_end && tick < sched[SCHED_IDLE_UNTIL];
}

// Control block of a rank (one allocation, mapped into every peer): per exchange parity the entry counts and epoch flags
// the peers write, then the peers' trace rows of that tick (the device-side sum of the per-tick counters).
constexpr u32 CTRL_U32 = 2 * 16;                        // [parity][ counts[8] | flags[8] ]
constexpr u32 CTRL_SUMS_OFF = CTRL_U32 * 4;             // byte offset of u64 sums[2][8][CTRL_FIELDS]  ([parity][source rank][field])
constexpr u32 CTRL_FIELDS = 11;                         // the 8 trace-row fields, then the rank's scheduler verdict: 8 = quiet (0 / 1), 9 = sleep until, 10 = views with business in the next tick
constexpr size_t CTRL_BYTES = CTRL_SUMS_OFF + 2 * 8 * CTRL_FIELDS * sizeof(u64);
struct PublishParams {        // after the tick kernel: tell every peer how much was written and this rank's row, then raise its flag
  u32 world, rank, stamp, xpar;
  u32* send_count;            // [world] local, reset here
  u32* const* peer_ctrl;      // [world] peers' control blocks
  const u64* row;             // this rank's trace row of the tick (complete: the tick kernels precede the publish kernel)
  const u32* gate;            // sticky done word of the convergence gate (null: off)
  const u32* sched;           // scheduler words: the rank's verdict (quiet, sleep until) goes out with its row
  u32 loopback;               // profiling aid (serfsim_comm_loopback): every peer is this rank itself; counts / rows / flags go to the slot of the
                              // "peer" they are addressed to instead of this rank's own slot
};

struct DrainParams {
  u32 n_local, stride, R, world, rank, win_cap, stamp, n_tiles;
  const u32* kinds_prev;      // [4] the kind counters the tick kernel of this tick based its dense/sparse decision on
  u64* win_data;              // my window of this exchange parity: [world][win_cap]; entries are cleared as they are consumed
  const u32* ctrl;            // my control block of this parity: counts[8] | flags[8], written by the peers
  u32* inbox_wr;
  u8* hot_wr;
  u32* kinds_cur;             // [4] kind counters of this tick (received kinds are added so the next tick reads their planes)
  u32* overflow;
  // byzantine triples (see ByzParams): judged here against the receiver's end-of-tick record
  u32 byz_on, byz_delta, shard_size;
  const uint4* rec; const u64* node_state;
  u8* const* peer_anomaly;    // [world] every rank's sender-flag array
  // user-event entries (kind 3: slot = tracked event, value = its Lamport time + 1); null / 0 when user events are off
  u32 ue_n;
  u32* ue_inbox_wr;
  u32* ue_ltime;
  // device-side sum of the tick's trace row over all ranks: grow[i] = my_row[i] + Σ peers' published rows
  const u64* my_row; const u64* sums; u64* grow;
  const u32* gate;
  u32* sched_rw;              // the same words, writable: the peers' views with business are added to SCHED_VIEWS_CUR
  const u32* sched; u32* host_idle_until;   // the ranks' verdicts combined: every rank hands the same "sleep until" tick to its host
  u32 tick, sleep_on;
};

void launch_tick(const TickParams& p, bool trace, int grid, cudaStream_t st);
void launch_tick_single_view(const TickParams& p, int grid, cudaStream_t st);
void launch_fill_idle_rows(u64* rows, u64* grow_rows, u32 n, const u32* sched, bool trace, cudaStream_t st);
void launch_pushpull(const TickParams& p, const uint4* snap_rec, const u64* snap_node, bool trace, cudaStream_t st);
void launch_drain(const DrainParams& p, cudaStream_t st);
void launch_publish(const PublishParams& p, cudaStream_t st);
void launch_init_state(uint4* rec, u64* node_state, u32 n_local, u32 stride, u32 R, u32 init_st, u32 init_clock, cudaStream_t st);
void launch_mark_events(u8* busy, u8* hot_rd, const u32* ev_node, u32 ev_begin, u32 ev_end, u32 first, u32 n_local, cudaStream_t st);
void launch_extract(const uint4* rec, const u64* node_state, u32 n_local, u32 stride, u32 slot, int what, void* out, cudaStream_t st);
void launch_compose_records(const uint4* rec, const u32* qword, u32 n_local, u32 stride, u32 slot, uint4* out, cudaStream_t st);
void launch_state_hash(const uint4* rec, const u32* qword, const u64* node_state, u32 n_local, u32 stride, u32 first, u32 n_global, u32 R, u64* out, cudaStream_t st);
void launch_summary(const uint4* rec, const u32* qword, const u64* node_state, u32 n_local, u32 stride, u32 first, u32 R, const u32* subj_dev, u64* out /*[2 + 2*R + 2]*/, cudaStream_t st);
int tick_grid_size(u32 n_local, int ctas_per_sm);
int tick_ctas_per_sm_r1();
int tick_ctas_per_sm_r1s();
int tick_ctas_per_sm_rn();
void launch_compute_watch(const u32* row_ptr, const u32* col, const u32* subj_dev, u32 R, u32 first, u32 n_local, u16* watch, cudaStream_t st);
void launch_apply_watch(const u16* watch, u32 n_local, u8* busy, u8* hot_static, cudaStream_t st);

// User-event tick (uevent_kernel.cu; rules in uevent.cuh)
struct UeParams {
  u32 n_local, first, n_global, R, fanout, tick, seed_lo, seed_hi, limit;
  u32 ev_begin, ev_end;
  UeTable table;
  uint4* state;               // [n_local] 16-byte event records
  u32* inbox_rd;              // [n_local] arrived-event masks written during the previous tick (consumed and cleared)
  u32* inbox_wr;              // [n_local] masks being filled by this tick's sends
  u32* ltime;                 // [MAX_UEVENTS] Lamport time of each tracked event, stamped by its origin
  const u64* node_state;      // membership node words (up flag), pre-operation
  const u8* busy;             // bit 1: a host operation targets the node this tick
  const u32* row_ptr; const u32* col;
  const u32* ev_node; const u32* ev_op; const u32* ev_slot;
  u64* row;                   // this tick's trace row (shared with the membership kernel)
  u64* totals;                // run totals: 0 messages, 1 edges, 2 delivered, 3 duplicates, 4 too_old
  u32* overflow;
  u32* sched;                 // scheduler words of the membership kernel (idle-tick skipping): this kernel reports its activity there
  Gate gate;                  // the user-event kernel is the first kernel of a tick when user events are on
  // sharded runs: a target outside [first, first + n_local) gets one window entry per event (kind 3) over NVLink
  u32 world, rank, shard_size, win_cap;
  u64* const* win_data;       // [world] peers' receive windows of this exchange parity
  u32* send_count;            // [world] entries written into each peer's window this tick (shared with the tick kernel)
};
void launch_uevent(const UeParams& p, bool trace, cudaStream_t st);
void launch_ue_init(uint4* state, u32 n_local, cudaStream_t st);
void launch_ue_extract(const uint4* state, u32 n_local, int what, u32 e, void* out, cudaStream_t st);
void launch_ue_summary(const uint4* state, u32 n_local, u32 first, u32 n_global, u32 R, u32 n_events, u64* out, cudaStream_t st);

// Byzantine injectors (byz_kernel.cu; model in byz.cuh)
struct ByzParams {
  u32 n_byz, first, R, stride, fanout, tick, seed_lo, seed_hi, delta;
  const u32* ids;             // [n_byz] byzantine node ids (ascending)
  const uint4* rec;           // end-of-tick records
  const u64* node_state;
  const u32* row_ptr; const u32* col;
  u32* inbox_wr;              // the planes this tick's membership kernel filled
  u8* hot_wr;
  u32* kinds_cur;
  u8* anomaly;                // [n_local] sender flags
  u64* totals;                // 0 injected entries, 1 injected (peer, subject) pairs
  // sharded runs: a peer in another shard gets a TRIPLE of window entries — serf entry and memberlist entry, both with
  // BYZ_FLAG set in the destination field, then an annotation (kind 3, slot 15) carrying the sender's global id + 1 —
  // and the receiving shard's drain kernel judges it against ITS record and raises the flag in the sender's shard.
  u32 n_local, world, rank, shard_size, win_cap;
  u64* const* win_data;
  u32* send_count;
  u32* overflow;
  const u32* gate;
};
constexpr u32 BYZ_FLAG = 1u << 25;          // in the 26-bit destination field of a window entry (shards hold < 2^25 nodes when injectors are on)
constexpr u32 BYZ_ANNOT_SLOT = 15;
void launch_byz(const ByzParams& p, cudaStream_t st);

enum { EXTRACT_STATUS = 0, EXTRACT_STATUS_LTIME = 1, EXTRACT_CLOCK = 2, EXTRACT_INC = 3, EXTRACT_ML = 4, EXTRACT_STATUS_LTIME32 = 5, EXTRACT_CLOCK32 = 6 };

}  // namespace sfs
