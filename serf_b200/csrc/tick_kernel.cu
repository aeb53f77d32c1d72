// tick_kernel.cu — the fused gossip tick for sm_100a.
//
// One launch = one gossip tick of every virtual node of this shard:
//   Phase R  receive: fold the reduced inbox of the previous tick into the node's views
//            (SerfDelegate::notify_message → handle_node_{join,leave}_intent, serf/delegate.rs:157-315,
//             serf/base.rs:1338-1373, 1442-1572; LamportClock::witness, types/clock.rs:155-172;
//             memberlist alive/suspect/dead merge [external]);
//   Phase E  host operations scheduled for this tick (Serf::join/leave/remove_failed_node, serf/api.rs);
//   Phase T  suspicion-timer expiry and the SWIM probe [external];
//   Phase S  gossip: pick `fanout` distinct peers with the counter RNG and reduce every queued
//            entry into their inbox with RED.MAX (SerfDelegate::broadcast_messages + the
//            TransmitLimitedQueue budget, serf/delegate.rs:317-384, serf/base.rs:179-190).
// Sends of tick t land in inbox parity t&1 and are consumed by Phase R of tick t+1, so a launch
// never reads what it writes: bulk-synchronous, order-independent, bit-reproducible.
//
// Memory behaviour (HBM-bound integer work, no tensor cores): one thread per node; a node's 32-byte record is one
// 256-bit load (LDG.E.256 = one DRAM sector, a warp covers 1 KB contiguous) and, if changed, one 256-bit store; node
// word, busy byte, inbox words and row offsets are coalesced streams with an evict_first / no-L1-allocate policy; the
// four neighbour gathers stay inside the node's own 64-byte CSR row; the sends are 32-bit RED.MAX to random peers with
// an evict_last policy — the inbox planes are the only randomly addressed data and are sized to stay L2-resident.
// Tiles (256 nodes) nobody delivered to and that hold no pending work are skipped outright in sparse ticks.
// The multi-GPU variant stages cross-shard entries in shared memory and stores them into the peer GPU's window over NVLink.
#include "tick_kernel.cuh"
#include "byz.cuh"

namespace sfs {

namespace {

constexpr int BLOCK = 256;
constexpr int MB_R1 = 4;                    // resident CTAs per SM of the single-slot kernels (64 registers per thread)
constexpr int MB_R1S = MB_R1;               // … of the sharded single-slot kernel (its send path needs more registers: A/B in profiles/r2_notes.md)
constexpr int MB_RN = 2;                    // resident CTAs per SM of the multi-slot kernels (128 registers per thread: at 3 CTAs / 80 registers the
                                            // view loop spills, and local-memory traffic goes through the LSU the kernel is bound by: −7 % per run, profiles/r2_notes.md)
constexpr u32 TILE_SHIFT = 8;              // one tile = one CTA pass = 256 nodes
constexpr u32 MAX_TILES_PER_CTA = 1024;
static_assert((1u << TILE_SHIFT) == BLOCK, "tile = block");

// ---- cache-policy plumbing -------------------------------------------------------------------
// The only randomly addressed data of a tick are the inbox planes the sends reduce into (RED.MAX,
// 4 B at a random node).  They are kept L2-resident with an evict_last policy; everything that is
// streamed exactly once per tick (records, node state, the inbox parity being consumed) goes
// through evict_first / no-L1-allocate so it does not push the inbox out of the 126 MB L2.
struct Words { u32 w[8]; };   // one 32-byte record

#ifndef SERFSIM_EMU
__device__ __forceinline__ u64 policy_evict_first() { u64 p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ u64 policy_evict_last() { u64 p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }

__device__ __forceinline__ Words ld_rec256(const uint4* ptr, u64 pol) {   // one 256-bit load = one DRAM sector
  Words r;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
               : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
               : "l"(ptr), "l"(pol));
  return r;
}
__device__ __forceinline__ void st_rec256(uint4* ptr, const Words& r, u64 pol) {
  asm volatile("st.global.L2::cache_hint.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8}, %9;"
               :: "l"(ptr), "r"(r.w[0]), "r"(r.w[1]), "r"(r.w[2]), "r"(r.w[3]), "r"(r.w[4]), "r"(r.w[5]), "r"(r.w[6]), "r"(r.w[7]), "l"(pol) : "memory");
}
__device__ __forceinline__ u64 ld_u64_stream(const u64* ptr, u64 pol) {
  u64 v; asm volatile("ld.global.L1::no_allocate.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(ptr), "l"(pol)); return v;
}
__device__ __forceinline__ u32 ld_u32_stream(const u32* ptr, u64 pol) {
  u32 v; asm volatile("ld.global.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(ptr), "l"(pol)); return v;
}
__device__ __forceinline__ void st_u32_stream(u32* ptr, u32 v, u64 pol) {
  asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" :: "l"(ptr), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_u64_stream(u64* ptr, u64 v, u64 pol) {
  asm volatile("st.global.L2::cache_hint.u64 [%0], %1, %2;" :: "l"(ptr), "l"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void red_max_resident(u32* ptr, u32 v, u64 pol) {   // RED.MAX, result unused, line kept in L2
  asm volatile("red.relaxed.gpu.global.max.L2::cache_hint.u32 [%0], %1, %2;" :: "l"(ptr), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_release_sys(u32* ptr, u32 v) { asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(ptr), "r"(v) : "memory"); }
__device__ __forceinline__ u32 ld_acquire_sys(const u32* ptr) { u32 f; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(f) : "l"(ptr) : "memory"); return f; }
#else   // SERFSIM_EMU: the same accessors as plain C++ (tests/emu compiles this file for the host; cache hints have no meaning there)
inline u64 policy_evict_first() { return 0; }
inline u64 policy_evict_last() { return 0; }
// byte counters of the host build (probes 8..14): what the accessors of one run ISSUE, by class — an accounting aid for
// layout experiments (tools/emu_traffic.py), not a DRAM model
inline Words ld_rec256(const uint4* ptr, u64) { emu::probes[8] += 32; Words r; const u32* q = reinterpret_cast<const u32*>(ptr); for (int i = 0; i < 8; ++i) r.w[i] = q[i]; return r; }
inline void st_rec256(uint4* ptr, const Words& r, u64) { emu::probes[9] += 32; u32* q = reinterpret_cast<u32*>(ptr); for (int i = 0; i < 8; ++i) q[i] = r.w[i]; }
inline u64 ld_u64_stream(const u64* ptr, u64) { emu::probes[10] += 8; return *ptr; }
inline u32 ld_u32_stream(const u32* ptr, u64) { emu::probes[11] += 4; return *ptr; }
inline void st_u32_stream(u32* ptr, u32 v, u64) { emu::probes[12] += 4; *ptr = v; }
inline void st_u64_stream(u64* ptr, u64 v, u64) { emu::probes[13] += 8; *ptr = v; }
inline void red_max_resident(u32* ptr, u32 v, u64) { emu::probes[14] += 4; if (v > *ptr) *ptr = v; }
inline void st_release_sys(u32* ptr, u32 v) { __atomic_store_n(ptr, v, __ATOMIC_RELEASE); }     // peers are other threads of the test process
inline u32 ld_acquire_sys(const u32* ptr) {                 // polled in a loop by the drain kernel: be polite to the peer threads, and never hang a test run
  static thread_local const u32* last = nullptr;
  static thread_local unsigned long spins = 0;
  if (ptr != last) { last = ptr; spins = 0; }
  if (++spins > 64) emu::polite_wait(spins);
  return __atomic_load_n(ptr, __ATOMIC_ACQUIRE);
}
#endif

struct Counters {          // per-thread, reduced once per CTA; rare counters (events, suspects) go straight to the trace row
  u32 packets, edges, changed, pending, kL, kJ, kM, views;
  // single-view kernels (64 registers per thread, on the edge of spilling) keep six of them in three: a thread visits at most
  // MAX_TILES_PER_CTA = 1024 nodes, each adds at most MAX_FANOUT = 8 to a counter — 16 bits hold that
  u32 pe /* packets | edges << 16 */, cp /* changed | pending << 16 */, kLJ /* kL | kJ << 16 */;
  u64 hash;
};

__device__ __forceinline__ u32 warp_sum(u32 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ u64 warp_sum64(u64 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Deliver one entry to `dst` (global id): local → RED.MAX into this shard's inbox plane `plane`
// (= inbox_wr + (kind·R + slot)·n_local) and mark the destination tile hot for the next tick;
// cross-shard → append to the peer's receive window over NVLink.
// Cross-shard staging: every WARP owns one small buffer per destination shard in shared memory; entries are appended
// with a warp-aggregated shared-memory atomic and a buffer that holds at least 32 entries is copied into the peer's
// window by its own warp — 256+ contiguous bytes over NVLink, one global counter atomic per flush, no CTA barrier
// anywhere (a per-tile CTA-wide flush cost four barriers per tile and made every warp wait for the slowest one).
constexpr u32 MAX_WORLD = 8;
constexpr u32 XW_TOTAL = 392;              // staged entries per warp (3 KB), split evenly over the world-1 peers (world 8: 56 each)
constexpr u32 XW_FLUSH = 32;               // flush threshold: a full warp-wide store
struct XStage { u64 buf[(BLOCK / 32) * XW_TOTAL]; u32 cnt[BLOCK / 32][MAX_WORLD]; };
// (no integer division on the send path: the sharded kernel issues on every cycle it can — 2.4× the instructions of the unsharded one —
// and `x / runtime value` is ≈ 25 of them; capacity and reciprocal come with the parameters)
__device__ __forceinline__ u32 xcap(const TickParams& p) { return p.xcap; }
__device__ __forceinline__ u32 xseg(const TickParams& p, u32 shard) { return (shard - (shard > p.rank ? 1u : 0u)) * p.xcap; }
__device__ __forceinline__ u32 shard_of(const TickParams& p, u32 dst, u32& dloc) {
  u32 q = mulhi32(dst, p.shard_inv);           // floor(dst / shard_size) or one less
  u32 r = dst - q * p.shard_size;
  if (r >= p.shard_size) { ++q; r -= p.shard_size; }
  dloc = r;
  return q;
}

template <bool SHARDED>
__device__ __forceinline__ void deliver(const TickParams& p, XStage* xs, u32* plane, u32 dst, u32 kind, u32 s, u32 val1, u64 pol_last, bool mark) {
  const u32 dl = dst - p.first;
  if (!SHARDED || dl < p.n_local) {
    red_max_resident(plane + dl, val1, pol_last);
    if (mark) p.hot_wr[dl >> TILE_SHIFT] = 1;  // sparse ticks only: tell the next tick which tiles received something
  } else {
    u32 dloc;
    const u32 shard = shard_of(p, dst, dloc);
    const u64 e = ((u64)val1 << 32) | ((u64)(s + p.sv_wshift) << 28) | ((u64)kind << 26) | dloc;   // (a single-view launch numbers its view 0: the entry carries the real one)
    // append to the warp's own buffer for that shard: one shared-memory atomic per lane on the warp's counter (the hardware
    // serialises the lanes that hit the same counter; divergent callers of the same warp may interleave: keep it atomic)
    const u32 wid = threadIdx.x >> 5;
    const u32 pos = atomicAdd(&xs->cnt[wid][shard], 1u);
    if (pos < xcap(p)) {
      xs->buf[wid * XW_TOTAL + xseg(p, shard) + pos] = e;
    } else {                                   // buffer full: write this one straight through
      const u32 g = atomicAdd(p.send_count + shard, 1u);
      if (g < p.win_cap) p.win_data[shard][(size_t)p.rank * p.win_cap + g] = e;
      else *p.overflow = 2;
    }
  }
}

// Copy the warp's staged entries into the peers' windows (whole warp, convergent) in runs of whole 32-entry blocks (256+
// contiguous bytes over NVLink).  Space in a peer's window is reserved with an atomic on this rank's per-peer counter — one
// flush AHEAD: after its blocks have been written, the lane whose index is the peer's rank reserves as many entries as this
// flush used and keeps base and length in its own registers (`resv`, `rlen`); nothing reads them before the next flush, so the
// atomic's round trip on a counter the whole grid hammers is off the critical path (reserving at flush time cost 17 % of the
// sharded kernel's stall samples, profiles/r2g_hot_loop8_tick13.txt; so did a reservation issued inside the per-peer loop,
// whose next warp shuffle had to wait for it, profiles/r2h_hot_loop8_tick13.txt).  In saturated ticks the first reservation is
// made when the kernel starts.  A flush that needs more than it holds takes the rest synchronously.  Reserved entries that stay
// unwritten read as zeros at the receiver: the drain kernel skips zero entries and clears every entry it consumes, so a window
// is all zeros again before it is written next.  force = false: whole blocks only; force = true (end of the kernel): everything.
constexpr u32 XW_RESERVE_MAX = 128;        // entries reserved ahead per warp and peer, at most (bounds the padding, serfsim_create)
__device__ __forceinline__ bool flush_xwarp(const TickParams& p, XStage* xs, bool force, u32& resv, u32& rlen) {
  const u32 lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncwarp();
  bool wrote = false;
  u32 want = 0;                                // this lane's peer: entries to reserve for the next flush
  // peers whose buffer holds a whole block (anything, when forced): lane s looks at peer s, one vote, then only those are visited
  const u32 mine = lane < p.world ? xs->cnt[wid][lane] : 0u;
  u32 ready = __ballot_sync(0xffffffffu, lane != p.rank && (force ? mine != 0 : mine >= XW_FLUSH));
  while (ready) {
    const u32 sh = (u32)__ffs((int)ready) - 1u;
    ready &= ready - 1u;
    const u32 staged = __shfl_sync(0xffffffffu, mine, sh);
    if (staged > xcap(p)) wrote = true;        // the excess went straight through
    const u32 n = min(staged, xcap(p));
    const u32 m = force ? n : (n & ~(XW_FLUSH - 1u));          // entries to write now
    u64* src = xs->buf + wid * XW_TOTAL + xseg(p, sh);
    u64* dst = p.win_data[sh] + (size_t)p.rank * p.win_cap;
    const u32 base = __shfl_sync(0xffffffffu, resv, sh), avail = __shfl_sync(0xffffffffu, rlen, sh);
    const u32 take = min(m, avail);
    for (u32 i = lane; i < take; i += 32) {
      if (base + i < p.win_cap) dst[base + i] = src[i];
      else *p.overflow = 2;
    }
    if (m > take) {                            // not (enough) reserved ahead: take the rest now
      u32 b2 = 0;
      if (lane == sh) b2 = atomicAdd(p.send_count + sh, m - take);
      b2 = __shfl_sync(0xffffffffu, b2, sh);
      for (u32 i = lane; i < m - take; i += 32) {
        if (b2 + i < p.win_cap) dst[b2 + i] = src[take + i];
        else *p.overflow = 2;
      }
    }
    if (lane == sh) { resv += take; rlen -= take; want = min(m, XW_RESERVE_MAX); }
    wrote = true;
    const u32 rem = n - m;                     // < 32 entries stay staged: move them to the front
    u64 keep = 0;
    if (lane < rem) keep = src[m + lane];
    __syncwarp();
    if (lane < rem) src[lane] = keep;
    if (lane == 0) xs->cnt[wid][sh] = rem;
  }
  // reservations for the next flush: issued last, consumed by the shuffles of the NEXT call
  if (!force && want && rlen == 0) { resv = atomicAdd(p.send_count + lane, want); rlen = want; }
  __syncwarp();
  return wrote;
}

__device__ __forceinline__ void unpack_words(const Words& x, Rec& r) {
  r.st = x.w[0]; r.qjoin = x.w[1]; r.qleave = x.w[2]; r.inc = x.w[3]; r.deadline = x.w[4]; r.leave_tick = x.w[5];
  r.status = x.w[6] & 0xff; r.mlstate = (x.w[6] >> 8) & 3; r.qfrom = (x.w[6] >> 10) & 15; r.txj = (x.w[6] >> 16) & 0xff; r.txl = x.w[6] >> 24;
  r.txm = x.w[7] & 0xff; r.flags = (x.w[7] >> 8) & 0xff; r.mask = x.w[7] >> 16;
}
__device__ __forceinline__ void pack_words(const Rec& r, Words& x) {
  x.w[0] = r.st; x.w[1] = r.qjoin; x.w[2] = r.qleave; x.w[3] = r.inc; x.w[4] = r.deadline; x.w[5] = r.leave_tick;
  x.w[6] = r.status | (r.mlstate << 8) | (r.qfrom << 10) | (r.txj << 16) | (r.txl << 24);
  x.w[7] = r.txm | (r.flags << 8) | (r.mask << 16);
}
__device__ __forceinline__ void merge_q(Words& x, u32 q) { x.w[6] |= ((q & 0xffu) << 16) | (((q >> 8) & 0xffu) << 24); x.w[7] |= (q >> 16) & 0xffu; }
__device__ __forceinline__ u32 split_q(Words& x) {
  const u32 q = ((x.w[6] >> 16) & 0xffu) | ((x.w[6] >> 24) << 8) | ((x.w[7] & 0xffu) << 16);
  x.w[6] &= 0x0000ffffu; x.w[7] &= ~0xffu;
  return q;
}
__device__ __forceinline__ bool differs(const Words& a, const Words& b) {
  return ((a.w[0] ^ b.w[0]) | (a.w[1] ^ b.w[1]) | (a.w[2] ^ b.w[2]) | (a.w[3] ^ b.w[3]) | (a.w[4] ^ b.w[4]) | (a.w[5] ^ b.w[5]) | (a.w[6] ^ b.w[6]) | (a.w[7] ^ b.w[7])) != 0;
}

// Gossip peers of one node for one tick — memberlist kRandomNodes (k uniformly random distinct members
// other than ourselves): m = min(fanout, deg) distinct slots of the node's CSR row, sampled without
// replacement by rank from ONE Philox4x32-10 block (eight 16-bit draws: low half, then high half of words
// 0..3): draw k picks rank j = (h16_k·(deg−k)) >> 16 among the slots not chosen yet; slots pointing at the
// node itself are dropped; peers are used in draw order.  No rejection loop, no divergence, m gathers.
constexpr u32 NO_TARGET = 0xffffffffu;
__device__ __forceinline__ u32 draw16(const u32 (&w)[4], int i) { const u32 x = w[(i >> 1) & 3]; return (i & 1) ? (x >> 16) : (x & 0xffffu); }
// pick_issue draws the slots and requests the neighbour ids (cand[]: loads in flight), pick_finish drops self slots and packs the targets.
#define SFS_LD_COL(ptr, pol) __ldg(ptr)     // read-only path WITH L1 allocation: the four picks of a node fall into its two CSR sectors, later picks hit L1 (an evict_first / no-allocate gather was 6 % slower in plateau ticks)
template <int FMAX>
__device__ __forceinline__ void pick_issue(const TickParams& p, u32 v, u32 row0, u32 deg, u64 pol_first, u32 (&cand)[FMAX]) {
  const u32 m = min(p.fanout, deg);
  u32 w[4];
  philox4x32_10(p.tick, v, 0, DOMAIN_GOSSIP, p.seed_lo, p.seed_hi, w);
  u32 srt[FMAX];                                           // chosen slots so far, ascending; unused entries = NO_TARGET (sort last)
#pragma unroll
  for (int k = 0; k < FMAX; ++k) srt[k] = NO_TARGET;
#pragma unroll
  for (int k = 0; k < FMAX; ++k) {
    u32 j = (draw16(w, k) * (deg - min((u32)k, deg))) >> 16;
#pragma unroll
    for (int i = 0; i < k; ++i) j += (j >= srt[i]) ? 1u : 0u;         // rank → slot: skip the slots already taken
    const bool use = (u32)k < m;
    const u32 e = row0 + (use ? j : 0u);
    cand[k] = use ? SFS_LD_COL(p.col + e, pol_first) : v;
    // insert j into the ascending list (only if used): bubble it down from position k
    u32 x = use ? j : NO_TARGET;
#pragma unroll
    for (int i = 0; i < k; ++i) { const u32 lo = min(srt[i], x), hi = max(srt[i], x); srt[i] = lo; x = hi; }
    srt[k] = x;
  }
}
template <int FMAX>
__device__ __forceinline__ u32 pick_finish(u32 v, const u32 (&cand)[FMAX], u32 (&tg)[FMAX]) {
  u32 nt = 0;
#pragma unroll
  for (int k = 0; k < FMAX; ++k) tg[k] = NO_TARGET;
#pragma unroll
  for (int k = 0; k < FMAX; ++k) {
    if (cand[k] != v) {                                    // self slots (and the unused tail) are dropped
#pragma unroll
      for (int j2 = 0; j2 <= k; ++j2) tg[j2] = ((u32)j2 == nt) ? cand[k] : tg[j2];
      ++nt;
    }
  }
  return nt;
}

// What decides whether a node has anything to do this tick: its busy byte and the inbox words of the previous tick
// (slot 0 kept; per slot one "has mail" bit), plus — multi-slot runs — one "has queued transmits" bit per slot from the
// queue words.  13 bytes per node instead of 45 (single slot).
// busy byte: bit 0 awake (queued transmits / probe duty), bit 1 host operation this tick, bit 2 watcher (static),
// bit 3 some view of the node runs a suspicion timer (it sleeps until its tile comes due, tick_kernel.cuh).
// nd: the node's own earliest suspicion deadline (node_due), read only in tiles that have come due
struct Pre { u32 busy, mL, mJ, mM, any, qw, mailmask, qmask, keep, nd; };   // mL, mJ, mM, qw: the words of view `keep` (0 in single-slot runs)
template <bool R1>
__device__ __forceinline__ Pre prefetch_node(const TickParams& p, u32 vl, bool kL, bool kJ, bool kM, u64 pol_first, bool due, u32 keep = 0) {
  // R1: the kernel visits exactly one view, the one its planes start with (single-slot runs; single-view ticks of multi-slot runs, whose
  // parameter block points at the active view — the distance between the planes of two kinds is p.R views either way)
  const u32 nl = p.stride, R = p.R, s_hi = R1 ? 1u : R;
  Pre x;
  x.busy = p.busy[vl];
  x.nd = (!R1 && due) ? p.node_due[vl] : NO_DEADLINE;    // single-view kernels (64 registers) read it where it is needed instead: one register less across the tile loop
  x.keep = R1 ? 0u : keep;
  x.mL = x.mJ = x.mM = x.qw = 0; x.any = 0; x.mailmask = 0; x.qmask = 0;
  for (u32 s2 = 0; s2 < s_hi; ++s2) {
    const u32 l = kL ? ld_u32_stream(p.inbox_rd + (size_t)(KIND_LEAVE * R + s2) * nl + vl, pol_first) : 0u;
    const u32 j = kJ ? ld_u32_stream(p.inbox_rd + (size_t)(KIND_JOIN * R + s2) * nl + vl, pol_first) : 0u;
    const u32 m = kM ? ld_u32_stream(p.inbox_rd + (size_t)(KIND_ML * R + s2) * nl + vl, pol_first) : 0u;
    const u32 q = p.qword[(size_t)s2 * nl + vl];        // queue word (transmit budgets)
    SFS_COUNT(6, 4);
    if (R1 || s2 == x.keep) { x.mL = l; x.mJ = j; x.mM = m; x.qw = q; }
    x.any |= l | j | m;
    x.mailmask |= ((l | j | m) ? 1u : 0u) << s2;
    x.qmask |= (q ? 1u : 0u) << s2;
  }
  return x;
}
// Has the node anything to do this tick?  (due: its tile's earliest suspicion deadline has been reached — then a node that runs timers
// looks at its OWN earliest deadline: only if that has been reached too does it visit its views; otherwise it hands the deadline back
// to the timer wheel, sleeping_deadline(), without touching a record.)
__device__ __forceinline__ bool node_active(const TickParams& p, const Pre& x, bool due) {
  return (x.busy & 7u) != 0 || x.any != 0 || p.reap_now != 0 || (due && (x.busy & 8u) && x.nd <= p.tick);
}

// Multi-slot runs, saturated ticks: what a node needs beyond its `Pre` words, requested ONE TILE AHEAD together with them — the node
// word, the neighbour ids of its gossip peers (uniform out-degree: the row offset is arithmetic, the draw needs only tick and id) and the
// record of the view it will most probably visit first (`keep`: the first view this thread visited in its previous tile; in a
// dissemination wave nearly every node has the same views active).  The multi-slot kernel holds 16 warps per SM (128 registers per
// thread): without this every tile pays three dependent round trips (Pre → node word + record → neighbour ids) with too few warps to
// hide them.  A guess that turns out wrong costs one unused 32-byte load; results never depend on it.
template <int FMAX>
struct Ahead { u64 ns; Words rec; u32 cand[FMAX]; u32 valid; };

__device__ __forceinline__ u32 sleeping_deadline(const Pre& x, bool due) { return (due && (x.busy & 8u)) ? x.nd : NO_DEADLINE; }

// ---- cold paths of a node's tick, kept out of line: host operations, the reaper round and the SWIM probe run for a handful of
// nodes per tick (or for all of them once in a long while); inlined, their temporaries (a second Philox block, the operation
// scan) raise the register demand of the path every node takes and make it spill.  They are called on COPIES of the view and
// the node's scalars: a variable whose address is passed to a call lives in local memory for its whole lifetime, and the
// hot path's record must stay in registers (measured: 4.6 extra L2 sectors per node and +25 % per plateau tick otherwise).
#ifdef SERFSIM_EMU
#define SFS_COLD __attribute__((noinline))
#else
#define SFS_COLD __noinline__
#endif
// Phase E — what the API call does at its origin (SURVEY Appendix A.8): Serf::join / leave / remove_failed_node[_prune], crash, restart.
__device__ SFS_COLD void cold_host_op(Rec& r, u32& clock, u32& sstate, u32 op, bool op_here, bool self, bool up_r, u32 limit) {
  if (op == OP_REJOIN && self && !up_r) {
    r.inc += 1; r.mlstate = ML_ALIVE; r.qfrom = 0; r.txm = limit; r.deadline = 0; r.mask = 0;
    sstate = SS_ALIVE;
    node_join(r);
  }
  if (((op == OP_JOIN && up_r) || (op == OP_REJOIN && !up_r)) && self) {     // serf/api.rs:339-342 → serf/base.rs:381-397
    const u32 T = clock; witness(clock, T);
    join_intent(r, T, limit);
    r.qjoin = T; r.txj = limit;
  }
  if (op == OP_LEAVE && up_r && self && sstate == SS_ALIVE) {                // serf/api.rs:422-449
    sstate = SS_LEAVING;
    const u32 T = clock; clock += 1;
    bool rf = false;
    leave_intent(r, T, false, true, sstate, rf, limit);
    r.qleave = T; r.txl = limit; r.flags &= ~FLAG_QPRUNE;
  }
  if ((op == OP_FORCE_LEAVE || op == OP_FORCE_LEAVE_PRUNE) && up_r && op_here) {   // serf/base.rs:454-480 (remove_failed_node[_prune], serf/api.rs:500-515)
    const u32 T = clock; witness(clock, T);
    const bool prune = op == OP_FORCE_LEAVE_PRUNE;
    bool rf = false;
    leave_intent(r, T, prune, self, sstate, rf, limit);
    r.qleave = T; r.txl = limit; r.flags = (r.flags & ~FLAG_QPRUNE) | (prune ? FLAG_QPRUNE : 0u);   // queued whatever the handler said
    if (rf) { const u32 T2 = clock; witness(clock, T2); join_intent(r, T2, limit); r.qjoin = T2; r.txj = limit; }
  }
}
// Which host operation targets node v this tick (the mark kernel set bit 1 of its busy byte)?
__device__ SFS_COLD u32 cold_find_op(const TickParams& p, u32 v, u32& op_slot) {
  atomicAdd((unsigned long long*)(p.row + 5), 1ull);
  for (u32 e = p.ev_begin; e < p.ev_end; ++e)
    if (p.ev_node[e] == v) { op_slot = p.ev_slot[e]; return p.ev_op[e]; }
  return 0;
}
// Reaper round (serf/base.rs:483-610): Left / Failed members past their timeouts are erased, stale buffered intents dropped.
__device__ SFS_COLD void cold_reap(Rec& r, u32 t, u32 tombstone, u32 reconnect, u32 intent) {
  const u32 age = r.leave_tick ? (t + 1 - r.leave_tick) : 0;
  if ((r.flags & 1) && r.leave_tick && ((r.status == ST_LEFT && age > tombstone) || (r.status == ST_FAILED && age > reconnect))) {
    r.flags &= ~1u; r.status = TY_NONE; r.st = 0; r.leave_tick = 0;           // erase_node! :499-519
  } else if (!(r.flags & 1) && r.status != TY_NONE && r.leave_tick && age > intent) {
    r.status = TY_NONE; r.st = 0; r.leave_tick = 0;                           // reap_intents :1817-1822
  }
}
// SWIM probe target of a watcher's round: a uniformly random neighbour (memberlist walks a shuffled list).
__device__ SFS_COLD u32 cold_probe_target(const TickParams& p, u32 v, u32 row0, u32 deg) {
  u32 w[4];
  philox4x32_10(p.tick, v, 0, DOMAIN_PROBE, p.seed_lo, p.seed_hi, w);
  return __ldg(p.col + row0 + (((w[0] & 0xffffu) * deg) >> 16));
}
// The probe found the subject down: suspect it (or confirm with this node's bucket).
__device__ SFS_COLD void cold_probe_hit(const TickParams& p, Rec& r, u32 v) {
  if (r.mlstate == ML_ALIVE || r.mlstate == ML_SUSPECT) {
    if (r.mlstate == ML_ALIVE) atomicAdd((unsigned long long*)(p.row + 6), 1ull);
    ml_suspect(r, r.inc, from_bucket(v), p.tick, false, p.rules);
  }
}
// Refutation of a leave intent about ourselves: serf/base.rs:1470-1480 → broadcast_join(clock.time()), :381-397
__device__ SFS_COLD void cold_refute(Rec& r, u32& clock, u32 limit) {
  const u32 T = clock; witness(clock, T);
  join_intent(r, T, limit);
  r.qjoin = T; r.txj = limit;
}
// Is a watcher's own failed probe still a confirmation (its bucket not in the confirmer set, the set not full)?
__device__ SFS_COLD bool cold_can_confirm(u32 k, u32 mask, u32 v) {
  return (u32)__popc(mask) - 1u < k && !(mask & (1u << from_bucket(v)));
}

// Returns true when the node stays awake (queued transmits, probe duty): that keeps its tile hot for the next tick.
// A view whose only business is a running suspicion timer does not: its deadline goes to `mind` (the caller registers the
// minimum in tile_due) and the view sleeps until its tile comes due.  `due`: this tile's earliest deadline has been reached —
// every node of it that carries a timer (busy bit 3) visits all its views.
template <bool TRACE, int FMAX, bool SHARDED, bool R1>
__device__ __forceinline__ bool process_node(const TickParams& p, XStage* xs, const u32 vl, const Pre& pre, const bool kL, const bool kJ, const bool kM, const bool mark, const bool saturated,
                                             const bool due, const u64 pol_first, const u64 pol_last, Counters& c, u32& mind, int& dsusp, const Ahead<FMAX>& ah, u32& first_view, const u32 sv_views = 0xffffffffu) {
  const u32 v = p.first + vl;
  const u32 t = p.tick;
  const u32 limit = p.rules.limit;
  const u32 nl = p.stride;               // plane stride (n_local rounded up to a whole tile)
  const u32 R = p.R;                     // R1: one view is visited, the first of the planes as this launch sees them (they keep the distance of p.R views between kinds)

  // ---- loads.  Saturated ticks (the previous tick delivered to at least half of the nodes): everything a node
  // needs is requested up front, independent loads in flight together.  Otherwise most nodes are idle: read only
  // the busy byte and the inbox words, and fetch the 8-byte node word and the 32-byte record just for the nodes
  // that have something to do.  Multi-slot runs fetch the records of the views that have something to do. ----
  const bool upfront = R1 && (saturated || TRACE);
  u64 ns = 0;
  u32 row0 = 0, row1 = 0;
  Words cur;
  auto load_node = [&]() {
    ns = ld_u64_stream(p.node_state + vl, pol_first);
    if (p.udeg) { row0 = vl * p.udeg; row1 = row0 + p.udeg; }     // uniform out-degree: the row offsets are arithmetic
    else { row0 = __ldg(p.row_ptr + vl); row1 = __ldg(p.row_ptr + vl + 1); }
  };
  auto load_rec0 = [&]() {
    cur = ld_rec256(p.rec + 2 * (size_t)vl, pol_first);
    merge_q(cur, pre.qw);                                  // the record image everything below works on is record | budgets
  };
  if (upfront) { load_node(); load_rec0(); }
  const u32 busy = pre.busy;
  u32 mL = pre.mL, mJ = pre.mJ, mM = pre.mM;

  // ---- idle exit: nothing received (any slot), nothing queued, no host operation, no probe duty, no timer due ----
  u32 nd = pre.nd;                                       // the node's own earliest deadline: matters in due tiles, for nodes that run timers
  if (R1 && due && (busy & 8u)) nd = p.node_due[vl];
  const u32 sleeping = (due && (busy & 8u)) ? nd : NO_DEADLINE;
  const bool timers_due = sleeping <= p.tick;
  if (!TRACE && !((busy & 7u) != 0 || pre.any != 0 || p.reap_now != 0 || timers_due)) { mind = min(mind, sleeping); if (due && (busy & 8u)) SFS_PROBE(20); return false; }
  // (the watcher mask — subjects this node can probe, it has them as neighbours — is re-read where a watcher needs it: a handful of nodes)
#define SFS_WMASK() ((busy & 4u) ? ((u32)p.watch[vl] >> p.sv_wshift) : 0u)   /* sv_wshift: the view a single-view launch works on (0 in every other launch) */
  const bool ahead = !R1 && ah.valid;                  // node word, peers' ids and the record of view pre.keep were requested a tile ago
  if (ahead) { ns = ah.ns; row0 = vl * p.udeg; row1 = row0 + p.udeg; }
  else if (!upfront) { load_node(); if (R1) load_rec0(); }

  u32 clock = (u32)ns;
  const bool up_r = (ns & NS_UP) != 0;
  u32 sstate = (u32)(ns >> 40) & 3;
  const u32 deg = row1 - row0;

  // host operation for this node (at most one per tick; the mark kernel set bit 1 of the busy byte)
  u32 op = 0, op_slot = 0;
  if (busy & 2) { u32 slot_tmp = 0; op = cold_find_op(p, v, slot_tmp); op_slot = slot_tmp; }
  bool up_s = up_r;
  if (op == OP_FAIL) up_s = false;
  if (op == OP_REJOIN) up_s = true;

  // SWIM probe target of this round (only matters while some tracked subject is down)
  bool have_probe = false;
  u32 ptarget = 0;
  if (up_s && (busy & 4u) && p.probe_every && p.down_mask && ((t + v) % p.probe_every) == 0 && deg) {
    ptarget = cold_probe_target(p, v, row0, deg);
    have_probe = true;
  }

  u32 tg[FMAX];
  u32 nt = 0;
  bool have_targets = false;
  u32 max_tx = 0;
  bool awake = false, has_timer = false, dl_moved = false;
  // (`mind`, NO_DEADLINE on entry: the earliest running suspicion deadline among the views visited)

  // Views to visit: all of them when the node as a whole has business (trace, reaper round, host operation, timers due);
  // otherwise those with mail, queued transmits or probe duty (a watcher's view of a subject that is down).
  const u32 all_views = (R >= 32u) ? 0xffffffffu : ((1u << R) - 1u);
  const bool visit_all = R1 || TRACE || p.reap_now || (busy & 2u) || timers_due || !p.sleep_on;
  u32 todo = visit_all ? all_views : ((pre.mailmask | pre.qmask | (p.probe_every ? (SFS_WMASK() & p.down_mask) : 0u)) & all_views);
  if (!R1) SFS_COUNT(5, R - (u32)__popc(todo));             // views left asleep by a visited node

  // multi-slot runs: the record and inbox words of the next view to visit are requested once the current one is stored
  // (requesting them while it is processed keeps 12 more registers live and was measured slower)
  Words nxt = {};
  u32 nL = 0, nJ = 0, nM = 0, nq = 0;
  auto load_view = [&](u32 s2, Words& w, u32& q, u32& iL, u32& iJ, u32& iM) {
    const size_t idn = (size_t)s2 * nl + vl;
    w = ld_rec256(p.rec + 2 * idn, pol_first);
    if (s2 == pre.keep) { q = pre.qw; iL = pre.mL; iJ = pre.mJ; iM = pre.mM; return; }
    q = p.qword[idn];
    SFS_COUNT(6, 4);
    iL = kL ? ld_u32_stream(p.inbox_rd + (size_t)(KIND_LEAVE * R + s2) * nl + vl, pol_first) : 0;
    iJ = kJ ? ld_u32_stream(p.inbox_rd + (size_t)(KIND_JOIN * R + s2) * nl + vl, pol_first) : 0;
    iM = kM ? ld_u32_stream(p.inbox_rd + (size_t)(KIND_ML * R + s2) * nl + vl, pol_first) : 0;
  };
  u32 s = R;
  if (R1) { s = 0; todo = 0; }
  else if (todo) {
    s = (u32)__ffs((int)todo) - 1u; todo &= todo - 1u;
    u32 q0;
    if (ahead && s == pre.keep) { cur = ah.rec; q0 = pre.qw; mL = pre.mL; mJ = pre.mJ; mM = pre.mM; SFS_PROBE(18); }
    else load_view(s, cur, q0, mL, mJ, mM);
    merge_q(cur, q0);
    first_view = s;
  }
#pragma unroll 1
  while (s < R) {
    const size_t idx = (size_t)s * nl + vl;
    u32 s_next = R;
    if (!R1 && todo) { s_next = (u32)__ffs((int)todo) - 1u; todo &= todo - 1u; }
    if (mL) st_u32_stream(p.inbox_rd + (size_t)(KIND_LEAVE * R + s) * nl + vl, 0u, pol_first);   // consume: clear for reuse in two ticks
    if (mJ) st_u32_stream(p.inbox_rd + (size_t)(KIND_JOIN * R + s) * nl + vl, 0u, pol_first);
    if (mM) st_u32_stream(p.inbox_rd + (size_t)(KIND_ML * R + s) * nl + vl, 0u, pol_first);
    const Words orig = cur;
    Rec r;
    unpack_words(cur, r);
    const bool self = (p.subj[s] == v);
    const bool susp_before = up_r && r.mlstate == ML_SUSPECT;
    if (!R1 && p.sv_mode == SV_CHECK && !((sv_views >> s) & 1u) && up_r &&
        ((mL | mJ | mM) || (r.txl | r.txj | r.txm) || r.mlstate == ML_SUSPECT)) *p.overflow = 4;     // SERFSIM_SV=2: the set of views with business was not a superset

    // ---------------- Phase R ----------------
    if (up_r && (mL | mJ | mM)) {
      if (mM) {
        const u32 key = mM - 1, inc = key >> 6, kind = (key >> 4) & 3, fromb = key & 15;
        if (kind == ML_ALIVE) ml_alive(r, inc, self, limit);
        else if (kind == ML_SUSPECT) ml_suspect(r, inc, fromb, t, self, p.rules);
        else ml_dead(r, inc, kind == ML_LEFT, t, self, limit);
      }
      bool refute = false;
      if (mL) { const u32 key = mL - 1, lt = key >> 1; witness(clock, lt); leave_intent(r, lt, !(key & 1u), self, sstate, refute, limit); }
      if (mJ) { const u32 lt = mJ - 1; witness(clock, lt); join_intent(r, lt, limit); }
      if (refute) { Rec tr = r; u32 ck = clock; cold_refute(tr, ck, limit); r = tr; clock = ck; }
      if (!(r.flags & 1) && r.status != TY_NONE && (r.status != (orig.w[6] & 0xff) || r.st != orig.w[0])) r.leave_tick = t + 1;   // NodeIntent.wall_time (types/member.rs:32)
      Words mid;
      pack_words(r, mid);
      if (R1) c.cp += differs(mid, orig) ? 1u : 0u; else c.changed += differs(mid, orig) ? 1 : 0;
    }
    // ---------------- Phase E ----------------
    if (op) { Rec tr = r; u32 ck = clock, ss = sstate; cold_host_op(tr, ck, ss, op, op_slot == s, self, up_r, limit); r = tr; clock = ck; sstate = ss; }
    if (op && !(r.flags & 1) && r.status != TY_NONE && r.leave_tick == 0) r.leave_tick = t + 1;
    if (up_s) {
      // ---------------- Phase T: reaper (serf/base.rs:483-610), suspicion timer, probe ----------------
      if (p.reap_now) { Rec tr = r; cold_reap(tr, t, p.tombstone_ticks, p.reconnect_ticks, p.intent_ticks); r = tr; }
      if (r.mlstate == ML_SUSPECT && r.deadline != 0 && t >= r.deadline) ml_dead(r, r.inc, false, t, false, limit);
      if (have_probe && !self && ptarget == p.subj[s] && ((p.down_mask >> s) & 1)) { Rec tr = r; cold_probe_hit(p, tr, v); r = tr; }
      // ---------------- Phase S ----------------
      const u32 mx = max(r.txl, max(r.txj, r.txm));
      if (mx) {
        if (!have_targets) {
          if (ahead) nt = pick_finish<FMAX>(v, ah.cand, tg);
          else {
            u32 cand[FMAX];
            pick_issue<FMAX>(p, v, row0, deg, pol_first, cand);
            nt = pick_finish<FMAX>(v, cand, tg);
          }
          have_targets = true;
        }
        u32* const planeL = p.inbox_wr + (size_t)(KIND_LEAVE * R + s) * nl;
        u32* const planeJ = p.inbox_wr + (size_t)(KIND_JOIN * R + s) * nl;
        u32* const planeM = p.inbox_wr + (size_t)(KIND_ML * R + s) * nl;
        const u32 vL = leave_key(r.qleave, (r.flags & FLAG_QPRUNE) != 0) + 1, vJ = r.qjoin + 1, vM = ml_key(r) + 1;
        const u32 sL = min(r.txl, nt), sJ = min(r.txj, nt), sM = min(r.txm, nt);     // entry e goes to targets 0 .. min(tx_e, nt)-1
#pragma unroll
        for (int k = 0; k < FMAX; ++k) {
          if ((u32)k < sL) deliver<SHARDED>(p, xs, planeL, tg[k], KIND_LEAVE, s, vL, pol_last, mark);
          if ((u32)k < sJ) deliver<SHARDED>(p, xs, planeJ, tg[k], KIND_JOIN, s, vJ, pol_last, mark);
          if ((u32)k < sM) deliver<SHARDED>(p, xs, planeM, tg[k], KIND_ML, s, vM, pol_last, mark);
        }
        if (R1) { c.kLJ += sL | (sJ << 16); c.kM += sM; c.pe += min(mx, nt) << 16; }
        else { c.kL += sL; c.kJ += sJ; c.kM += sM; c.edges += min(mx, nt); }
        max_tx = max(max_tx, mx);
        r.txl -= sL; r.txj -= sJ; r.txm -= sM;
      }
      // Serf::leave: our own leave intent is out → memberlist.leave() → dead{node == from}  (serf/api.rs:451-476)
      if (self && sstate == SS_LEAVING && r.txl == 0 && r.mlstate == ML_ALIVE) {
        r.mlstate = ML_LEFT; r.qfrom = 0; r.txm = limit; sstate = SS_LEFT;
      }
      // The trace's `pending` counts the views with queued transmits, a running suspicion timer, or a watcher that has not
      // noticed yet.  Suspect views are counted by the persistent counter (they sleep), the others here.  A watcher's view of
      // a down subject stays awake while it is Alive or Suspect: its own failed probe may still start or confirm the suspicion.
      const bool queued = (r.txl | r.txj | r.txm) != 0;
      if (!R1 && (queued || mx)) c.views |= 1u << s;                  // the view sent mail or keeps a queue: it has business in the next tick (single-view ticks)
      const bool watching = (busy & 4u) && p.probe_every && ((p.down_mask >> s) & 1) && !self && ((SFS_WMASK() >> s) & 1);
      const bool suspect = r.mlstate == ML_SUSPECT;
      { const u32 pnd = (!suspect && (queued || (watching && r.mlstate == ML_ALIVE))) ? 1u : 0u; if (R1) c.cp += pnd << 16; else c.pending += pnd; }
      // (its own failed probe is a confirmation only while its bucket is not in the confirmer set and the set is not full)
      awake |= queued || (watching && (r.mlstate == ML_ALIVE || (suspect && cold_can_confirm(p.rules.k, r.mask, v))));
      if (suspect && r.deadline != 0) { has_timer = true; mind = min(mind, r.deadline); dl_moved |= r.deadline != orig.w[4]; }
    }
    dsusp += ((up_s && r.mlstate == ML_SUSPECT) ? 1 : 0) - (susp_before ? 1 : 0);
    pack_words(r, cur);
    {
      Words o2 = orig, c2 = cur;                           // storage image: record without budgets, budgets in the queue word
      const u32 q_old = split_q(o2), q_new = split_q(c2);
      if (differs(c2, o2)) st_rec256(p.rec + 2 * idx, c2, pol_first);
      if (q_new != q_old) { p.qword[idx] = q_new; SFS_COUNT(7, 4); }
    }
    if (TRACE) c.hash += rec_hash((u64)s * p.n_global + v, make_uint4(cur.w[0], cur.w[1], cur.w[2], cur.w[3]), make_uint4(cur.w[4], cur.w[5], cur.w[6], cur.w[7]));
    if (r.inc >= INC_LIMIT) *p.overflow = 1;
    if (!R1) {
      if (s_next < R) load_view(s_next, nxt, nq, nL, nJ, nM);
      cur = nxt; merge_q(cur, nq); mL = nL; mJ = nJ; mM = nM;
    }
    s = s_next;
  }
  const u64 ns2 = (u64)clock | (up_s ? NS_UP : 0) | ((u64)sstate << 40);
  if (ns2 != ns) st_u64_stream(p.node_state + vl, ns2, pol_first);
  if (TRACE) c.hash += node_hash((u64)R * p.n_global + v, ns2);
  if (clock >= LTIME_LIMIT) *p.overflow = 1;
  if (R1) c.pe += min(nt, max_tx); else c.packets += min(nt, max_tx);
  // busy byte: the op bit is consumed, the watcher bit is static; the timer bit is exact after a visit of every view and
  // sticky otherwise (a view that was not visited may run a timer: it is found when its tile comes due)
  const u32 busy2 = (awake ? 1u : 0u) | (busy & 4u) | ((has_timer || (!visit_all && (busy & 8u))) ? 8u : 0u);
  if (busy2 != busy) p.busy[vl] = (u8)busy2;
  // node_due: a lower bound of the node's earliest running deadline, exact after a visit of every view.  A view's deadline only moves
  // while the view is visited, so views that were not visited are still covered by the word as it stands.
  if (has_timer) {
    if (visit_all || !(busy & 8u)) p.node_due[vl] = mind;
    else if (dl_moved) atomicMin(p.node_due + vl, mind);
  }
  if (!visit_all) mind = min(mind, sleeping);   // its tile's entry was reset: timers of the views not visited go back with the node's word
  // The scheduler must know whether anybody stays awake.  A node that sent a packet this tick shows in the row's message count;
  // the others (a watcher on probe duty, a queue that has no peer to go to, a transmit queued after the send phase) are rare.
  if (awake && min(nt, max_tx) == 0) atomicAdd(p.sched + SCHED_AWAKE, 1u);
  return awake;
}

__device__ __forceinline__ u32 warp_min(u32 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// After a warp has processed its nodes of one tile: register the earliest running suspicion deadline in the timer wheel and add
// the warp's net change of Suspect views to the CTA's shared counter (both rare outside suspicion waves: one vote each).
__device__ __forceinline__ void note_timers(const TickParams& p, u32 tile, u32 mind, int dsusp, int* dsusp_s) {
  if (!__any_sync(0xffffffffu, (mind != NO_DEADLINE) | (dsusp != 0))) return;      // one vote on the common path
  const u32 wm = warp_min(mind);
  const u32 ws = warp_sum((u32)dsusp);                     // two's complement: the sum of the lanes' signed changes
  if ((threadIdx.x & 31) == 0) {
    if (wm != NO_DEADLINE) atomicMin(p.tile_due + tile, wm);
    if (ws) atomicAdd(dsusp_s, (int)ws);
  }
}

// A skipped tick (tick_is_idle): nothing can happen, so the only trace it leaves is its row — nothing delivered, nothing
// changed, `pending` = the sleeping Suspect views, and (trace runs) the state hash of the previous tick.
template <bool TRACE>
__device__ __forceinline__ void write_idle_row(const TickParams& p) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    SFS_PROBE(3);                                          // skipped ticks
    p.row[4] += *reinterpret_cast<const u64*>(p.sched + SCHED_SUSPECTS);
    if (TRACE && p.tick > 0) p.row[7] = *(p.row - 8 + 7);
  }
}

// Scan of the CTA's tile flags.  hot_s[i]: bit 0 = process the tile, bit 1 = its earliest suspicion deadline has been reached
// (the entry is reset here, by the tile's owner, before any of its nodes runs: the timers that are still running re-register).
__device__ __forceinline__ void scan_tiles(const TickParams& p, u8* hot_s, u32 tile0, u32 ntile, bool all_hot) {
  for (u32 i = threadIdx.x; i < ntile; i += BLOCK) {
    const u8 f = p.hot_rd[tile0 + i];
    if (f) p.hot_rd[tile0 + i] = 0;                      // consumed; this parity is written again two ticks from now
    const bool due = p.tile_due[tile0 + i] <= p.tick;
    if (due) { p.tile_due[tile0 + i] = NO_DEADLINE; SFS_PROBE(4); }     // tiles woken by the timer wheel
    hot_s[i] = (u8)(((f || all_hot || due || p.hot_static[tile0 + i]) ? 1u : 0u) | (due ? 2u : 0u));
  }
}

// What publish_kernel does, for one peer per calling thread (threads 0 .. world-1 of one CTA): entry count, this rank's trace row and
// scheduler verdict into the peer's control block, then the release flag of this exchange.
__device__ __forceinline__ void publish_to_peer(u32 r, u32 world, u32 rank, u32 xpar, u32 stamp, u32 loopback, u32* const* peer_ctrl, u32* send_count,
                                                const volatile u64* row, const volatile u32* sched) {
  if (r >= world || r == rank) return;
  const u32 me = loopback ? r : rank;                       // the slot this rank owns in the peer's control block
  u32* ctrl = peer_ctrl[r] + xpar * 16;
  ctrl[me] = send_count[r];
  u64* sums = reinterpret_cast<u64*>(reinterpret_cast<unsigned char*>(peer_ctrl[r]) + CTRL_SUMS_OFF) + ((size_t)xpar * 8 + me) * CTRL_FIELDS;
#pragma unroll
  for (int i = 0; i < 8; ++i) sums[i] = row[i];              // this rank's counters of the tick: every rank sums them on the device
  sums[8] = sched[SCHED_LOCAL_QUIET]; sums[9] = sched[SCHED_LOCAL_UNTIL]; sums[10] = sched[SCHED_VIEWS_NEW];
  __threadfence_system();
  st_release_sys(ctrl + 8 + me, stamp);
  send_count[r] = 0;
}

// End of a tick: block reduction of the counters (warp shuffles, then shared memory) → one atomic per counter per CTA; the
// LAST CTA to finish (ticket) completes the row and decides how long the cluster can sleep.
// trace row: 0 packets, 1 edge_updates, 2 messages, 3 changed, 4 pending, (5 events, 6 suspects: direct), 7 hash
template <bool TRACE, bool PACKED>
__device__ __forceinline__ void finish_tick(const TickParams& p, const Counters& c, u64 (*red)[BLOCK / 32], int dsusp_cta) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __shared__ u32 last_s, due_min_s[BLOCK / 32];
  const u32 kL = PACKED ? (c.kLJ & 0xffffu) : c.kL, kJ = PACKED ? (c.kLJ >> 16) : c.kJ;
  const u64 vals[8] = {PACKED ? (c.pe & 0xffffu) : c.packets, PACKED ? (c.pe >> 16) : c.edges, (u64)kL + kJ + c.kM, PACKED ? (c.cp & 0xffffu) : c.changed,
                       PACKED ? (c.cp >> 16) : c.pending, kL, kJ, c.kM};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const u32 s = warp_sum((u32)vals[i]);
    if (lane == 0) red[i][wid] = s;
  }
  u64 hs = 0;
  if (TRACE) hs = warp_sum64(c.hash);
  __syncthreads();                                         // dsusp_cta is complete
  if (threadIdx.x == 0 && dsusp_cta) atomicAdd(reinterpret_cast<unsigned long long*>(p.sched + SCHED_SUSPECTS), (unsigned long long)(long long)dsusp_cta);
  if (threadIdx.x < 8) {
    u64 s = 0;
#pragma unroll
    for (int w = 0; w < BLOCK / 32; ++w) s += red[threadIdx.x][w];
    if (s) {
      if (threadIdx.x < 5) atomicAdd((unsigned long long*)(p.row + threadIdx.x), (unsigned long long)s);
      else atomicAdd(p.kinds_cur + (threadIdx.x - 5), (u32)min(s, (u64)0xffffffffu));
    }
  }
  if (TRACE && lane == 0 && hs) atomicAdd((unsigned long long*)(p.row + 7), (unsigned long long)hs);
  { const u32 vw = __reduce_or_sync(0xffffffffu, c.views); if (lane == 0 && vw) atomicOr(p.sched + SCHED_VIEWS_NEXT, vw); }
  // ---- ticket: every CTA's counters are in the row before the last one reads it ----
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last_s = (atomicAdd(p.sched + SCHED_TICKET, 1u) == gridDim.x - 1) ? 1u : 0u;
  __syncthreads();
  if (!last_s) return;
  __threadfence();
  volatile u32* sched = p.sched;
  volatile u64* row = p.row;
  const u64 suspects = *reinterpret_cast<volatile u64*>(p.sched + SCHED_SUSPECTS);
  // Can the next ticks do anything?  Not if nothing was sent (no mail), nobody stays awake (no queued transmit, no probe duty),
  // the user-event kernel reported nothing queued or sent (with injectors sleep_on is off): then the cluster sleeps until the earliest
  // suspicion deadline or the next anti-entropy / reaper round (host operations are checked at launch).  Sharded runs: this is
  // the rank's verdict; it travels with the row and the drain kernel combines the ranks' (all quiet, earliest deadline).
  // (decided by ONE thread and broadcast: the words it reads are cleared below by thread 0, and a warp that evaluated them later than
  // thread 0 cleared them would take the other side of a branch that contains a barrier)
  __shared__ u32 quiet_s;
  if (threadIdx.x == 0) quiet_s = (p.sleep_on && row[1] == 0 && row[2] == 0 && sched[SCHED_AWAKE] == 0 && sched[SCHED_UE_ACTIVITY] == 0) ? 1u : 0u;
  __syncthreads();
  const bool quiet = quiet_s != 0;
  u32 until = p.tick + 1;
  if (quiet) {                                             // uniform over the CTA
    u32 m = NO_DEADLINE;
    for (u32 i = threadIdx.x; i < p.n_tiles; i += BLOCK) m = min(m, __ldcg(p.tile_due + i));
    m = warp_min(m);
    if (lane == 0) due_min_s[wid] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 0; w < BLOCK / 32; ++w) m = min(m, due_min_s[w]);
      // a round runs in tick u when (u + 1) % period == 0; the first such u > tick:
      if (p.pp_every) m = min(m, ((p.tick + 1) / p.pp_every + 1) * p.pp_every - 1);
      if (p.reap_every) m = min(m, ((p.tick + 1) / p.reap_every + 1) * p.reap_every - 1);
      until = max(m, p.tick + 1);
    }
  }
  if (threadIdx.x == 0) {
    row[4] = row[4] + suspects;                            // pending = awake views counted above + sleeping Suspect views
    if (p.world == 1) {
      sched[SCHED_IDLE_UNTIL] = until;
      if (p.host_idle_until) *p.host_idle_until = until;
    } else {
      sched[SCHED_LOCAL_QUIET] = quiet ? 1u : 0u; sched[SCHED_LOCAL_UNTIL] = until;
    }
    const u32 awake_n = sched[SCHED_AWAKE];
    sched[SCHED_AWAKE] = 0; sched[SCHED_UE_ACTIVITY] = 0; sched[SCHED_TICKET] = 0;
    // (the single-view kernel keeps no per-thread set: its view has business again iff anything was sent or anybody stays awake)
    const u32 sv_next = (p.sv_mode == SV_SINGLE && (row[2] != 0 || awake_n != 0)) ? (1u << p.sv_slot) : 0u;
    // this tick's set stays readable (OLD) for the kernel of this tick that is launched after this one and must return
    const u32 sv_base = p.tick >= sched[SCHED_VIEWS_FROM] ? sched[SCHED_VIEWS_NEW] : sched[SCHED_VIEWS_OLD];   // what this kernel's CTAs read when they started (nobody else writes these words)
    sched[SCHED_VIEWS_OLD] = sv_base; sched[SCHED_VIEWS_NEW] = sched[SCHED_VIEWS_NEXT] | sv_next; sched[SCHED_VIEWS_FROM] = p.tick + 1; sched[SCHED_VIEWS_NEXT] = 0;   // the views with business in the next tick (kernels that follow in this tick — anti-entropy, drain — add to it)
  }
  if (p.world > 1 && p.fuse_publish) {
    // every CTA fenced its peer-window stores (system scope) before it took its ticket; this one saw all tickets
    __syncthreads();
    __threadfence();
    publish_to_peer(threadIdx.x, p.world, p.rank, p.xpar, p.stamp, p.loopback, p.peer_ctrl, p.send_count, row, sched);
  }
}

// Persistent CTAs; each owns a contiguous range of 256-node tiles.  A tile is processed only if it is
// "hot": somebody delivered into it during the previous tick, it holds a node that stays awake (queued transmits,
// probe duty), a host operation targets it, or a suspicion timer of one of its nodes has come due — otherwise not a
// single byte of it is touched.
template <bool TRACE, int FMAX, bool SHARDED, bool R1, int MB>
__global__ void __launch_bounds__(BLOCK, MB) tick_kernel(const __grid_constant__ TickParams p) {
  __shared__ u8 hot_s[MAX_TILES_PER_CTA];
  __shared__ u64 red[8][BLOCK / 32];
  __shared__ int dsusp_s;                                  // net change of the number of Suspect views at up nodes, this CTA
  __shared__ __align__(16) unsigned char xs_mem[SHARDED ? sizeof(XStage) : 16];
  XStage* xs = reinterpret_cast<XStage*>(xs_mem);
  if (gate_closed(p.gate, blockIdx.x == 0 && threadIdx.x == 0)) return;   // the run is over (uniform over the grid): this tick does not exist
  if (tick_is_idle(p.sched, p.tick, p.ev_begin, p.ev_end)) { if (p.sv_mode != SV_SINGLE) write_idle_row<TRACE>(p); return; }   // nothing can happen in this tick (uniform)
  // Single-view ticks of multi-slot runs (tick_kernel.cuh, SV_*): the general kernel and the single-view kernel are both launched; the
  // set of views that can have business in this tick — known on the device since the end of the previous tick — decides which one runs.
  u32 sv_views = 0xffffffffu;
  if (p.sv_mode != SV_OFF) {
    // (the kernel of this tick that ran before this one, if any, has already published the NEXT tick's set: SCHED_VIEWS_FROM says since when it holds)
    const u32 sv_base = p.tick >= p.sched[SCHED_VIEWS_FROM] ? p.sched[SCHED_VIEWS_NEW] : p.sched[SCHED_VIEWS_OLD];
    const u32 views = (sv_base | p.views_host) & ((1u << p.sv_R) - 1u);
    const bool single = views == (1u << p.sv_slot);        // exactly the one view the single-view launch was set up for
    if (p.sv_mode == SV_SINGLE) { if (!single) return; SFS_PROBE(21); }
    else if (p.sv_mode == SV_GENERAL && single) return;
    if (p.sv_mode == SV_CHECK && single) sv_views = views;   // checked only where the single-view kernel would have run
  }
  if (threadIdx.x == 0) dsusp_s = 0;                       // ordered before its first use by the barrier after the tile scan
  Counters c = {};
  const bool kL = p.kinds_prev[KIND_LEAVE] != 0, kJ = p.kinds_prev[KIND_JOIN] != 0, kM = p.kinds_prev[KIND_ML] != 0;
  const u64 pol_first = policy_evict_first(), pol_last = policy_evict_last();
  const int lane = threadIdx.x & 31;
  if (SHARDED && threadIdx.x < (BLOCK / 32) * MAX_WORLD) xs->cnt[threadIdx.x / MAX_WORLD][threadIdx.x % MAX_WORLD] = 0;
  bool wrote_remote = false;
  u32 resv = 0, rlen = 0;                                  // lane s: the entries this warp holds reserved in peer s's window (flush_xwarp)

  // Dense / sparse ticks.  While the gossip front is wide (the previous tick sent at least one message per
  // two tiles) every tile will be hot anyway: senders skip the per-message tile marking and the next tick
  // simply processes everything (kinds[3] of this tick's row records the decision).  In sparse ticks each
  // delivery marks its destination tile, and tiles nobody touched are not read at all.
  const u32 prev_msgs = p.kinds_prev[KIND_LEAVE] + p.kinds_prev[KIND_JOIN] + p.kinds_prev[KIND_ML];
  const bool dense_now = prev_msgs >= (p.n_tiles >> 1) + 1;      // what this tick's sends will look like
  const bool all_hot = p.force_all || p.kinds_prev[3] != 0;      // the previous tick was dense (or skipping is off)
  const bool mark = !dense_now;
  const bool saturated = prev_msgs >= (p.n_local >> 1);          // most nodes have mail: request record + node word up front
  if (dense_now && blockIdx.x == 0 && threadIdx.x == 0) p.kinds_cur[3] = 1;

  const u32 tile0 = blockIdx.x * p.tiles_per_cta;
  const u32 ntile = tile0 < p.n_tiles ? min(p.tiles_per_cta, p.n_tiles - tile0) : 0;
  if (SHARDED && saturated && ntile && (u32)lane < p.world && (u32)lane != p.rank) { resv = atomicAdd(p.send_count + lane, XW_FLUSH); rlen = XW_FLUSH; }   // every warp will send to every peer
  scan_tiles(p, hot_s, tile0, ntile, all_hot);
  __syncthreads();
  // Unsaturated ticks (ramp-up and tail of a dissemination: a few per cent of the nodes have anything to do, spread
  // one or two per warp): a tile-by-tile walk pays one chain of dependent round trips (state → row → peers) per TILE
  // for a handful of active lanes.  Instead the CTA scans GROUP hot tiles at once — the 13 "anything to do?" bytes
  // of every node, all loads in flight together — compacts the active nodes into a shared-memory list and runs the
  // node logic on dense blocks of 256 list entries: one chain per 256 ACTIVE nodes.  Nodes are independent within a
  // tick and every cross-node effect is a commutative reduction, so the visiting order changes nothing.
  constexpr u32 GROUP = SHARDED ? 4 : 8;
  __shared__ uint4 act_s[GROUP * BLOCK];                   // x: tile-in-group << 8 | lane, busy << 16, any << 24; y, z, w: inbox words
  __shared__ u32 act_n;
  __shared__ u8 pend_s[GROUP];
  __shared__ u16 gt_s[GROUP];
  const bool compact = !TRACE && !saturated && !p.reap_now && p.compact;
  if (compact) {
    u32 i = 0;
    while (i < ntile) {
      u32 ng = 0;                                          // the next GROUP hot tiles of this CTA (every thread walks the same flags)
      while (i < ntile && ng < GROUP) { if (hot_s[i]) { if (threadIdx.x == 0) gt_s[ng] = (u16)i; ++ng; } ++i; }
      if (!ng) break;
      if (threadIdx.x == 0) act_n = 0;
      if (threadIdx.x < GROUP) pend_s[threadIdx.x] = 0;
      __syncthreads();
      Pre pr[GROUP];
#pragma unroll
      for (u32 g = 0; g < GROUP; ++g) {
        pr[g] = Pre{};
        if (g < ng) {
          const u32 vn = ((tile0 + gt_s[g]) << TILE_SHIFT) + threadIdx.x;
          if (vn < p.n_local) pr[g] = prefetch_node<R1>(p, vn, kL, kJ, kM, pol_first, false);   // (a node's own deadline is read below, in due tiles only: eight more live registers otherwise)
        }
      }
#pragma unroll
      for (u32 g = 0; g < GROUP; ++g) {
        const bool due_g = g < ng && (hot_s[gt_s[g]] & 2u) != 0;
        Pre prg = pr[g];
        if (due_g && (prg.busy & 8u)) prg.nd = p.node_due[((tile0 + gt_s[g]) << TILE_SHIFT) + threadIdx.x];
        const bool act = g < ng && node_active(p, prg, due_g);   // lanes past n_local hold an empty Pre
        if (due_g) {                                         // (warp-uniform) nodes whose own timers run later hand their deadline back to the wheel
          const u32 wm = warp_min(act ? NO_DEADLINE : sleeping_deadline(prg, true));
          if (lane == 0 && wm != NO_DEADLINE) atomicMin(p.tile_due + tile0 + gt_s[g], wm);
          if (!act && (prg.busy & 8u)) SFS_PROBE(20);
        }
        const u32 bal = __ballot_sync(0xffffffffu, act);
        if (bal) {
          u32 base = 0;
          if (lane == 0) base = atomicAdd(&act_n, (u32)__popc(bal));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (act) act_s[base + (u32)__popc(bal & ((1u << lane) - 1u))] =
              make_uint4((g << 8) | threadIdx.x | (pr[g].busy << 16) | ((pr[g].any ? 1u : 0u) << 24), pr[g].mL, pr[g].mJ, pr[g].mM);
        }
      }
      __syncthreads();
      const u32 na = act_n;
      if (threadIdx.x == 0) { SFS_PROBE(0); if (ng > 1) SFS_PROBE(1); if (na > BLOCK) SFS_PROBE(2); }   // groups, multi-tile groups, multi-pass groups
      for (u32 b0 = 0; b0 < na; b0 += BLOCK) {
        const u32 e = b0 + threadIdx.x;
        if (e < na) {
          const uint4 a = act_s[e];
          const u32 g = (a.x >> 8) & 0xffu;
          const u32 ti = gt_s[g];
          const u32 vl = ((tile0 + ti) << TILE_SHIFT) + (a.x & 0xffu);
          Pre pre;
          if (R1) {
            pre.busy = (a.x >> 16) & 0xffu; pre.any = (a.x >> 24) & 1u; pre.mL = a.y; pre.mJ = a.z; pre.mM = a.w; pre.keep = 0;
            pre.nd = NO_DEADLINE;
            pre.qw = p.qword[vl];                             // not carried through the list: issued here, in flight with the state loads
            pre.mailmask = pre.any ? 1u : 0u; pre.qmask = pre.qw ? 1u : 0u;
            SFS_COUNT(6, 4);
          } else {
            pre = prefetch_node<R1>(p, vl, kL, kJ, kM, pol_first, (hot_s[ti] & 2u) != 0);   // per-view masks are not carried through the list: the few active nodes read them again
          }
          u32 mind = NO_DEADLINE, fv_unused = 0;
          int dsusp = 0;
          const bool pend = process_node<TRACE, FMAX, SHARDED, R1>(p, xs, vl, pre, kL, kJ, kM, mark, false, (hot_s[ti] & 2u) != 0, pol_first, pol_last, c, mind, dsusp, Ahead<FMAX>{}, fv_unused, sv_views);
          if (mark && pend) pend_s[g] = 1;
          if (mind != NO_DEADLINE) atomicMin(p.tile_due + tile0 + ti, mind);      // the list mixes tiles: per-lane registration (few active nodes)
          if (dsusp) atomicAdd(&dsusp_s, dsusp);
        }
        if (SHARDED) wrote_remote |= flush_xwarp(p, xs, false, resv, rlen);
      }
      __syncthreads();
      if (mark && threadIdx.x < ng && pend_s[threadIdx.x]) p.hot_wr[tile0 + gt_s[threadIdx.x]] = 1;
      __syncthreads();                                     // gt_s / act_s are rewritten by the next group
    }
  } else {
  // Walk the hot tiles of this CTA.  The 13 "is there anything to do" bytes of the NEXT hot tile (busy byte, inbox
  // words) are requested before the current tile is processed, so an idle tile costs no exposed round trip.
  // Multi-slot runs, saturated ticks: node word, peers' ids and the probable first view's record travel one tile ahead too (Ahead).
  const bool ahead_on = !R1 && p.udeg != 0 && (p.ahead == 2u || (p.ahead == 1u && saturated));
  u32 first_view = 0;                                      // the first view this thread visited in its last tile
  auto prefetch_tile = [&](u32 ti) -> Pre {
    const u32 vn = ((tile0 + ti) << TILE_SHIFT) + threadIdx.x;
    return vn < p.n_local ? prefetch_node<R1>(p, vn, kL, kJ, kM, pol_first, (hot_s[ti] & 2u) != 0, first_view) : Pre{};
  };
  auto ahead_tile = [&](u32 ti, u32 keep) -> Ahead<FMAX> {
    Ahead<FMAX> a = {};
    const u32 vn = ((tile0 + ti) << TILE_SHIFT) + threadIdx.x;
    if (!R1 && ahead_on && vn < p.n_local) {
      a.ns = ld_u64_stream(p.node_state + vn, pol_first);
      a.rec = ld_rec256(p.rec + 2 * ((size_t)keep * p.stride + vn), pol_first);
      pick_issue<FMAX>(p, p.first + vn, vn * p.udeg, p.udeg, pol_first, a.cand);
      a.valid = 1;
      SFS_PROBE(19);
    }
    return a;
  };
  u32 i = 0;
  while (i < ntile && !hot_s[i]) ++i;
  Pre pre_next = {};
  Ahead<FMAX> ah_next = {};
  if (i < ntile) { pre_next = prefetch_tile(i); ah_next = ahead_tile(i, pre_next.keep); }
  while (i < ntile) {
    const Pre pre = pre_next;
    const Ahead<FMAX> ah = ah_next;
    u32 j = i + 1;
    while (j < ntile && !hot_s[j]) ++j;
    if (j < ntile) { pre_next = prefetch_tile(j); ah_next = ahead_tile(j, pre_next.keep); }
    const u32 vl = ((tile0 + i) << TILE_SHIFT) + threadIdx.x;
    bool pend = false;
    u32 mind = NO_DEADLINE;
    int dsusp = 0;
    if (vl < p.n_local) pend = process_node<TRACE, FMAX, SHARDED, R1>(p, xs, vl, pre, kL, kJ, kM, mark, saturated, (hot_s[i] & 2u) != 0, pol_first, pol_last, c, mind, dsusp, ah, first_view, sv_views);
    if (mark && __any_sync(0xffffffffu, pend) && lane == 0) p.hot_wr[tile0 + i] = 1;
    note_timers(p, tile0 + i, mind, dsusp, &dsusp_s);
    if (SHARDED) wrote_remote |= flush_xwarp(p, xs, false, resv, rlen);
    i = j;
  }
  }
  if (SHARDED) {
    wrote_remote |= flush_xwarp(p, xs, true, resv, rlen);
    if (wrote_remote) __threadfence_system();            // peer-window stores are performed before the publish kernel raises the flags
  }
  __syncthreads();
  finish_tick<TRACE, R1>(p, c, red, dsusp_s);
}

// Anti-entropy round — memberlist push-pull + SerfDelegate::merge_remote_state (serf/delegate.rs:386-554; "next"
// row 1 of SURVEY §8f).  Runs after the tick kernel every push_pull_interval ticks on a SNAPSHOT of the end-of-tick
// state: each up node pulls the state of one random neighbour and merges it — clock witness(ltime−1), per subject
// the memberlist state (alive → aliveNode, suspect/dead → suspectNode{from = self}, left → deadNode{from = node}),
// then serf's view (Left member → leave intent at status_ltime+1, any other → join intent at status_ltime) with the
// handlers' results discarded: nothing is re-queued (delegate.rs:495-523).  A node writes only its own records.
template <bool TRACE>
__global__ void __launch_bounds__(BLOCK) pushpull_kernel(const __grid_constant__ TickParams p, const uint4* __restrict__ snap_rec, const u64* __restrict__ snap_node) {
  if (p.gate.ctl && p.gate.ctl[0]) return;
  // a round can queue transmits and start timers after the tick kernel has decided how long the cluster may sleep: take the decision back
  if (blockIdx.x == 0 && threadIdx.x == 0) { p.sched[SCHED_IDLE_UNTIL] = 0; if (p.host_idle_until) *p.host_idle_until = 0; }
  long long d_changed = 0, d_pending = 0, d_susp = 0;
  u64 d_hash = 0;
  u32 d_views = 0;                                         // views left with queued transmits: they have business in the next tick
  for (u32 vl = blockIdx.x * BLOCK + threadIdx.x; vl < p.n_local; vl += gridDim.x * BLOCK) {
    const u32 v = p.first + vl;
    const u64 ns = snap_node[vl];
    if (!(ns & NS_UP)) continue;
    const u32 row0 = p.row_ptr[vl], deg = p.row_ptr[vl + 1] - row0;
    if (!deg) continue;
    u32 w[4];
    philox4x32_10(p.tick, v, 0, DOMAIN_PUSHPULL, p.seed_lo, p.seed_hi, w);
    const u32 u = p.col[row0 + (((w[0] & 0xffffu) * deg) >> 16)];
    if (u == v) continue;
    // the partner may live in another shard: its rank's snapshot is read through the peer mapping (the host
    // separates "every rank has taken its snapshot" and "every rank has finished reading" with barriers)
    u32 ul = u - p.first;
    const u64* part_node = snap_node;
    const uint4* part_rec = snap_rec;
    u32 part_stride = p.stride;
    if (p.world > 1) {
      const u32 shard = u / p.shard_size;
      ul = u - shard * p.shard_size;
      part_node = p.snap_node_peer[shard]; part_rec = p.snap_rec_peer[shard];
      const u32 cnt = min(p.shard_size, p.n_global - shard * p.shard_size);
      part_stride = ((cnt + BLOCK - 1) / BLOCK) * BLOCK;
    }
    const u64 nu = part_node[ul];
    if (!(nu & NS_UP)) continue;
    u32 clock = (u32)ns;
    const u32 sstate = (u32)(ns >> 40) & 3;
    const u32 cu = (u32)nu;
    if (cu > 0) witness(clock, cu - 1);
    bool awake = false, has_timer = false;
    u32 mind = NO_DEADLINE;
    const u32 wmask = p.watch[vl];
    for (u32 s = 0; s < p.R; ++s) {
      const size_t iv = (size_t)s * p.stride + vl, iu = (size_t)s * part_stride + ul;
      const uint4 a0 = p.rec[2 * iv];
      uint4 b0 = p.rec[2 * iv + 1];
      const u32 q0 = p.qword[iv];
      merge_queue_word(b0, q0);
      Rec r, q;
      unpack(a0, b0, r);
      unpack(part_rec[2 * iu], part_rec[2 * iu + 1], q);
      const bool self = (p.subj[s] == v);
      const bool was = (r.txl | r.txj | r.txm) || r.mlstate == ML_SUSPECT || (p.probe_every && ((p.down_mask >> s) & 1) && !self && ((wmask >> s) & 1) && r.mlstate == ML_ALIVE);
      if (q.flags & 1) {
        if (q.mlstate == ML_ALIVE) ml_alive(r, q.inc, self, p.rules.limit);
        else if (q.mlstate == ML_LEFT) ml_dead(r, q.inc, true, p.tick, self, p.rules.limit);
        else ml_suspect(r, q.inc, from_bucket(v), p.tick, self, p.rules);
        bool refute = false;
        if (q.status == ST_LEFT) { witness(clock, q.st + 1); leave_intent(r, q.st + 1, false, self, sstate, refute, p.rules.limit, false); }
        else { witness(clock, q.st); join_intent(r, q.st, p.rules.limit, false); }
        if (refute) { const u32 T = clock; witness(clock, T); join_intent(r, T, p.rules.limit); r.qjoin = T; r.txj = p.rules.limit; }
        if (!(r.flags & 1) && r.status != TY_NONE && (r.status != (b0.z & 0xff) || r.st != a0.x)) r.leave_tick = p.tick + 1;
      }
      uint4 a1, b1;
      pack(r, a1, b1);
      const bool ch = (a1.x ^ a0.x) | (a1.y ^ a0.y) | (a1.z ^ a0.z) | (a1.w ^ a0.w) | (b1.x ^ b0.x) | (b1.y ^ b0.y) | (b1.z ^ b0.z) | (b1.w ^ b0.w);
      if (ch) {
        uint4 bs = b1;
        const u32 q1 = split_queue_word(bs);
        p.rec[2 * iv] = a1; p.rec[2 * iv + 1] = bs;
        if (q1 != q0) p.qword[iv] = q1;
      }
      if ((a1.y ^ a0.y) | (a1.z ^ a0.z) | (a1.w ^ a0.w) | (b1.x ^ b0.x) | (b1.y ^ b0.y) | (b1.z ^ b0.z) | (b1.w ^ b0.w)) d_changed++;   // status_time creep is not a change
      if (TRACE && ch) d_hash += rec_hash((u64)s * p.n_global + v, a1, b1) - rec_hash((u64)s * p.n_global + v, a0, b0);
      const bool watching = p.probe_every && ((p.down_mask >> s) & 1) && !self && ((wmask >> s) & 1);
      const bool now = (r.txl | r.txj | r.txm) || r.mlstate == ML_SUSPECT || (watching && r.mlstate == ML_ALIVE);
      d_pending += (now ? 1 : 0) - (was ? 1 : 0);
      d_susp += (r.mlstate == ML_SUSPECT ? 1 : 0) - (((b0.z >> 8) & 3u) == ML_SUSPECT ? 1 : 0);     // the node is up: counted views
      awake |= (r.txl | r.txj | r.txm) != 0 || (watching && (r.mlstate == ML_ALIVE ||
               (r.mlstate == ML_SUSPECT && (u32)__popc(r.mask) - 1u < p.rules.k && !(r.mask & (1u << from_bucket(v))))));
      if (r.mlstate == ML_SUSPECT && r.deadline != 0) { has_timer = true; mind = min(mind, r.deadline); }
      if (r.txl | r.txj | r.txm) d_views |= 1u << s;
      if (r.inc >= INC_LIMIT) *p.overflow = 1;
    }
    if (p.ue_table.n) {                                        // the partner's event clock and ring (a snapshot, like its records)
      const uint4 pw = (p.world > 1 ? p.ue_snap_peer[u / p.shard_size] : p.ue_snap)[ul];
      const uint4 w0 = p.ue_state[vl];
      UeRec er;
      ue_unpack(w0, er);
      UeCounts ec = {};
      ue_replay(er, pw.x, pw.y & 0xffu, p.ue_ltime, p.ue_table, p.rules.limit, ec);
      const uint4 w1 = ue_pack(er);
      if ((w1.x ^ w0.x) | (w1.y ^ w0.y) | (w1.z ^ w0.z) | (w1.w ^ w0.w)) p.ue_state[vl] = w1;
      d_changed += ec.delivered;
      if (ec.delivered) atomicAdd((unsigned long long*)(p.ue_totals + 2), (unsigned long long)ec.delivered);
      if (ec.duplicates) atomicAdd((unsigned long long*)(p.ue_totals + 3), (unsigned long long)ec.duplicates);
      if (ec.too_old) atomicAdd((unsigned long long*)(p.ue_totals + 4), (unsigned long long)ec.too_old);
      if (TRACE) d_hash += ue_hash((u64)(p.R + 1) * p.n_global + v, w1) - ue_hash((u64)(p.R + 1) * p.n_global + v, w0);
      if (er.clock >= LTIME_LIMIT) *p.overflow = 1;
    }
    const u64 ns2 = (ns & ~0xffffffffull) | clock;
    if (ns2 != ns) {
      p.node_state[vl] = ns2;
      if (TRACE) d_hash += node_hash((u64)p.R * p.n_global + v, ns2) - node_hash((u64)p.R * p.n_global + v, ns);
    }
    if (clock >= LTIME_LIMIT) *p.overflow = 1;
    // every view of the node was visited: its busy byte is exact (bit 0 awake, bit 2 watcher, bit 3 running timer)
    p.busy[vl] = (u8)((awake ? 1u : 0u) | (wmask ? 4u : 0u) | (has_timer ? 8u : 0u));
    if (awake) p.hot_wr[vl >> TILE_SHIFT] = 1;
    if (has_timer) { atomicMin(p.tile_due + (vl >> TILE_SHIFT), mind); p.node_due[vl] = mind; }
  }
  const u64 c = warp_sum64((u64)d_changed), q = warp_sum64((u64)d_pending), ds = warp_sum64((u64)d_susp), h = TRACE ? warp_sum64(d_hash) : 0;
  d_views = __reduce_or_sync(0xffffffffu, d_views);
  if ((threadIdx.x & 31) == 0) {
    if (d_views) atomicOr(p.sched + SCHED_VIEWS_NEW, d_views);
    if (c) atomicAdd((unsigned long long*)(p.row + 3), (unsigned long long)c);
    if (q) atomicAdd((unsigned long long*)(p.row + 4), (unsigned long long)q);
    if (ds) atomicAdd(reinterpret_cast<unsigned long long*>(p.sched + SCHED_SUSPECTS), (unsigned long long)ds);
    if (TRACE && h) atomicAdd((unsigned long long*)(p.row + 7), (unsigned long long)h);
  }
}

// After the tick kernel: publish, to every peer, how many entries this rank wrote into its window, then raise
// the peer's flag for this exchange (system-scope release).  One warp.
__global__ void publish_kernel(const __grid_constant__ PublishParams p) {
  if (p.gate && *p.gate) return;
  publish_to_peer(threadIdx.x, p.world, p.rank, p.xpar, p.stamp, p.loopback, p.peer_ctrl, p.send_count, p.row, p.sched);
}

// Fold the cross-shard windows into the inbox.  Waits (system-scope acquire) until every peer has raised
// this exchange's flag — the peers' publish kernels precede their own drains in stream order, so the wait
// cannot deadlock — then reduces the entries exactly like local deliveries.
__global__ void __launch_bounds__(BLOCK) drain_kernel(const __grid_constant__ DrainParams p) {
  if (p.gate && *p.gate) return;
  if (threadIdx.x < p.world && threadIdx.x != p.rank) {
    u32 f;
    do { f = ld_acquire_sys(p.ctrl + 8 + threadIdx.x); } while (f != p.stamp);
  }
  __syncthreads();
  // global trace row of this tick: my counters + the rows the peers published with their flags (acquired above)
  if (blockIdx.x == 0 && threadIdx.x < 8) {
    u64 s = p.my_row[threadIdx.x];
    for (u32 src = 0; src < p.world; ++src) if (src != p.rank) s += __ldcg(p.sums + (size_t)src * CTRL_FIELDS + threadIdx.x);
    p.grow[threadIdx.x] = s;
  }
  // The ranks' scheduler verdicts: the cluster sleeps iff every rank is quiet, until the earliest of their deadlines.  Every rank
  // computes the same value from the same published words and hands it to its HOST only (mapped memory): in sharded runs the
  // device never skips a launched tick — a skipped exchange would let a fast rank reuse a window parity its peer is still
  // draining — the hosts simply do not launch the ticks the cluster sleeps through (serfsim_run_until_converged), all alike.
  if (blockIdx.x == 0 && threadIdx.x == 0 && p.sched) {
    bool quiet = p.sleep_on && p.sched[SCHED_LOCAL_QUIET] != 0;
    u32 until = p.sched[SCHED_LOCAL_UNTIL];
    for (u32 src = 0; src < p.world; ++src) {
      if (src == p.rank) continue;
      quiet = quiet && __ldcg(p.sums + (size_t)src * CTRL_FIELDS + 8) != 0;
      until = min(until, (u32)__ldcg(p.sums + (size_t)src * CTRL_FIELDS + 9));
    }
    if (p.host_idle_until) *p.host_idle_until = quiet ? max(until, p.tick + 1) : p.tick + 1;
    u32 views = 0;                                        // views with business in the next tick: anywhere in the cluster (their mail crosses shards)
    for (u32 src = 0; src < p.world; ++src) if (src != p.rank) views |= (u32)__ldcg(p.sums + (size_t)src * CTRL_FIELDS + 10);
    if (views) atomicOr(p.sched_rw + SCHED_VIEWS_NEW, views);
  }
  // same dense / sparse decision as the tick kernel of this tick: in a dense tick the next tick processes every
  // tile anyway, so per-entry tile marking (millions of byte stores onto a few thousand flags) is skipped
  const u32 prev_msgs = p.kinds_prev[KIND_LEAVE] + p.kinds_prev[KIND_JOIN] + p.kinds_prev[KIND_ML];
  const bool mark = prev_msgs < (p.n_tiles >> 1) + 1;
  u32 seen = 0;                                 // kinds this thread folded (bit per kind)
  for (u32 src = 0; src < p.world; ++src) {
    if (src == p.rank) continue;
    const u32 n = min(p.ctrl[src], p.win_cap);
    u64* w = p.win_data + (size_t)src * p.win_cap;
    for (u32 i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) {
      const u64 e = __ldcg(w + i);
      if (e == 0) continue;                          // padding of a partly filled block (a real entry has value + 1 > 0 in its high word)
      if (!p.byz_on) w[i] = 0;                       // consumed: the window reads as zeros when it is written next (injector triples are
                                                     // read by a neighbouring thread too: those runs clear the windows in a kernel of their own)
      const u32 val1 = (u32)(e >> 32), s = (u32)(e >> 28) & 15, kind = (u32)(e >> 26) & 3;
      u32 dl = (u32)e & ((1u << 26) - 1);
      const bool byz = p.byz_on && (dl & BYZ_FLAG);
      if (byz) dl &= ~BYZ_FLAG;
      if (byz && kind == 3 && s == BYZ_ANNOT_SLOT) continue;           // third entry of a triple: read by the thread holding the first
      if (dl < p.n_local && s < p.R && kind < 3) {
        atomicMax(p.inbox_wr + ((size_t)(kind * p.R + s)) * p.stride + dl, val1);
        if (mark) p.hot_wr[dl >> TILE_SHIFT] = 1;
        seen |= 1u << kind;
        if (byz && kind < 2 && i + 2 < n) {                            // first entry of a triple: judge it against MY record, flag the sender in ITS shard
          const u64 e1 = __ldcg(w + i + 1), e2 = __ldcg(w + i + 2);
          const u32 src = (u32)(e2 >> 32) - 1u;
          ByzEntries be{};
          be.serf_lt = kind == KIND_LEAVE ? (val1 - 1u) >> 1 : val1 - 1u; be.ml_inc = ((u32)(e1 >> 32) - 1u) >> 6;
          if (p.node_state[dl] & NS_UP) {
            const size_t iv = (size_t)s * p.stride + dl;
            Rec q;
            unpack(p.rec[2 * iv], p.rec[2 * iv + 1], q);
            if (byz_anomalous(q, be, p.byz_delta)) { const u32 sh = src / p.shard_size; p.peer_anomaly[sh][src - sh * p.shard_size] = 1; }
          }
        }
      } else if (dl < p.n_local && kind == 3 && s < p.ue_n && val1) {   // user event s arrived: one bit, and the time its origin stamped
        atomicOr(p.ue_inbox_wr + dl, 1u << s);
        p.ue_ltime[s] = val1 - 1;                      // every copy carries the same value; this shard learns it no later than the event itself
      }
      else *p.overflow = 3;
    }
  }
  // received kinds count as "in flight" for the next tick's plane skipping; the received volume feeds its dense/sparse decision
  seen = __reduce_or_sync(0xffffffffu, seen);
  if ((threadIdx.x & 31) == 0 && seen) {
    for (u32 k = 0; k < 3; ++k) if ((seen >> k) & 1) atomicAdd(p.kinds_cur + k, 1u);
  }
}

// Rows of ticks the host did not launch because the cluster sleeps through them (serfsim_run_until_converged): what
// write_idle_row would have written.  rows = first of the n rows; the row before it belongs to the last executed / skipped tick.
__global__ void fill_idle_rows_kernel(u64* rows, u64* grow_rows, u32 n, const u32* sched, int trace) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rows[(size_t)i * 8 + 4] = *reinterpret_cast<const u64*>(sched + SCHED_SUSPECTS);
  if (trace) rows[(size_t)i * 8 + 7] = *(rows - 8 + 7);
  if (grow_rows) {                                         // sharded: the global rows repeat the global pending count / hash
    grow_rows[(size_t)i * 8 + 4] = *(grow_rows - 8 + 4);
    if (trace) grow_rows[(size_t)i * 8 + 7] = *(grow_rows - 8 + 7);
  }
}

// Injector runs: the drain kernel leaves its windows as they are (a triple is read by two threads); this clears what it consumed.
__global__ void __launch_bounds__(BLOCK) clear_windows_kernel(const __grid_constant__ DrainParams p) {
  if (p.gate && *p.gate) return;
  for (u32 src = 0; src < p.world; ++src) {
    if (src == p.rank) continue;
    const u32 n = min(p.ctrl[src], p.win_cap);
    u64* w = p.win_data + (size_t)src * p.win_cap;
    for (u32 i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) w[i] = 0;
  }
}

// watch[v]: bit s set iff subject s appears in node v's neighbour list — only such nodes can ever pick it as a probe
// target, so they alone evaluate the SWIM probe (and stay scheduled while it is down).
__global__ void compute_watch_kernel(const u32* __restrict__ row_ptr, const u32* __restrict__ col, const u32* __restrict__ subj, u32 R, u32 first, u32 n_local, u16* watch) {
  const u32 vl = blockIdx.x * blockDim.x + threadIdx.x;
  if (vl >= n_local) return;
  u32 m = 0;
  const u32 v = first + vl;
  for (u32 e = row_ptr[vl]; e < row_ptr[vl + 1]; ++e) {
    const u32 c = col[e];
    if (c == v) continue;
    for (u32 s = 0; s < R; ++s) m |= (c == subj[s]) ? (1u << s) : 0u;
  }
  watch[vl] = (u16)m;
}
__global__ void apply_watch_kernel(const u16* __restrict__ watch, u32 n_local, u8* busy, u8* hot_static) {
  const u32 vl = blockIdx.x * blockDim.x + threadIdx.x;
  if (vl >= n_local || watch[vl] == 0) return;
  busy[vl] |= 4;
  hot_static[vl >> TILE_SHIFT] = 1;              // a watcher's tile is scheduled every tick (static flags: never consumed)
}

__global__ void init_state_kernel(uint4* rec, u64* node_state, u32 n_local, u32 stride, u32 R, u32 init_st, u32 init_clock) {
  const u32 vl = blockIdx.x * blockDim.x + threadIdx.x;
  if (vl >= n_local) return;
  Rec r = {};
  r.st = init_st; r.inc = 1; r.status = ST_ALIVE; r.mlstate = ML_ALIVE; r.flags = 1;
  uint4 a, b;
  pack(r, a, b);
  for (u32 s = 0; s < R; ++s) {
    const size_t idx = (size_t)s * stride + vl;
    rec[2 * idx] = a; rec[2 * idx + 1] = b;
  }
  node_state[vl] = (u64)init_clock | NS_UP;
}

__global__ void mark_events_kernel(u8* busy, u8* hot_rd, const u32* ev_node, u32 ev_begin, u32 ev_end, u32 first, u32 n_local) {
  const u32 e = ev_begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ev_end) return;
  const u32 vl = ev_node[e] - first;
  if (vl < n_local) {
    busy[vl] |= 2;                                 // one op per (node, tick): no two threads touch the same byte
    hot_rd[vl >> TILE_SHIFT] = 1;                  // the tile must run this tick
  }
}

__global__ void extract_kernel(const uint4* rec, const u64* node_state, u32 n_local, u32 stride, u32 slot, int what, void* out) {
  const u32 vl = blockIdx.x * blockDim.x + threadIdx.x;
  if (vl >= n_local) return;
  if (what == EXTRACT_CLOCK) { ((u64*)out)[vl] = node_state[vl] & 0xffffffffull; return; }
  if (what == EXTRACT_CLOCK32) { ((u32*)out)[vl] = (u32)node_state[vl]; return; }
  const size_t idx = (size_t)slot * stride + vl;
  Rec r;
  unpack(rec[2 * idx], rec[2 * idx + 1], r);
  const bool known = r.flags & 1;
  switch (what) {
    case EXTRACT_STATUS: ((u8*)out)[vl] = known ? (u8)r.status : (u8)ST_NONE; break;
    case EXTRACT_STATUS_LTIME: ((u64*)out)[vl] = known ? r.st : 0; break;
    case EXTRACT_STATUS_LTIME32: ((u32*)out)[vl] = known ? r.st : 0; break;
    case EXTRACT_INC: ((u32*)out)[vl] = r.inc; break;
    case EXTRACT_ML: ((u8*)out)[vl] = (u8)r.mlstate; break;
  }
}

__global__ void compose_records_kernel(const uint4* rec, const u32* qword, u32 n_local, u32 stride, u32 slot, uint4* out) {
  const u32 vl = blockIdx.x * blockDim.x + threadIdx.x;
  if (vl >= n_local) return;
  const size_t idx = (size_t)slot * stride + vl;
  uint4 b = rec[2 * idx + 1];
  merge_queue_word(b, qword[idx]);
  out[2 * (size_t)vl] = rec[2 * idx]; out[2 * (size_t)vl + 1] = b;
}

__global__ void __launch_bounds__(BLOCK) state_hash_kernel(const uint4* rec, const u32* qword, const u64* node_state, u32 n_local, u32 stride, u32 first, u32 n_global, u32 R, u64* out) {
  u64 h = 0;
  for (u32 vl = blockIdx.x * BLOCK + threadIdx.x; vl < n_local; vl += gridDim.x * BLOCK) {
    for (u32 s = 0; s < R; ++s) {
      const size_t idx = (size_t)s * stride + vl;
      uint4 b = rec[2 * idx + 1];
      merge_queue_word(b, qword[idx]);
      h += rec_hash((u64)s * n_global + first + vl, rec[2 * idx], b);
    }
    h += node_hash((u64)R * n_global + first + vl, node_state[vl]);
  }
  h = warp_sum64(h);
  if ((threadIdx.x & 31) == 0 && h) atomicAdd((unsigned long long*)out, (unsigned long long)h);
}

// out[0] = max clock, out[1] = queued intents, out[2+2s] = min key, out[3+2s] = max key of slot s over
// up nodes other than the subject (agreement check for Stats / convergence studies).
__global__ void __launch_bounds__(BLOCK) summary_kernel(const uint4* rec, const u32* qword, const u64* node_state, u32 n_local, u32 stride, u32 first, u32 R, const u32* subj, u64* out) {
  u64 maxclock = 0, queued = 0;
  for (u32 s = 0; s < R; ++s) {
    u64 kmin = ~0ull, kmax = 0;
    const u32 sid = subj[s];
    for (u32 vl = blockIdx.x * BLOCK + threadIdx.x; vl < n_local; vl += gridDim.x * BLOCK) {
      const u64 ns = node_state[vl];
      if (s == 0) maxclock = max(maxclock, (u64)(ns & 0xffffffffull));
      const size_t idx = (size_t)s * stride + vl;
      Rec r;
      unpack(rec[2 * idx], rec[2 * idx + 1], r);
      { const u32 q = qword[idx]; queued += ((q & 0xffu) ? 1 : 0) + (((q >> 8) & 0xffu) ? 1 : 0); }
      if ((ns & NS_UP) && sid != first + vl) {
        const bool known = r.flags & 1;
        const u64 key = (((u64)r.st << 32) ^ ((u64)r.inc << 8) ^ ((u64)(known ? r.status : 0) << 4) ^ r.mlstate ^ ((u64)known << 63));
        kmin = min(kmin, key); kmax = max(kmax, key);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
      kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin((unsigned long long*)(out + 2 + 2 * s), (unsigned long long)kmin);
      atomicMax((unsigned long long*)(out + 3 + 2 * s), (unsigned long long)kmax);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) maxclock = max(maxclock, __shfl_xor_sync(0xffffffffu, maxclock, o));
  queued = warp_sum64(queued);
  if ((threadIdx.x & 31) == 0) {
    atomicMax((unsigned long long*)out, (unsigned long long)maxclock);
    if (queued) atomicAdd((unsigned long long*)(out + 1), (unsigned long long)queued);
  }
}

}  // namespace

int tick_ctas_per_sm_r1() { return MB_R1; }
int tick_ctas_per_sm_r1s() { return MB_R1S; }
int tick_ctas_per_sm_rn() { return MB_RN; }
int tick_grid_size(u32 n_local, int ctas_per_sm) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  const u32 tiles = (n_local + BLOCK - 1) / BLOCK;
  u32 grid = (u32)sms * (u32)ctas_per_sm * 2u;          // persistent: SM count × resident CTAs × 2 (two waves for balance)
  if (tiles < grid) grid = tiles ? tiles : 1;
  while ((tiles + grid - 1) / grid > MAX_TILES_PER_CTA) grid += (u32)sms * (u32)ctas_per_sm;
  return (int)grid;
}

template <bool TRACE, int FMAX>
static void launch_tick_v(const TickParams& p, int grid, cudaStream_t st) {
  const bool sharded = p.world > 1, r1 = p.R == 1;
  if (sharded) { if (r1) SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<TRACE, FMAX, true, true, MB_R1S>)(p); else SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<TRACE, FMAX, true, false, MB_RN>)(p); }
  else if (r1) SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<TRACE, FMAX, false, true, MB_R1>)(p);
  else SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<TRACE, FMAX, false, false, MB_RN>)(p);
}
void launch_tick(const TickParams& p, bool trace, int grid, cudaStream_t st) {
  const bool small = p.fanout <= 4;          // the common fan-outs (3, 4) get the 4-wide target array
  if (trace) { if (small) launch_tick_v<true, 4>(p, grid, st); else launch_tick_v<true, 8>(p, grid, st); }
  else { if (small) launch_tick_v<false, 4>(p, grid, st); else launch_tick_v<false, 8>(p, grid, st); }
}
// The single-view kernel of a dual launch (SV_SINGLE): the single-slot kernel on the one view that has business (multi-slot plane layout).
void launch_tick_single_view(const TickParams& p, int grid, cudaStream_t st) {
  const bool sharded = p.world > 1;
  if (p.fanout <= 4) {
    if (sharded) SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<false, 4, true, true, MB_R1S>)(p);
    else SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<false, 4, false, true, MB_R1>)(p);
  } else {
    if (sharded) SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<false, 8, true, true, MB_R1S>)(p);
    else SFS_LAUNCH(grid, BLOCK, 0, st, tick_kernel<false, 8, false, true, MB_R1>)(p);
  }
}
void launch_fill_idle_rows(u64* rows, u64* grow_rows, u32 n, const u32* sched, bool trace, cudaStream_t st) {
  if (n) SFS_LAUNCH((n + 127) / 128, 128, 0, st, fill_idle_rows_kernel)(rows, grow_rows, n, sched, trace ? 1 : 0);
}
void launch_pushpull(const TickParams& p, const uint4* snap_rec, const u64* snap_node, bool trace, cudaStream_t st) {
  if (trace) SFS_LAUNCH(SFS_SMS * 8, BLOCK, 0, st, pushpull_kernel<true>)(p, snap_rec, snap_node);
  else SFS_LAUNCH(SFS_SMS * 8, BLOCK, 0, st, pushpull_kernel<false>)(p, snap_rec, snap_node);
}
void launch_compute_watch(const u32* row_ptr, const u32* col, const u32* subj_dev, u32 R, u32 first, u32 n_local, u16* watch, cudaStream_t st) {
  SFS_LAUNCH((n_local + 255) / 256, 256, 0, st, compute_watch_kernel)(row_ptr, col, subj_dev, R, first, n_local, watch);
}
void launch_apply_watch(const u16* watch, u32 n_local, u8* busy, u8* hot_static, cudaStream_t st) {
  SFS_LAUNCH((n_local + 255) / 256, 256, 0, st, apply_watch_kernel)(watch, n_local, busy, hot_static);
}
void launch_drain(const DrainParams& p, cudaStream_t st) {
  SFS_LAUNCH(SFS_SMS * 8, BLOCK, 0, st, drain_kernel)(p);
  if (p.byz_on) SFS_LAUNCH(SFS_SMS * 2, BLOCK, 0, st, clear_windows_kernel)(p);
}
void launch_publish(const PublishParams& p, cudaStream_t st) { SFS_LAUNCH(1, 32, 0, st, publish_kernel)(p); }
void launch_init_state(uint4* rec, u64* node_state, u32 n_local, u32 stride, u32 R, u32 init_st, u32 init_clock, cudaStream_t st) {
  SFS_LAUNCH((n_local + 255) / 256, 256, 0, st, init_state_kernel)(rec, node_state, n_local, stride, R, init_st, init_clock);
}
void launch_mark_events(u8* busy, u8* hot_rd, const u32* ev_node, u32 ev_begin, u32 ev_end, u32 first, u32 n_local, cudaStream_t st) {
  const u32 n = ev_end - ev_begin;
  if (!n) return;
  SFS_LAUNCH((n + 127) / 128, 128, 0, st, mark_events_kernel)(busy, hot_rd, ev_node, ev_begin, ev_end, first, n_local);
}
void launch_extract(const uint4* rec, const u64* node_state, u32 n_local, u32 stride, u32 slot, int what, void* out, cudaStream_t st) {
  SFS_LAUNCH((n_local + 255) / 256, 256, 0, st, extract_kernel)(rec, node_state, n_local, stride, slot, what, out);
}
void launch_compose_records(const uint4* rec, const u32* qword, u32 n_local, u32 stride, u32 slot, uint4* out, cudaStream_t st) {
  SFS_LAUNCH((n_local + 255) / 256, 256, 0, st, compose_records_kernel)(rec, qword, n_local, stride, slot, out);
}
void launch_state_hash(const uint4* rec, const u32* qword, const u64* node_state, u32 n_local, u32 stride, u32 first, u32 n_global, u32 R, u64* out, cudaStream_t st) {
  SFS_LAUNCH(SFS_SMS * 4, BLOCK, 0, st, state_hash_kernel)(rec, qword, node_state, n_local, stride, first, n_global, R, out);
}
void launch_summary(const uint4* rec, const u32* qword, const u64* node_state, u32 n_local, u32 stride, u32 first, u32 R, const u32* subj_dev, u64* out, cudaStream_t st) {
  SFS_LAUNCH(SFS_SMS * 4, BLOCK, 0, st, summary_kernel)(rec, qword, node_state, n_local, stride, first, R, subj_dev, out);
}

}  // namespace sfs
