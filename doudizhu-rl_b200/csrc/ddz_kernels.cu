// ddz_kernels.cu -- sm_100a kernels and the C-ABI launchers of libddz_b200.so (see include/ddz_b200.h).
//
// k_env<V, MODE> is the whole env-step in ONE launch.  The unit of work is a WARP: warp <-> 32 consecutive envs
// (lane <-> env for the rule work, the whole warp for the output).  Warps never synchronise with each other; a CTA is
// only a container of kWarpsPerCta independent warps.
//   1. tile id = launch position when the whole grid is resident at once, else an atomic ticket in start order;
//      coalesced SoA load of the packed state (+ previous offsets / choice, all in flight together)
//   2. [MODE step] pick the move (index / entropy % N / Philox % N / explicit), apply it, terminal + rewards,
//      [re-deal finished envs from the host-supplied permutation pool, the whole warp working on one deal at a time],
//      store the state
//   3. count legal moves (closed form: popc x binomial), warp exclusive scan (shfl), publish the warp total for the
//      decoupled look-back that turns per-warp totals into global CSR offsets without a second pass over the state
//   4. face rows: the C count planes of every env go to shared memory; lanes 0..29 are (row parity, rank) pairs, so
//      one warp instruction writes two whole 240-byte rows as 30 coalesced 128-bit streaming stores (st.global.cs),
//      each value coming from a 5-entry thermometer LUT
//   5. enumerate the legal moves in canonical order into a shared-memory window: short lists one env per lane, long
//      lists (> kHeavy moves) by the whole warp (lane j = j-th rank / j-th chunk of kicker sets, found by unranking)
//   6. look-back (kLookBack windows of 32 predecessor tiles per round trip; any wait is hidden behind 4 or 5)
//      -> global base, offsets; packed list (coalesced) and the action rows (same row writer as the face)
//   Odd tiles run 5-6 before 4, even tiles 4 before 5-6: about half of an SM's warps stream rows while the other half
//   does rule work.
// Stores are fire-and-forget: no staging tiles, no waits.  Nothing is re-read from HBM: algorithmic bytes == DRAM
// traffic (profiles/).  Two earlier variants that staged rows in shared memory and pushed them with TMA bulk stores
// (cp.async.bulk) measured slower (DESIGN.md, profiles/r1b*, r1c*): the path is nowhere near issue-bound, what it
// needs is many independent warps with stores in flight and no synchronisation.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cfloat>
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>
#include <type_traits>

#include "../../include/ddz_b200.h"
#include "ddz_device.cuh"
#include <cuda_bf16.h>
#include <math_constants.h>
#include "ddz_flat.cuh"
#include "ddz_search.cuh"
#include "ddz_ids.cuh"
#include "ddz_policy.cuh"
#include "ddz_policy_linear.cuh"

namespace ddz {

#ifndef DDZ_THREADS
#define DDZ_THREADS 64
#endif
constexpr int kThreads = DDZ_THREADS;            // threads per CTA
constexpr int kWarpsPerCta = kThreads / 32;
constexpr int kEnvs = 128;                       // envs per CTA for the simple thread-per-env kernels
constexpr int kWin = 320;                        // legal moves staged per window (one warp)
constexpr int kMinCtasPerSm = 28 / kWarpsPerCta;  // 28 warps per SM (one wave at 131 072 envs): <= 72 registers
#ifdef DDZ_PLAIN_STORES
#define DDZ_STORE(p, v) (*(p) = (v))
#else
#define DDZ_STORE(p, v) __stcs((p), (v))
#endif
#ifndef DDZ_HEAVY
#define DDZ_HEAVY 32
#endif
#ifndef DDZ_ROW_UNROLL
#define DDZ_ROW_UNROLL 4
#endif
#ifndef DDZ_LOOKBACK
#define DDZ_LOOKBACK 4
#endif
#ifndef DDZ_TILE_ENVS
#define DDZ_TILE_ENVS 32
#endif
constexpr int kTile = DDZ_TILE_ENVS;                     // envs per warp tile (lane <-> env for lanes < kTile)
constexpr int kRowUnroll = DDZ_ROW_UNROLL;               // row-writer iterations in flight per lane
constexpr int kHeavy = DDZ_HEAVY;                       // envs with more legal moves than this are expanded by the whole warp
#ifndef DDZ_PHASE_ORDER
#define DDZ_PHASE_ORDER 0
#endif
// which of the two output phases a tile runs first: 0 = odd tiles rule work first, even tiles face rows first (default),
// 1 = every tile face rows first, 2 = every tile rule work first
DDZ_DEV bool kFaceSecond(int t) { return DDZ_PHASE_ORDER == 0 ? (t & 1) != 0 : DDZ_PHASE_ORDER == 2; }
constexpr int kLookBack = DDZ_LOOKBACK;                     // look-back windows (of 32 predecessor tiles) fetched per round trip

enum Mode { kStepOnly = 0, kObserve = 1, kStepObserve = 2 };

// The two probability planes of a face (native get_state_prob, envi.py:94; get_state_prob_manual, server/core.py:26-33) are
// "cards nobody has shown yet", scaled by the share of each opponent's hand.  Their layout inside a rank's four slots is
// not pinned by anything in the reference (oracle/SEMANTICS.md):
//   form A (default)        thermometer(unknown count), left-aligned like every other plane;
//   form B (-DDDZ_PROB_FORM_B)  deck60 - known60 element-wise: the ones are RIGHT-aligned (jokers have one slot: unchanged).
// Form B rows carry bit 3 in the nibbles of ranks 0..12 and read the reversed half of a 16-entry thermometer LUT.
#ifdef DDZ_PROB_FORM_B
constexpr int kProbForm = 1, kLutEntries = 16;
constexpr uint64_t kProbMark = 0x0008888888888888ull;
#else
constexpr int kProbForm = 0, kLutEntries = 8;
constexpr uint64_t kProbMark = 0ull;
#endif
// entry i of the thermometer LUT: i = count 0..4 -> {c>0, c>1, c>2, c>3}; i = 8 + count -> the same ones right-aligned
DDZ_DEV float4 lut_entry(int i) {
    const int c = i & 7;
    return (i & 8) ? make_float4(c > 3 ? 1.f : 0.f, c > 2 ? 1.f : 0.f, c > 1 ? 1.f : 0.f, c > 0 ? 1.f : 0.f)
                   : make_float4(c > 0 ? 1.f : 0.f, c > 1 ? 1.f : 0.f, c > 2 ? 1.f : 0.f, c > 3 ? 1.f : 0.f);
}

// workspace: header (ticket, finished, epoch) + one look-back word per warp tile.  Must be zero when first used.
struct WsHeader { unsigned int ticket, finished, epoch, auto_step; };
struct Workspace { WsHeader* h; unsigned long long* tile; };
static inline int ntiles(int B) { return (B + kTile - 1) / kTile; }
static inline int nblocks(int B) { return (B + kEnvs - 1) / kEnvs; }
static inline Workspace ws_of(void* p) {
    Workspace w; w.h = (WsHeader*)p; w.tile = (unsigned long long*)((char*)p + 256);
    return w;
}
// look-back word: [63:34] epoch, [33:32] status (1 = tile total, 2 = inclusive prefix), [31:0] value
constexpr unsigned long long kAggregate = 1ull << 32, kInclusive = 2ull << 32;

// ------------------------------------------------------------------------------------------------
// small PTX wrappers
// ------------------------------------------------------------------------------------------------
DDZ_DEV unsigned long long ld_relaxed(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
DDZ_DEV void st_relaxed(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

#ifdef DDZ_TRACE
// developer build only (profiles/trace_phases.py): per-warp phase timestamps, 8 x uint64 per tile
__device__ unsigned long long* g_trace = nullptr;
DDZ_DEV void trace(int tile, int slot) {
    if (g_trace && (threadIdx.x & 31) == 0) {
        unsigned long long ts; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(ts));
        g_trace[(size_t)tile * 8 + slot] = ts;
    }
}
#else
DDZ_DEV void trace(int, int) {}
#endif

DDZ_DEV long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}
DDZ_DEV void stat_add(int64_t* stats, int slot, long long v) {   // per-lane values are small (|v| <= a few hundred)
    const int s = __reduce_add_sync(0xFFFFFFFFu, (int)v);
    if ((threadIdx.x & 31) == 0 && s != 0 && stats) atomicAdd((unsigned long long*)&stats[slot], (unsigned long long)(long long)s);
}
// per-lane step summary (see `sf` in k_env) -> the stats vector; rewards per game.py:109-118
DDZ_DEV void step_stats(int64_t* stats, unsigned int sf, const int32_t* rewards, int extra_err) {
    const int over = (sf >> 2) & 1, winner = (sf >> 3) & 3;
    stat_add(stats, 4, sf & 1);
    stat_add(stats, 9, (sf >> 1) & 1);
    stat_add(stats, 0, over);
    stat_add(stats, 1, over && winner == 1);
    stat_add(stats, 2, over && winner == 2);
    stat_add(stats, 3, over && winner == 0);
    stat_add(stats, 5, over ? (winner == 1 ? rewards[1] : -rewards[1]) : 0);
    stat_add(stats, 6, over ? (winner == 1 ? -(rewards[0] + rewards[2]) : rewards[0] + rewards[2]) : 0);
    stat_add(stats, 7, (int)((sf >> 5) & 3) + extra_err);
}


// Decoupled look-back over the per-tile words: sum of the totals of all tiles before `t` (kLookBack windows of 32
// predecessors per round trip), then publish this tile's inclusive prefix.  Never hangs: after 2^22 polls the tile flags
// an error (stats[7]), sets `timed_out` -- the caller then writes none of its rows, its base being unknown -- and carries on.
DDZ_DEV long long tile_lookback(const Workspace& ws, int t, unsigned long long epoch_tag, int total, int lane, int64_t* stats,
                                bool& timed_out) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    long long base = 0;
    timed_out = false;
    if (t <= 0) return 0;
    int p = t - 1;
    unsigned int spins = 0;
    bool finished = false;
    while (!finished) {
        unsigned long long w[kLookBack];
#pragma unroll
        for (int j = 0; j < kLookBack; j++) {
            const int idx = p - 32 * j - lane;
            w[j] = idx >= 0 ? ld_relaxed(&ws.tile[idx]) : (epoch_tag | kInclusive);   // before tile 0: prefix 0
        }
#pragma unroll
        for (int j = 0; j < kLookBack; j++) {
            if (finished) break;
            const bool ok = ((w[j] >> 34) == (epoch_tag >> 34)) && ((w[j] >> 32) & 3ull) != 0;
            if (!__all_sync(FULL, ok)) {    // not published yet: poll again from this window
                __nanosleep(64);
                if (++spins > (1u << 22)) { // never hang the GPU: flag the error and carry on
                    if (lane == 0 && stats) atomicAdd((unsigned long long*)&stats[7], 1ull);
                    finished = true; timed_out = true;
                }
                break;
            }
            const unsigned int incmask = __ballot_sync(FULL, ((w[j] >> 32) & 3ull) == 2ull);
            // lanes up to and including the nearest inclusive predecessor contribute
            const int stop = incmask ? (__ffs(incmask) - 1) : 31;
            base += warp_sum_ll(lane <= stop ? (long long)(unsigned int)w[j] : 0ll);
            p -= 32;
            if (incmask) finished = true;
        }
    }
    if (lane == 0) st_relaxed(&ws.tile[t], epoch_tag | kInclusive | (unsigned int)(base + total));
    return base;
}

// ------------------------------------------------------------------------------------------------
// deal
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kEnvs) k_reset(void* state, const int8_t* __restrict__ perm,
                                                 const int8_t* __restrict__ lord_pile, int pool_games,
                                                 int only_done, int64_t* stats, int B) {
    const int b = blockIdx.x * kEnvs + threadIdx.x, lane = threadIdx.x & 31;
    const bool valid = b < B;
    StateView v = view_of(state, B);
    Env e;
    if (valid) e = load_env(v, b); else e.meta = 0;
    const bool want = valid && (!only_done || e.done());
    const unsigned int need = __ballot_sync(0xFFFFFFFFu, want);
    const unsigned int bad = warp_deal(need, e, perm, lord_pile, pool_games, B, b, lane);
    if (want) store_env(v, b, e);
    if (lane == 0 && bad && stats) atomicAdd((unsigned long long*)&stats[7], (unsigned long long)__popc(bad));
}

// ------------------------------------------------------------------------------------------------
// thermometer rows (envi.py:140-146): 240-byte rows of 15 float4, rank k -> {c>0, c>1, c>2, c>3} * s
// ------------------------------------------------------------------------------------------------
// Lane l < 30 owns rank k = l % 15 of the rows with parity l / 15: one warp store instruction covers two complete
// rows (480 contiguous bytes).  The nibble position is a per-lane constant, the row index an immediate.
struct RowLane {
    int first;        // 0 or 1: first row of this lane; huge for the parked lanes 30, 31
    int k;            // rank
    uint32_t sh;      // shift of the rank's nibble inside its 32-bit half, pre-scaled to a LUT byte offset
    bool hi;          // rank >= 8 -> upper half of the packed word
    DDZ_DEV static RowLane make(int lane) {
        RowLane r; r.first = lane / 15; r.k = lane - 15 * r.first; r.hi = r.k >= 8; r.sh = 4u * (uint32_t)(r.k & 7);
        if (lane >= 30) { r.first = 0x3FFFFFFF; r.k = 0; }   // parked: the row loops never run
        return r;
    }
    DDZ_DEV const float4& thermo(uint64_t packed, const float4* lut) const {
        const uint32_t w = hi ? (uint32_t)(packed >> 32) : (uint32_t)packed;
        return lut[(w >> sh) & 15u];
    }
};
struct FaceRow { uint64_t packed; float s; float pad; };   // 16 B: one LDS.128 per store

// rows [0, nrows) of the warp's contiguous block starting at gdst; src(r) yields the packed counts (and scale)
template <class RowT>
DDZ_DEV void write_rows(float4* __restrict__ gdst, int nrows, const RowLane& rl, const float4* __restrict__ lut,
                        const RowT* __restrict__ rows);
template <>
DDZ_DEV void write_rows<FaceRow>(float4* __restrict__ gdst, int nrows, const RowLane& rl, const float4* __restrict__ lut,
                                 const FaceRow* __restrict__ rows) {
    float4* dst = gdst + (rl.first & 1) * 15 + rl.k;
#pragma unroll (kRowUnroll)
    for (int r = rl.first; r < nrows; r += 2, dst += 30) {
        const float4 raw = *reinterpret_cast<const float4*>(&rows[r]);
        const uint64_t packed = ((uint64_t)__float_as_uint(raw.y) << 32) | __float_as_uint(raw.x);
        const float s = raw.z;
        float4 q = rl.thermo(packed, lut);
        q.x *= s; q.y *= s; q.z *= s; q.w *= s;
        DDZ_STORE(dst, q);
    }
}
template <>
DDZ_DEV void write_rows<uint64_t>(float4* __restrict__ gdst, int nrows, const RowLane& rl, const float4* __restrict__ lut,
                                  const uint64_t* __restrict__ rows) {
    float4* dst = gdst + (rl.first & 1) * 15 + rl.k;
#pragma unroll (kRowUnroll)
    for (int r = rl.first; r < nrows; r += 2, dst += 30) DDZ_STORE(dst, rl.thermo(rows[r], lut));
}

template <int V> struct FaceCfg;
template <> struct FaceCfg<0> { static constexpr int C = 4; };
template <> struct FaceCfg<1> { static constexpr int C = 7; };
template <> struct FaceCfg<2> { static constexpr int C = 9; };
template <> struct FaceCfg<3> { static constexpr int C = 6; };

// the C count planes of env e for variant V (envi.py:87-217); the last two are the unknown-card plane,
// scaled by p[0], p[1] = share of the next / next-next player's hand (get_state_prob, SURVEY App. A)
template <int V>
DDZ_DEV void face_planes(const Env& e, uint64_t* planes /*[C]*/, float* p /*[2]*/) {
    int s = e.cur(), prev = (s + 2) % 3, next = (s + 1) % 3;
    uint64_t hand = pick3(s, e.hand[0], e.hand[1], e.hand[2]);
    uint64_t taken = e.hist[0] + e.hist[1] + e.hist[2];
    int n = 0;
    planes[n++] = hand;
    planes[n++] = taken;
    if (V == 1 || V == 2) {
        planes[n++] = pick3(prev, e.hist[0], e.hist[1], e.hist[2]);
        planes[n++] = pick3(s, e.hist[0], e.hist[1], e.hist[2]);
        planes[n++] = pick3(next, e.hist[0], e.hist[1], e.hist[2]);
    }
    if (V == 2 || V == 3) {
        planes[n++] = pick3(prev, e.recent[0], e.recent[1], e.recent[2]);
        planes[n++] = pick3(next, e.recent[0], e.recent[1], e.recent[2]);   // (role-2)%3 == next
    }
    uint64_t unknown = (kDeckPacked - taken - hand) | kProbMark;
    planes[n++] = unknown;
    planes[n++] = unknown;
    int size1 = card_count(pick3(next, e.hand[0], e.hand[1], e.hand[2]));
    int size2 = card_count(pick3(prev, e.hand[0], e.hand[1], e.hand[2]));
    int tot = size1 + size2;
    p[0] = tot > 0 ? __fdiv_rn((float)size1, (float)tot) : 0.f;
    p[1] = tot > 0 ? __fdiv_rn((float)size2, (float)tot) : 0.f;
}

struct StepArgs {
    const int32_t* offsets; const uint64_t* actions; const void* choice; int mode;
    uint64_t seed, env0; uint32_t stepno; int32_t rewards[3];
    const int8_t* perm; const int8_t* lord_pile; int pool_games;
    int8_t* r; uint8_t* done; int8_t* cat; float* reward;
    long long prev_cap;   // capacity of `actions` (-1 = unknown, lists complete): a list cut off by an overflow is never read
                          // past it; 0 is a capacity like any other (nothing stored: every live env sits the step out)
};
struct OutArgs {
    int32_t* offsets; uint64_t* actions_u64; float4* actions_f32; long long cap; float4* face;
    int static_tiles;   // 1: the whole grid is resident at once, tile = launch position (no ticket round trip)
};


struct SeqWindowEmitter {  // enumerate_legal functor: keeps the moves that fall into the warp's current window
    uint64_t* out; int pos, win;   // pos = index of the next move relative to the window start (may be negative)
    DDZ_DEV void operator()(uint64_t mv) { if ((unsigned)pos < (unsigned)win) out[pos] = mv; pos++; }
};
struct WindowEmitter {   // enumerate_legal_warp functor: move number idx of the env goes to window slot base + idx
    uint64_t* out; int base, win;
    DDZ_DEV void operator()(int idx, uint64_t mv) { const unsigned rel = (unsigned)(base + idx); if (rel < (unsigned)win) out[rel] = mv; }
};

struct __align__(128) WarpSmem {
    FaceRow face[32 * 9];                                   // 4 608 B
    uint64_t moves[kWin];                                   // 2 560 B
    float4 lut[kLutEntries];
};

// V: face variant or -1 (no face).  MODE: see enum Mode.  The body of k_env and of lean::k_step_observe.
template <int V, int MODE>
DDZ_DEV void env_kernel(void* state, const StepArgs& a, const OutArgs& o, const Workspace& ws, int64_t* stats, int B) {
    constexpr bool STEP = (MODE == kStepOnly || MODE == kStepObserve);
    constexpr bool EMIT = (MODE != kStepOnly);
    constexpr int C = FaceCfg<(V < 0 ? 0 : V)>::C;
    constexpr unsigned FULL = 0xFFFFFFFFu;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    WarpSmem& sm = reinterpret_cast<WarpSmem*>(smem_raw)[wib];
    const RowLane rl = RowLane::make(lane);
    const int nt = (B + kTile - 1) / kTile;
    const unsigned int nwarps = gridDim.x * kWarpsPerCta;

    // ---- 1. tile ticket: tiles are handed out in start order, so every lower tile is already running
    int t = blockIdx.x * kWarpsPerCta + wib;
    unsigned int epoch = 0, autostep = 0, stepno = a.stepno;   // epoch / autostep: valid in lane 0 until broadcast below
    if (EMIT) {
        // Tiles must be handed out so that every lower tile is already running (the look-back waits on them): by a
        // ticket in start order, or -- when the whole grid is resident at once -- simply by launch position, which
        // saves a dependent round trip before the first state load.
        if (lane == 0) {
            if (!o.static_tiles) t = (int)atomicAdd(&ws.h->ticket, 1u);
            epoch = ws.h->epoch; autostep = ws.h->auto_step;
        }
        if (!o.static_tiles) t = __shfl_sync(FULL, t, 0);
        if (lane < kLutEntries) sm.lut[lane] = lut_entry(lane);
        __syncwarp();
    }
    if (t < nt) {
    const int b0 = t * kTile, b = b0 + lane;
    const bool valid = lane < kTile && b < B;
    const int nenv = min(kTile, B - b0);
    trace(t, 0);

    // ---- 2. state transition
    Env e;
    e.meta = 0;
    uint64_t hand = 0, last = 0;
    Masks hm{0, 0, 0, 0};
    Rule ru{true, 0, 1, 0};
    int n = 0;
    unsigned int sf = 0;   // per-lane step summary for the stats: bit0 stepped, bit1 pass, bit2 game over, bits3-4 winner, bits5-6 errors
    int prev_off = 0, prev_end = 0;
    uint64_t choice_raw = 0;
    if (valid) {
        if (STEP) {   // independent of the state: all of these loads are in flight together
            prev_off = a.offsets[b]; prev_end = a.offsets[b + 1];
            if (a.mode == DDZ_CHOICE_MOVE) choice_raw = ((const uint64_t*)a.choice)[b];
            else if (a.mode != DDZ_CHOICE_PHILOX) choice_raw = ((const uint32_t*)a.choice)[b];
        }
        e = load_env(view_of(state, B), b);
        if (STEP && a.perm) {   // most envs will not need it this step, but an L2 prefetch of the env's next deal
            const char* prow = reinterpret_cast<const char*>(a.perm) +   // takes the HBM latency off the re-deal path
                               54 * ((size_t)((e.meta >> 8) % (uint32_t)a.pool_games) * B + b);
            asm volatile("prefetch.global.L2 [%0];" ::"l"(prow));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(prow + 53));
        }
    }
    if (EMIT) {   // broadcast what lane 0 read at the top -- after the state loads were issued, not before
        epoch = __shfl_sync(FULL, epoch, 0);
        autostep = __shfl_sync(FULL, autostep, 0);
        if (STEP && a.stepno == DDZ_STEPNO_AUTO) stepno = autostep;
    }
    const unsigned long long epoch_tag = (unsigned long long)(epoch & 0x3FFFFFFFu) << 34;
    if (valid) {
        if (STEP) {
            int o_r = 0, o_cat = -1;
            float rw0 = 0.f, rw1 = 0.f, rw2 = 0.f;
            if (!e.done()) {
                // A list cut off by an overflow of the action buffer (stats[7] said so when it was written) is played from
                // its visible part: `cnt` counts the entries that were stored.  An env whose list was dropped altogether
                // sits this step out -- counted in stats[7], but NOT a sticky error: its next list may fit again.
                const int base = prev_off, full = prev_end - prev_off;
                const int cnt = a.prev_cap >= 0 ? (int)max(0ll, min((long long)full, a.prev_cap - base)) : full;
                long long idx = -1;
                if (a.mode == DDZ_CHOICE_INDEX) idx = (int32_t)(uint32_t)choice_raw;
                else if (a.mode == DDZ_CHOICE_MOD) idx = cnt > 0 ? (long long)((uint32_t)choice_raw % (uint32_t)cnt) : -1;
                else if (a.mode == DDZ_CHOICE_PHILOX) idx = cnt > 0 ? (long long)(philox(a.seed, a.env0 + (uint64_t)b, stepno) % (uint32_t)cnt) : -1;
                else {
                    const uint64_t want = choice_raw;
                    for (int i = 0; i < cnt; i++) if (a.actions[base + i] == want) { idx = i; break; }
                }
                if (idx < 0 || idx >= cnt) {
                    sf += 32u;
                    if (!(cnt == 0 && full > 0)) e.meta |= 0x20u;      // illegal choice: sticky; dropped list: wait for the next one
                } else {
                    const uint64_t mv = a.actions[base + idx];
                    StepOut so = apply_move(e, mv, a.rewards);
                    o_r = so.r; o_cat = so.cat; rw0 = so.reward[0]; rw1 = so.reward[1]; rw2 = so.reward[2];
                    sf |= 1u | (so.pass ? 2u : 0u);
                    if (so.done) sf |= 4u | ((unsigned int)so.winner << 3);
                }
            }
            if (a.r) a.r[b] = (int8_t)o_r;
            if (a.done) a.done[b] = (uint8_t)e.done();
            if (a.cat) a.cat[b] = (int8_t)o_cat;
            if (a.reward) { a.reward[3 * (size_t)b] = rw0; a.reward[3 * (size_t)b + 1] = rw1; a.reward[3 * (size_t)b + 2] = rw2; }
        }
    }
    {
        if (STEP) {
            if (a.perm) {   // re-deal the finished envs, the whole warp working on one of them at a time
                const unsigned int need = __ballot_sync(FULL, valid && e.done());
                sf += ((warp_deal(need, e, a.perm, a.lord_pile, a.pool_games, B, b, lane) >> lane) & 1u) << 5;
            }
            if (valid) store_env(view_of(state, B), b, e);
        }
        if (valid && EMIT && !e.done()) {
            hand = hand_to_move(e); last = trick_of(e);
            hm = masks_of(hand); ru = rule_of(last); n = count_legal(hm, ru, last != 0);
        }
    }
    if (STEP && !EMIT) step_stats(stats, sf, a.rewards, 0);
    if (EMIT) {
    // ---- 3. warp scan, publish the warp total for the look-back (other tiles wait on it: nothing else comes first)
    int inc = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int u = __shfl_up_sync(FULL, inc, d); if (lane >= d) inc += u; }
    const int local = inc - n;
    const int total = __shfl_sync(FULL, inc, 31);
    if (lane == 0) st_relaxed(&ws.tile[t], epoch_tag | (t == 0 ? kInclusive : kAggregate) | (unsigned int)total);

    // ---- 4. the face planes of every env go to shared memory while the state is still in registers
    if (V >= 0 && o.face && valid) {
        uint64_t pl[C]; float p[2];
        face_planes<(V < 0 ? 0 : V)>(e, pl, p);
#pragma unroll
        for (int c = 0; c < C; c++) {
            FaceRow fr; fr.packed = pl[c]; fr.s = (c >= C - 2) ? p[c - (C - 2)] : 1.f; fr.pad = 0.f;
            *reinterpret_cast<float4*>(&sm.face[lane * C + c]) = *reinterpret_cast<const float4*>(&fr);
        }
    }
    __syncwarp();
    trace(t, 1);

    // Two output phases.  Odd tiles run them in the opposite order, so that at any moment about half of the warps
    // of an SM stream rows out while the other half does rule work (look-back, enumeration).
    int disagree = 0;
#pragma unroll 1
    for (int ph = 0; ph < 2; ph++) {
    if ((ph == 0) != kFaceSecond(t)) {
        // ---- 5. face rows: [nenv][C] rows of 240 B, contiguous for the warp
        trace(t, 2);
        if (V >= 0 && o.face) write_rows<FaceRow>(o.face + (size_t)b0 * C * 15, nenv * C, rl, sm.lut, sm.face);
        trace(t, 3);
    } else {
        trace(t, 4);
        // ---- 6..8. per window of kWin moves: enumerate into shared memory; (first window only) look-back for the
        // global base -- whatever wait it has is hidden behind the enumeration; then packed list + one-hot rows out
        long long base = 0, lim = 0;
        int w0 = 0;
        // without a face (ddz_legal_emit) the face-row buffer is free: the window grows from kWin to kWin + 576 moves
        uint64_t* const wbuf = (V < 0) ? reinterpret_cast<uint64_t*>(sm.face) : sm.moves;
        const int win = (V < 0) ? (int)(sizeof(sm.face) / 8) + kWin : kWin;
#pragma unroll 1
        do {
            const bool inwin = n > 0 && local < w0 + win && local + n > w0;
            if (inwin && n <= kHeavy) {                     // short lists: one env per lane
                SeqWindowEmitter em{wbuf, local - w0, win};
                enumerate_legal(hm, ru, last != 0, em);
                disagree |= (em.pos != local - w0 + n);
            }
            unsigned int heavy = __ballot_sync(FULL, inwin && n > kHeavy);
            while (heavy) {                                 // long lists: the whole warp expands one env at a time
                const int src = __ffs(heavy) - 1; heavy &= heavy - 1;
                Masks sm_; Rule sr;
                sm_.g1 = __shfl_sync(FULL, hm.g1, src); sm_.g2 = __shfl_sync(FULL, hm.g2, src);
                sm_.g3 = __shfl_sync(FULL, hm.g3, src); sm_.g4 = __shfl_sync(FULL, hm.g4, src);
                const int rpack = __shfl_sync(FULL, (int)ru.lead | (ru.cat << 1) | (ru.len << 8) | (ru.val << 16) | ((last != 0) << 24), src);
                sr.lead = rpack & 1; sr.cat = (rpack >> 1) & 127; sr.len = (rpack >> 8) & 255; sr.val = (rpack >> 16) & 255;
                const int loc = __shfl_sync(FULL, local, src), nn = __shfl_sync(FULL, n, src);
                WindowEmitter em{wbuf, loc - w0, win};
                const int got = enumerate_legal_warp(sm_, sr, (rpack >> 24) & 1, lane, em);
                disagree |= (got != nn);
            }
            __syncwarp();
            if (w0 == 0) trace(t, 7);

            if (w0 == 0) {
                bool timed_out;
                base = tile_lookback(ws, t, epoch_tag, total, lane, stats, timed_out);
                if (valid) o.offsets[b] = (int32_t)(base + local);
                if (t == nt - 1 && lane == 0) {
                    o.offsets[B] = (int32_t)(base + total);
                    if (stats) {
                        atomicAdd((unsigned long long*)&stats[8], (unsigned long long)(base + total));
                        if (base + total > o.cap) atomicAdd((unsigned long long*)&stats[7], 1ull);
                    }
                }
                lim = o.cap - base; if (lim > total) lim = total; if (lim < 0 || timed_out) lim = 0;   // rows of this warp that fit
                trace(t, 5);
            }

            const int keep = (int)max(0ll, min((long long)min(win, total - w0), lim - w0));
            for (int i = lane; i < keep; i += 32) o.actions_u64[base + w0 + i] = wbuf[i];   // coalesced
            if (o.actions_f32) write_rows<uint64_t>(o.actions_f32 + (size_t)(base + w0) * 15, keep, rl, sm.lut, wbuf);
            __syncwarp();  // the moves of this window are consumed before the next window overwrites them
            w0 += win;
        } while (w0 < total);
        trace(t, 6);
    }
    }
    step_stats(stats, STEP ? sf : 0u, a.rewards, disagree);
    }  // EMIT
    }  // t < nt
    if (EMIT && lane == 0) {
        const unsigned int fin = atomicAdd(&ws.h->finished, 1u);
        if (fin == nwarps - 1) {                            // the last warp of the launch re-arms the workspace
            ws.h->ticket = 0; ws.h->finished = 0; ws.h->epoch = epoch + 1;
            if (STEP) ws.h->auto_step = (a.stepno == DDZ_STEPNO_AUTO ? autostep : a.stepno) + 1;
            __threadfence();
        }
    }
}
template <int V, int MODE>
__global__ void __launch_bounds__(kThreads, kMinCtasPerSm) k_env(void* state, StepArgs a, OutArgs o,
                                                  Workspace ws, int64_t* stats, int B) {
    env_kernel<V, MODE>(state, a, o, ws, stats, B);
}

// The fused step with a face (ddz_rollout_step) at fewer resident warps: 16 per SM leave 110 registers to a warp, where
// k_env's 28 (one wave of 131 072 envs) leave 72 and spill.  The store stream does not need more warps than that: with
// four env groups of 32 768 envs in flight (bench.py config 4) the step is 5-6 % faster on a B200, 24 / 20 warps per SM
// give 3 % (profiles/r10_lean_step.json).  A launch whose grid does not fit at once at this occupancy runs k_env.
namespace lean {
#ifndef DDZ_LEAN_WARPS_PER_SM
#define DDZ_LEAN_WARPS_PER_SM 16
#endif
constexpr int kMinCtas = DDZ_LEAN_WARPS_PER_SM / kWarpsPerCta;
template <int V>
__global__ void __launch_bounds__(kThreads, kMinCtas) k_step_observe(void* state, StepArgs a, OutArgs o, Workspace ws,
                                                                     int64_t* stats, int B) {
    env_kernel<V, kStepObserve>(state, a, o, ws, stats, B);
}
}  // namespace lean

// ------------------------------------------------------------------------------------------------
// r.get_moves for n independent (hand, last) pairs, long lists welcome (ddz_legal_moves; BASELINE config 5).
// Warp tile = 32 pairs.  Phase A, one lane per pair: count moves and groups, write the hand's rank lists and its group
// descriptors into the warp's shared-memory arena (ddz_flat.cuh).  Phase B, one lane per two consecutive moves of the
// tile: 64 moves per warp iteration; which descriptor a move belongs to comes from a 64-bit bitmap of the group starts
// inside the window (one coalesced load of the next 32 descriptors + two warp OR-reductions), never from a search; the
// pair goes out as one aligned 16-byte store.  Arena rounds: as many whole hands as fit kFlatArena descriptors.
// The CSR offsets come from the same decoupled look-back as k_env; its wait hides behind phase A of the first round.
// ------------------------------------------------------------------------------------------------
#ifndef DDZ_FLAT_WARPS
#define DDZ_FLAT_WARPS 4
#endif
#ifndef DDZ_FLAT_ARENA
#define DDZ_FLAT_ARENA 512
#endif
#ifndef DDZ_FLAT_COUNT_WALK
#define DDZ_FLAT_COUNT_WALK 0     // 1: count moves and groups with a dry walk instead of the closed forms (1.7 % slower)
#endif
#ifndef DDZ_FLAT_MIN_CTAS
#define DDZ_FLAT_MIN_CTAS 7
#endif
#ifndef DDZ_FLAT_PAIR
#define DDZ_FLAT_PAIR 0     // 1: the two moves of a lane are decoded in one interleaved loop (measured 12 % slower), 0: one after the other
#endif
constexpr int kFlatWarps = DDZ_FLAT_WARPS;
constexpr int kFlatArena = DDZ_FLAT_ARENA;      // >= 160: the most groups any 15-rank hand can have is 155
__device__ const flat::SubsetTable g_subsets = flat::SubsetTable();

struct __align__(16) FlatWarpSmem {
    flat::Desc arena[kFlatArena + 2];
    uint8_t lists[32 * flat::kListsPerHand * flat::kListStride];
};

__global__ void __launch_bounds__(kFlatWarps * 32, DDZ_FLAT_MIN_CTAS) k_legal_flat(const uint64_t* __restrict__ hands,
                                                                  const uint64_t* __restrict__ lasts, OutArgs o,
                                                                  Workspace ws, int64_t* stats, int B) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    __shared__ __align__(16) uint16_t s_table[(flat::kTableSize + 7) / 8 * 8];
    __shared__ FlatWarpSmem s_warp[kFlatWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    FlatWarpSmem& sm = s_warp[wib];
    for (int i = threadIdx.x; i < flat::kTableSize; i += kFlatWarps * 32) s_table[i] = g_subsets.v[i];
    const int nt = (B + 31) / 32;
    const unsigned int nwarps = gridDim.x * kFlatWarps;
    int t = blockIdx.x * kFlatWarps + wib;
    unsigned int epoch = 0;
    if (lane == 0) {
        if (!o.static_tiles) t = (int)atomicAdd(&ws.h->ticket, 1u);
        epoch = ws.h->epoch;
    }
    if (!o.static_tiles) t = __shfl_sync(FULL, t, 0);
    __syncthreads();                                        // the subset table is staged
    if (t < nt) {
        const int b = t * 32 + lane;
        const bool valid = b < B;
        uint64_t hand = 0, last = 0;
        if (valid) { hand = hands[b]; last = lasts[b]; }
        epoch = __shfl_sync(FULL, epoch, 0);
        const unsigned long long epoch_tag = (unsigned long long)(epoch & 0x3FFFFFFFu) << 34;
        const Masks hm = masks_of(hand);
        const Rule ru = rule_of(last);
#if DDZ_FLAT_COUNT_WALK
        flat::CountSink cs;
        if (valid) flat::walk_groups(hm, ru, last != 0, 4 * lane, cs);
        const int n = cs.n, ng = cs.ng;
#else
        const int n = valid ? count_legal(hm, ru, last != 0) : 0;           // closed forms: no walk for the counts
        const int ng = valid ? flat::count_groups(hm, ru, last != 0) : 0;
#endif
        int inc = n, dinc = ng;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int u = __shfl_up_sync(FULL, inc, d), v = __shfl_up_sync(FULL, dinc, d);
            if (lane >= d) { inc += u; dinc += v; }
        }
        const int local = inc - n, total = __shfl_sync(FULL, inc, 31);
        const int dloc = dinc - ng, dtotal = __shfl_sync(FULL, dinc, 31);
        if (lane == 0) st_relaxed(&ws.tile[t], epoch_tag | (t == 0 ? kInclusive : kAggregate) | (unsigned int)total);
        if (valid) flat::write_lists(hm, 4 * lane, sm.lists);

        long long base = 0, lim = 0;
        int disagree = 0, h0 = 0;
        bool first = true;
#pragma unroll 1
        while (h0 < 32) {
            // ---- phase A of this round: the hands [h0, h1) whose descriptors fit the arena
            const int D0 = __shfl_sync(FULL, dloc, h0);
            const unsigned int fits = __ballot_sync(FULL, lane >= h0 && dloc + ng - D0 <= kFlatArena);
            const int h1 = h0 + __popc(fits);
            const int m0 = __shfl_sync(FULL, local, h0);
            const int m1s = __shfl_sync(FULL, local, h1 & 31), d1s = __shfl_sync(FULL, dloc, h1 & 31);
            const int m1 = h1 < 32 ? m1s : total, nd = (h1 < 32 ? d1s : dtotal) - D0;
            if (h1 == h0) { disagree = 1; break; }           // cannot happen (a hand has at most 155 groups)
            if (valid && lane >= h0 && lane < h1) {
                flat::WriteSink wsk{sm.arena, dloc - D0, kFlatArena, (uint32_t)local};
                flat::walk_groups(hm, ru, last != 0, 4 * lane, wsk);
                disagree |= (wsk.d != dloc - D0 + ng) | (wsk.start != (uint32_t)(local + n));
            }
            if (lane == 0) { flat::Desc e; e.start = (uint32_t)m1; e.prm = 0; sm.arena[nd] = e; }
            __syncwarp();
            if (first) {
                first = false;
                bool timed_out;
                base = tile_lookback(ws, t, epoch_tag, total, lane, stats, timed_out);
                if (valid) o.offsets[b] = (int32_t)(base + local);
                if (t == nt - 1 && lane == 0) {
                    o.offsets[B] = (int32_t)(base + total);
                    if (stats) {
                        atomicAdd((unsigned long long*)&stats[8], (unsigned long long)(base + total));
                        if (base + total > o.cap) atomicAdd((unsigned long long*)&stats[7], 1ull);
                    }
                }
                lim = o.cap - base; if (lim > total) lim = total; if (lim < 0 || timed_out) lim = 0;   // moves of this tile that fit
            }
            // ---- phase B: moves [m0, mEnd) of the tile, 64 per iteration, lane <-> two consecutive list slots
            const int mEnd = (int)min((long long)m1, lim);
            int gcur = 0;
#pragma unroll 1
            for (int w0 = m0 - (int)((base + m0) & 1); w0 < mEnd; w0 += 64) {
                uint32_t blo = 0, bhi = 0;
                for (int gq = gcur + 1;; gq += 32) {        // group starts inside the window (descriptors after gcur)
                    const int idx = gq + lane;
                    const uint32_t rel = idx <= nd ? sm.arena[idx].start - (uint32_t)w0 : 64u;   // past the sentinel: none
                    blo |= rel < 32u ? 1u << rel : 0u;
                    bhi |= (rel >= 32u && rel < 64u) ? 1u << (rel - 32u) : 0u;
                    if (!__shfl_sync(FULL, (int)(rel < 64u), 31)) break;
                }
                blo = __reduce_or_sync(FULL, blo); bhi = __reduce_or_sync(FULL, bhi);
                const int x = 2 * lane;
                const uint32_t mlo = x < 31 ? (2u << x) - 1u : 0xFFFFFFFFu, mhi = x < 32 ? 0u : (2u << (x - 32)) - 1u;
                const int g0 = gcur + __popc(blo & mlo) + __popc(bhi & mhi);
                const int g1 = g0 + (int)(((x + 1 < 32) ? (blo >> (x + 1)) : (bhi >> (x - 31))) & 1u);
                const int i0 = w0 + x;
                const bool v0 = i0 >= m0 && i0 < mEnd, v1 = i0 + 1 < mEnd;
                if (v0 || v1) {
                    uint64_t mv0, mv1;
                    const flat::Desc d0 = sm.arena[g0], d1 = sm.arena[g1];
                    const int c0 = (int)(sm.arena[g0 + 1].start - d0.start), c1 = (int)(sm.arena[g1 + 1].start - d1.start);
#if DDZ_FLAT_PAIR
                    flat::decode2(d0.prm, i0 - (int)d0.start, c0, v0, d1.prm, i0 + 1 - (int)d1.start, c1, v1, s_table, sm.lists, mv0, mv1);
#else
                    mv0 = v0 ? flat::decode(d0.prm, i0 - (int)d0.start, c0, s_table, sm.lists) : 0ull;
                    mv1 = v1 ? flat::decode(d1.prm, i0 + 1 - (int)d1.start, c1, s_table, sm.lists) : 0ull;
#endif
                    uint64_t* dst = o.actions_u64 + (base + i0);          // base + i0 is even: 16-byte aligned
                    if (v0 && v1) *reinterpret_cast<ulonglong2*>(dst) = make_ulonglong2(mv0, mv1);
                    else if (v0) dst[0] = mv0;
                    else dst[1] = mv1;
                }
                gcur += __popc(blo) + __popc(bhi);
            }
            __syncwarp();                                   // the arena is consumed before the next round overwrites it
            h0 = h1;
        }
        stat_add(stats, 7, disagree);
    }
    if (lane == 0) {
        const unsigned int fin = atomicAdd(&ws.h->finished, 1u);
        if (fin == nwarps - 1) {                            // the last warp of the launch re-arms the workspace
            ws.h->ticket = 0; ws.h->finished = 0; ws.h->epoch = epoch + 1;
            __threadfence();
        }
    }
}

// face only (ddz_encode_face): same planes + LUT rows, plain coalesced stores
template <int V>
__global__ void __launch_bounds__(kEnvs) k_face(const void* state, float4* __restrict__ face, int B) {
    constexpr int C = FaceCfg<V>::C;
    __shared__ uint64_t s_planes[kEnvs * C];
    __shared__ float s_p[kEnvs * 2];
    const int tid = threadIdx.x, b0 = blockIdx.x * kEnvs, b = b0 + tid;
    if (b < B) {
        Env e = load_env(view_of(const_cast<void*>(state), B), b);
        uint64_t pl[C]; float p[2];
        face_planes<V>(e, pl, p);
#pragma unroll
        for (int c = 0; c < C; c++) s_planes[tid * C + c] = pl[c];
        s_p[tid * 2] = p[0]; s_p[tid * 2 + 1] = p[1];
    }
    __syncthreads();
    float4* dst = face + (size_t)b0 * C * 15;
    const int nvec = min(kEnvs, B - b0) * C * 15;
    for (int i = tid; i < nvec; i += kEnvs) {
        int row = i / 15, rank = i - row * 15;
        int env = row / C, c = row - env * C;
        float s = (c >= C - 2) ? s_p[env * 2 + (c - (C - 2))] : 1.f;
        const float4 q = lut_entry((int)((uint32_t)(s_planes[row] >> (4 * rank)) & 15u));
        dst[i] = make_float4(q.x * s, q.y * s, q.z * s, q.w * s);
    }
}

// The Q-network's input built in place (net.py:81-90: face repeated per action, torch.cat with the action plane): for every
// legal move i of env b, out[dst + i] = [C face rows of env b | the move's one-hot row], 240 x (C+1) bytes.  One warp per
// env: the face planes are computed once and every row goes out through the same two-rows-per-instruction writer.
template <int V>
__global__ void __launch_bounds__(128) k_state_actions(const void* state, const int32_t* __restrict__ offsets,
                                                       const uint64_t* __restrict__ actions,
                                                       const uint8_t* __restrict__ env_mask,
                                                       const int32_t* __restrict__ dst_offsets,
                                                       float4* __restrict__ out, int B) {
    constexpr int C = FaceCfg<V>::C;
    __shared__ FaceRow s_face[4][C];
    __shared__ float4 s_lut[kLutEntries];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int b = blockIdx.x * 4 + wib;
    if (threadIdx.x < kLutEntries) s_lut[threadIdx.x] = lut_entry(threadIdx.x);
    const bool live = b < B && (!env_mask || env_mask[b]);
    int src = 0, n = 0;
    if (live) { src = offsets[b]; n = offsets[b + 1] - src; }
    if (live && n > 0 && lane == 0) {
        const Env e = load_env(view_of(const_cast<void*>(state), B), b);
        uint64_t pl[C]; float p[2];
        face_planes<V>(e, pl, p);
#pragma unroll
        for (int c = 0; c < C; c++) { s_face[wib][c].packed = pl[c]; s_face[wib][c].s = (c >= C - 2) ? p[c - (C - 2)] : 1.f; s_face[wib][c].pad = 0.f; }
    }
    __syncthreads();
    if (!live || n <= 0) return;
    const RowLane rl = RowLane::make(lane);
    const long long dst = dst_offsets ? dst_offsets[b] : src;
    float4* o = out + (size_t)dst * (C + 1) * 15 + (rl.first & 1) * 15 + rl.k;
    const int nrows = n * (C + 1);
#pragma unroll 2
    for (int r = rl.first; r < nrows; r += 2, o += 30) {
        const int m = r / (C + 1), c = r - m * (C + 1);
        uint64_t packed; float sc = 1.f;
        if (c < C) { packed = s_face[wib][c].packed; sc = s_face[wib][c].s; }
        else packed = __ldg(&actions[src + m]);
        float4 q = rl.thermo(packed, s_lut);
        q.x *= sc; q.y *= sc; q.z *= sc; q.w *= sc;
        DDZ_STORE(o, q);
    }
}

// The first layer of the reference's Q-networks (net.py:65-139, NetComplicated family) for every legal move, straight from
// the packed state and the packed move lists -- the [n, C+1, 15, 4] input of net.py:90 is never built.  Every input plane is,
// per rank, four 0/1 slots that are a function of ONE nibble, and conv_k ((1,k) kernel, stride (1,4)) produces exactly one
// output per rank from slots 0..k-1, so
//     conv_k[o][r] = bias_k[o] + sum_c scale_c * T[c][nibble_c(r)][o][k]        (T built on the host: agent.q_tables)
//     x_rank[o][r] = max_k conv_k[o][r]                                          (MaxPool2d((1,4)) over the concatenation)
//     x_line[o][j] = bias[o] + sum_{c,r} scale_c * L[c][r][o] * lut[nibble_c(r)][j]      (conv_shunzi, (15,1) kernel)
// One CTA per env, thread <-> output channel o.  The C face planes are summed ONCE per env into registers (15 ranks x 4
// convolutions + 4 line slots): a plane holds at most four different non-empty nibbles, so its four table rows (scaled) go
// to the thread's own column of shared memory and its 15 line weights to registers, all loads in flight together, and the
// ranks then pick by the nibble -- which is the same for every thread, so every branch is uniform.  Each legal move then adds
// its own plane, takes the maximum and writes its row straight from registers: the row is laid out RANK-MAJOR,
// [15][W] | [W][4], so a warp's 32 channels of one rank are one 128-byte line (float32; 64 bytes in bfloat16) -- no staging, no
// barrier between moves.  (net.py:93-97 lays the same numbers out channel-major, o * 15 + r; the caller permutes fc1's
// columns once, agent.FusedQScorer.refresh.)  The tables (<= 0.7 MB) live in L1 / L2.
constexpr int kQThreads = 256;
// WC: the width as a compile-time constant (256, the reference's networks: every table offset becomes an immediate) or 0
template <int V, bool BF16, int WC>
__global__ void __launch_bounds__(kQThreads) k_q_features(const void* state, const int32_t* __restrict__ offsets,
                                                           const uint64_t* __restrict__ actions,
                                                           const uint8_t* __restrict__ env_mask,
                                                           const int32_t* __restrict__ dst_offsets, int env_begin,
                                                           long long row_base, const float4* __restrict__ T,
                                                           const float4* __restrict__ rank_bias,
                                                           const float* __restrict__ L, const float* __restrict__ line_bias,
                                                           int Wrt, void* __restrict__ out, int B) {
    constexpr int C = FaceCfg<V>::C;
    const int W = WC ? WC : Wrt;
    extern __shared__ __align__(16) float4 s_t[];            // [5][kQThreads] a plane's scaled table rows
    __shared__ uint64_t s_planes[C];
    __shared__ float s_scale[C];
    __shared__ float4 s_lut[16];
    const int b = env_begin + blockIdx.x;
    if (b >= B || (env_mask && !env_mask[b])) return;
    const int src = offsets[b], n = offsets[b + 1] - src;
    if (n <= 0) return;
    if (threadIdx.x == 0) {
        const Env e = load_env(view_of(const_cast<void*>(state), B), b);
        uint64_t pl[C]; float p[2];
        face_planes<V>(e, pl, p);
#pragma unroll
        for (int c = 0; c < C; c++) { s_planes[c] = pl[c]; s_scale[c] = (c >= C - 2) ? p[c - (C - 2)] : 1.f; }
    }
    if (threadIdx.x < 16) s_lut[threadIdx.x] = lut_entry(threadIdx.x);
    __syncthreads();
    const long long row0 = (dst_offsets ? (long long)dst_offsets[b] : (long long)src) - row_base;
    const int rowlen = 19 * W;
    const int o = threadIdx.x;                                // W <= kQThreads (the reference's networks: W = 256)
    if (o >= W) return;                                       // no barrier below: idle threads may leave
    float4 F[15];                                             // F[r] = the four convolutions' sums over the face planes
    const float4 bk = __ldg(&rank_bias[o]);
#pragma unroll
    for (int r = 0; r < 15; r++) F[r] = bk;
    const float lb = __ldg(&line_bias[o]);
    float4 S = make_float4(lb, lb, lb, lb);
#pragma unroll 1
    for (int c = 0; c < C; c++) {
        const uint64_t pl = s_planes[c];
        if ((pl & 0x0777777777777777ull) == 0) continue;      // an empty plane (a pass, an untouched history) adds nothing
        const float sc = s_scale[c];
        // (form-B builds mark the nibbles of ranks 0..12 of a probability plane with bit 3 -- rows 9..12 --, its two joker
        // ranks stay unmarked: they hold 0 or 1 and use row 1)
        const int hi = kProbForm ? ((int)((pl >> 3) & 1ull) << 3) : 0;
        const float4* Tc = T + (c * 16 + hi) * W + o;
        const float* Lc = L + c * 15 * W + o;
        const float4 t1 = __ldg(Tc + 1 * W), t2 = __ldg(Tc + 2 * W), t3 = __ldg(Tc + 3 * W), t4 = __ldg(Tc + 4 * W);
        float4 tj = t1;
        if (kProbForm && hi) tj = __ldg(T + (c * 16 + 1) * W + o);
        float lw[15];
#pragma unroll
        for (int r = 0; r < 15; r++) lw[r] = sc * __ldg(Lc + r * W);
        // the thread's own column of s_t: written and read by this thread only, indexed by the (uniform) nibble
        s_t[0 * kQThreads + o] = make_float4(sc * tj.x, sc * tj.y, sc * tj.z, sc * tj.w);
        s_t[1 * kQThreads + o] = make_float4(sc * t1.x, sc * t1.y, sc * t1.z, sc * t1.w);
        s_t[2 * kQThreads + o] = make_float4(sc * t2.x, sc * t2.y, sc * t2.z, sc * t2.w);
        s_t[3 * kQThreads + o] = make_float4(sc * t3.x, sc * t3.y, sc * t3.z, sc * t3.w);
        s_t[4 * kQThreads + o] = make_float4(sc * t4.x, sc * t4.y, sc * t4.z, sc * t4.w);
        const uint32_t plo = (uint32_t)pl, phi = (uint32_t)(pl >> 32);
#pragma unroll
        for (int r = 0; r < 15; r++) {
            const int nib = (int)(((r < 8 ? plo : phi) >> (4 * (r & 7))) & 7u);
            if (nib == 0) continue;
            const bool joker = kProbForm && r >= 13;       // row 0 of s_t: the unmarked row 1 (form-B joker ranks)
            const float4 t = s_t[(joker ? 0 : nib) * kQThreads + o];
            F[r].x += t.x; F[r].y += t.y; F[r].z += t.z; F[r].w += t.w;
            const float4 q = s_lut[(joker ? 0 : hi) + nib];
            S.x = fmaf(lw[r], q.x, S.x); S.y = fmaf(lw[r], q.y, S.y); S.z = fmaf(lw[r], q.z, S.z); S.w = fmaf(lw[r], q.w, S.w);
        }
    }
    const float4* TA = T + C * 16 * W + o;                    // the move's own plane is input channel C
    const float* LA = L + C * 15 * W + o;
#pragma unroll 1
    for (int a = 0; a < n; a++) {
        const uint64_t mv = __ldg(&actions[src + a]);
        const uint32_t mlo = (uint32_t)mv, mhi = (uint32_t)(mv >> 32);
        float4 s = S;
        float* const row32 = reinterpret_cast<float*>(out) + (size_t)(row0 + a) * rowlen + o;
        __nv_bfloat16* const row16 = reinterpret_cast<__nv_bfloat16*>(out) + (size_t)(row0 + a) * rowlen + o;
#pragma unroll
        for (int r = 0; r < 15; r++) {
            const int nib = (int)(((r < 8 ? mlo : mhi) >> (4 * (r & 7))) & 15u);      // uniform over the CTA
            float m;
            if (nib) {
                const float4 t = __ldg(TA + nib * W);
                m = fmaxf(fmaxf(F[r].x + t.x, F[r].y + t.y), fmaxf(F[r].z + t.z, F[r].w + t.w));
                const float lw = __ldg(LA + r * W);
                const float4 q = s_lut[nib];
                s.x = fmaf(lw, q.x, s.x); s.y = fmaf(lw, q.y, s.y); s.z = fmaf(lw, q.z, s.z); s.w = fmaf(lw, q.w, s.w);
            } else m = fmaxf(fmaxf(F[r].x, F[r].y), fmaxf(F[r].z, F[r].w));
            if (BF16) row16[r * W] = __float2bfloat16_rn(m); else row32[r * W] = m;
        }
        if (BF16) {
            __nv_bfloat162 lo2 = __floats2bfloat162_rn(s.x, s.y), hi2 = __floats2bfloat162_rn(s.z, s.w);
            uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo2); pk.y = *reinterpret_cast<uint32_t*>(&hi2);
            *reinterpret_cast<uint2*>(row16 - o + 15 * W + 4 * o) = pk;
        } else *reinterpret_cast<float4*>(row32 - o + 15 * W + 4 * o) = s;
    }
}

// the thermometer one-hot of rank `rank` of a packed move (envi.py:140-146, batch_arr2onehot)
DDZ_DEV float4 move_thermo(uint64_t move, int rank) {
    const uint32_t c = (uint32_t)(move >> (4 * rank)) & 15u;
    return make_float4(c > 0 ? 1.f : 0.f, c > 1 ? 1.f : 0.f, c > 2 ? 1.f : 0.f, c > 3 ? 1.f : 0.f);
}

__global__ void __launch_bounds__(256) k_encode_actions(const uint64_t* __restrict__ actions, long long n,
                                                        float4* __restrict__ out) {
    long long nvec = n * 15;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
        long long row = i / 15; int rank = (int)(i - row * 15);
        out[i] = move_thermo(actions[row], rank);
    }
}

// Replay decode (ddz_encode_face_gather): k_face over env rows[i] of a stored state, plus the one-hot row of that env's
// packed move.  CONCAT: face [n][C+1] rows with the move row last (k_state_actions' rows); else face [n][C] rows and, when
// move_rows != NULL, move_rows [n].  A row outside [0, B) reads nothing and gives zero rows.
template <int V, bool CONCAT>
__global__ void __launch_bounds__(kEnvs) k_face_gather(const void* state, const int64_t* __restrict__ rows, long long n,
                                                       const uint64_t* __restrict__ moves, float4* __restrict__ face,
                                                       float4* __restrict__ move_rows, int B) {
    constexpr int C = FaceCfg<V>::C, R = CONCAT ? C + 1 : C;   // R: rows per sample in `face`
    __shared__ uint64_t s_planes[kEnvs * (C + 1)];              // the C face planes, then the move
    __shared__ float s_p[kEnvs * 2];
    const int tid = threadIdx.x;
    const long long i0 = (long long)blockIdx.x * kEnvs;
    if (i0 + tid < n) {
        const long long b = rows[i0 + tid];
        uint64_t pl[C], mv = 0; float p[2] = {0.f, 0.f};
        if (b >= 0 && b < B) {
            const Env e = load_env(view_of(const_cast<void*>(state), B), (int)b);
            face_planes<V>(e, pl, p);
            if (moves) mv = moves[b];
        } else {
#pragma unroll
            for (int c = 0; c < C; c++) pl[c] = 0;
        }
#pragma unroll
        for (int c = 0; c < C; c++) s_planes[tid * (C + 1) + c] = pl[c];
        s_planes[tid * (C + 1) + C] = mv;
        s_p[tid * 2] = p[0]; s_p[tid * 2 + 1] = p[1];
    }
    __syncthreads();
    const int ns = (int)min((long long)kEnvs, n - i0);
    float4* dst = face + (size_t)i0 * R * 15;
    const int nvec = ns * R * 15;
    for (int i = tid; i < nvec; i += kEnvs) {
        const int row = i / 15, rank = i - row * 15;
        const int smp = row / R, c = row - smp * R;
        if (CONCAT && c == C) { dst[i] = move_thermo(s_planes[smp * (C + 1) + C], rank); continue; }
        const float s = (c >= C - 2) ? s_p[smp * 2 + (c - (C - 2))] : 1.f;
        const float4 q = lut_entry((int)((uint32_t)(s_planes[smp * (C + 1) + c] >> (4 * rank)) & 15u));
        dst[i] = make_float4(q.x * s, q.y * s, q.z * s, q.w * s);
    }
    if (!CONCAT && move_rows) {
        float4* mdst = move_rows + (size_t)i0 * 15;
        for (int i = tid; i < ns * 15; i += kEnvs) {
            const int smp = i / 15, rank = i - smp * 15;
            mdst[i] = move_thermo(s_planes[smp * (C + 1) + C], rank);
        }
    }
}

// number of legal moves of the player to move in every env, closed form (no list): one thread per env
__global__ void __launch_bounds__(256) k_legal_count(const void* state, int32_t* __restrict__ counts, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const Env e = load_env(view_of(const_cast<void*>(state), B), b);
    int n = 0;
    if (!e.done()) {
        const uint64_t hand = hand_to_move(e), last = trick_of(e);
        n = count_legal(masks_of(hand), rule_of(last), last != 0);
    }
    counts[b] = n;
}

// idx-th legal move of n independent (hand, last) pairs in closed form (no list): the building block of the playout
__global__ void __launch_bounds__(256) k_kth_moves(const uint64_t* __restrict__ hands, const uint64_t* __restrict__ lasts,
                                                   const int32_t* __restrict__ idx, uint64_t* __restrict__ moves,
                                                   int32_t* __restrict__ counts, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t hand = hands[i], last = lasts[i];
    const Masks m = masks_of(hand);
    const Rule ru = rule_of(last);
    const int c = count_legal(m, ru, last != 0);
    if (counts) counts[i] = c;
    const int k = idx[i];
    moves[i] = (k >= 0 && k < c) ? select_legal(m, ru, last != 0, k) : ~0ull;
}

// Random playout (the default policy of the reference's MCTS, server/mcts/default_policy.py:4-10: "play random legal
// moves until the game ends"): every lane plays ITS env forward for up to max_steps decisions, move number
// philox(seed, env, stepno0 + t) % N of the canonical list each time -- the same stream the stepping API uses, so a
// playout equals max_steps calls of ddz_rollout_step without re-deal.  No lists, no features, no inter-env traffic:
// the state stays in registers, one load and one store per env.
// PRUNED: the default policy the reference's search bot really plays -- a uniform draw from ITS move list, the pruned one
// of server/mcts/get_moves.py:36-69 (tree.py:83-91 calls it for every playout move): the draw picks an entry of the pruned
// list, search::pruned_pick finds which move of the full list that is.  The keys of one decision live in local memory.
struct KeySink {
    uint16_t* keys; int n, handnum;
    DDZ_DEV void operator()(uint64_t mv) { if (n < DDZ_MAX_LEGAL) keys[n] = (uint16_t)search::value_key(mv, handnum); n++; }
};
// one lane's playout of env e (Philox stream `env`, decisions stepno0, stepno0 + 1, ...): the body of k_playout, also
// the default policy of k_uct
template <bool PRUNED>
DDZ_DEV void playout_env(Env& e, int max_steps, uint64_t seed, uint64_t env, uint32_t stepno0, const int32_t* rewards,
                         int& steps, int& passes, int& over, int& winner) {
    for (int t = 0; t < max_steps && !e.done(); t++) {
        const uint64_t hand = hand_to_move(e), last = trick_of(e);
        const Masks m = masks_of(hand);
        const Rule ru = rule_of(last);
        const int n = count_legal(m, ru, last != 0);
        if (n <= 0) break;
        const uint32_t u = philox(seed, env, stepno0 + (uint32_t)t);
        int k;
        if (PRUNED && n > search::kPruneAbove) {
            uint16_t keys[DDZ_MAX_LEGAL];
            KeySink ks{keys, 0, card_count(hand)};
            enumerate_legal(m, ru, last != 0, ks);
            const int nk = min(n, DDZ_MAX_LEGAL);            // 512 bounds every list of hands dealt from one deck
            k = search::pruned_pick(keys, nk, (int)(u % (uint32_t)search::pruned_size(nk)));
        } else k = (int)(u % (uint32_t)n);
        const StepOut so = apply_move(e, select_legal(m, ru, last != 0, k), rewards);
        steps++; passes += so.pass;
        if (so.done) { over = 1; winner = so.winner; }
    }
}
template <bool PRUNED>
__global__ void __launch_bounds__(128) k_playout(void* state, int max_steps, uint64_t seed, uint64_t env0, uint32_t stepno0,
                                                 int32_t rw0, int32_t rw1, int32_t rw2, int32_t* __restrict__ steps_taken,
                                                 int64_t* stats, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int32_t rewards[3] = {rw0, rw1, rw2};
    int steps = 0, passes = 0, over = 0, winner = 0;
    if (b < B) {
        const StateView v = view_of(state, B);
        Env e = load_env(v, b);
        playout_env<PRUNED>(e, max_steps, seed, env0 + (uint64_t)b, stepno0, rewards, steps, passes, over, winner);
        store_env(v, b, e);
        if (steps_taken) steps_taken[b] = steps;
    }
    stat_add(stats, 4, steps); stat_add(stats, 9, passes); stat_add(stats, 0, over);
    stat_add(stats, 1, over && winner == 1); stat_add(stats, 2, over && winner == 2); stat_add(stats, 3, over && winner == 0);
    stat_add(stats, 5, over ? (winner == 1 ? rw1 : -rw1) : 0);
    stat_add(stats, 6, over ? (winner == 1 ? -(rw0 + rw2) : rw0 + rw2) : 0);
}

// mcts.get_moves.get_moves for n independent (hand, last) pairs (server/mcts/get_moves.py:36-69), one warp per pair: the
// full list is expanded into shared memory by the whole warp, every kept move gets its position in the stable ascending
// order of the keys by counting (no sort: position = how many kept moves come before it), and goes to the slots of the
// pruned list that position owns -- entry 2k for the k-th lowest, entry 2k+1 for the k-th highest.
constexpr int kSearchWarps = 4;
struct SlotEmitter {
    uint64_t* out;
    DDZ_DEV void operator()(int idx, uint64_t mv) { if ((unsigned)idx < (unsigned)DDZ_MAX_LEGAL) out[idx] = mv; }
};
// The whole warp builds the pruned list of (hand, last) into dst[0 .. returned count): the full canonical list goes to
// moves[0 .. nfull) and the keys to keys[] (per-warp scratch, DDZ_MAX_LEGAL entries each).  Shared by k_mcts_moves and k_uct.
DDZ_DEV int warp_mcts_list(uint64_t hand, uint64_t last, uint64_t* moves, uint16_t* keys, uint64_t* dst, int lane, int& nfull) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const Masks hm = masks_of(hand);
    const Rule ru = rule_of(last);
    SlotEmitter em{moves};
    const int n = min(enumerate_legal_warp(hm, ru, last != 0, lane, em), DDZ_MAX_LEGAL);   // 512 bounds every real list
    nfull = n;
    __syncwarp();
    int count = n;
    if (n <= search::kPruneAbove) {
        for (int i = lane; i < n; i += 32) dst[i] = moves[i];
    } else {
        const int handnum = card_count(hand);
        int kept = 0;
        for (int i = lane; i < n; i += 32) {
            const uint32_t key = search::value_key(moves[i], handnum);
            keys[i] = (uint16_t)key;
            kept += key != search::kDropped;
        }
        const int m = __reduce_add_sync(FULL, kept);
        __syncwarp();
        const int rounds = n / 3 + 1;
        count = 2 * rounds;
        for (int i = lane; i < n; i += 32) {
            const uint32_t key = keys[i];
            if (key == search::kDropped) continue;
            int pos = 0;
            for (int j = 0; j < n; j++) { const uint32_t kj = keys[j]; pos += (kj < key) | ((kj == key) & (j < i)); }
            const uint64_t mv = moves[i];
            const int top = m - 1 - pos;
            if (pos < rounds) dst[2 * pos] = mv;
            if (top < rounds) dst[2 * top + 1] = mv;
            if (pos == m - 1) for (int k = m; k < rounds; k++) dst[2 * k] = mv;       // clamped positions (never for one deck)
            if (pos == 0) for (int k = m; k < rounds; k++) dst[2 * k + 1] = mv;
        }
    }
    return count;
}
__global__ void __launch_bounds__(kSearchWarps * 32) k_mcts_moves(const uint64_t* __restrict__ hands,
                                                                  const uint64_t* __restrict__ lasts,
                                                                  uint64_t* __restrict__ out, int32_t* __restrict__ counts,
                                                                  int npairs) {
    __shared__ uint64_t s_moves[kSearchWarps][DDZ_MAX_LEGAL];
    __shared__ uint16_t s_keys[kSearchWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int pair = blockIdx.x * kSearchWarps + wib;
    if (pair >= npairs) return;
    int nfull;
    const int count = warp_mcts_list(hands[pair], lasts[pair], s_moves[wib], s_keys[wib],
                                     out + (size_t)pair * DDZ_MCTS_MAX_MOVES, lane, nfull);
    if (lane == 0) counts[pair] = count;
}

// ------------------------------------------------------------------------------------------------
// Batched UCT search (the reference's search bot, server/mcts/interface.py:37-45, for B positions in ONE launch):
// one warp per root, all `budget` iterations of  tree policy -> default policy -> back-up  inside the kernel.  The tree
// lives in the caller's workspace (UctNode, layout in ddz_b200.h); a node's children are the nodes whose parent it is, in
// node order = expansion order, all within [first_child, last_child].  A node's entries (its move list) are recomputed
// when one of them is expanded: the full canonical list (select_legal, closed form), or the bot's pruned list built by the
// warp (warp_mcts_list) when it has more than 10 moves.  Playouts are spread over the lanes (playout_env).
// Draws: the j-th tree draw of root b is philox(seed, env0 + b, 0x80000000 + j); playout w of iteration it draws from
// the stream ((env0 + b) * budget + it) * width + w at steps 0, 1, ...
// ------------------------------------------------------------------------------------------------
struct UctNode {
    uint32_t untried[16];       // bit j: entry j of the node's list is not expanded yet
    uint64_t hand[3], recent[3];
    uint64_t move;              // the move that led here (root: 0)
    int32_t parent, first_child, last_child, nchild;   // root: parent -1; no child: first = last = -1
    int32_t visits, wins;
    int16_t nentries, remaining;
    int16_t index;              // index of `move` in the parent's canonical legal list (root: -1)
    int8_t cur, winner;         // role to move; role that emptied its hand with `move`, or -1
    int32_t pad[2];
};
static_assert(sizeof(UctNode) == DDZ_UCT_NODE_BYTES, "UctNode layout is documented in ddz_b200.h");
constexpr int kUctWarps = 4;
constexpr int kUctPlayoutSteps = 512;   // a game ends within 3 x 54 decisions
__host__ __device__ inline size_t uct_header_bytes(int B) { return ((size_t)B * 4 + 255) / 256 * 256; }

struct UctArgs {
    const void* state; const uint8_t* mask; char* ws; const double* ln;
    int budget, width, prune; double c; uint64_t seed, env0;
    int32_t* choice; uint64_t* move; int32_t* root_n; uint64_t* root_moves; int32_t* root_visits; int32_t* root_wins;
    int root_stride, B;
};

// entries of the list of the player to move: the canonical list, or its pruned form (same length rule as ddz_mcts_moves)
DDZ_DEV int uct_entries(uint64_t hand, uint64_t last, int prune) {
    const int n = count_legal(masks_of(hand), rule_of(last), last != 0);
    return prune ? search::pruned_size(min(n, DDZ_MAX_LEGAL)) : n;
}
DDZ_DEV uint64_t uct_trick(const uint64_t* recent, int cur) {
    return last_move(recent[(cur + 2) % 3], recent[(cur + 1) % 3]);
}
// node `id` with the given position; lane 0 writes the scalars, lanes 0..15 the untried bits
DDZ_DEV void uct_init(UctNode* T, int id, const uint64_t* hand, const uint64_t* recent, int cur, int winner, uint64_t move,
                      int parent, int index, int prune, int lane) {
    UctNode& X = T[id];
    const int ne = winner >= 0 ? 0 : uct_entries(hand[cur], uct_trick(recent, cur), prune);
    if (lane < 16) {
        const int lo = 32 * lane;
        X.untried[lane] = ne >= lo + 32 ? 0xFFFFFFFFu : (ne > lo ? (1u << (ne - lo)) - 1u : 0u);
    }
    if (lane == 0) {
        for (int q = 0; q < 3; q++) { X.hand[q] = hand[q]; X.recent[q] = recent[q]; }
        X.move = move; X.parent = parent; X.first_child = X.last_child = -1; X.nchild = 0;
        X.visits = X.wins = 0; X.nentries = (int16_t)ne; X.remaining = (int16_t)ne; X.index = (int16_t)index;
        X.cur = (int8_t)cur; X.winner = (int8_t)winner; X.pad[0] = X.pad[1] = 0;
    }
}
// UCB1 of a child, in double with correctly rounded operations and no contraction: the CPU port (Python's float, C with
// -ffp-contract=off) computes the same bits, so both order every pair of children identically, near-ties included.
// ln_n comes from a host table (C library log), because the device log is not correctly rounded.
DDZ_DEV double uct_value(int wins, int visits, double c, double ln_n) {
    const double v = (double)visits;
    return __dadd_rn(__ddiv_rn((double)wins, v), __dmul_rn(c, __dsqrt_rn(__ddiv_rn(__dmul_rn(2.0, ln_n), v))));
}
// The child of x with the maximum (want_max) or minimum value, a uniformly drawn one of them among exact ties (in
// expansion order); final = the answer's rule: wins / visits, maximum.  Lane-parallel over the child range.
DDZ_DEV int uct_best_child(const UctNode* T, int x, bool want_max, bool final, double c, double ln_n, uint64_t seed,
                           uint64_t env, uint32_t& j, int lane) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const int f = T[x].first_child, l = T[x].last_child;
    double best = want_max ? -CUDART_INF : CUDART_INF;
    for (int k = f + lane; k <= l; k += 32) {
        if (T[k].parent != x) continue;
        const double v = final ? __ddiv_rn((double)T[k].wins, (double)T[k].visits) : uct_value(T[k].wins, T[k].visits, c, ln_n);
        best = want_max ? fmax(best, v) : fmin(best, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double w = __shfl_xor_sync(FULL, best, o);
        best = want_max ? fmax(best, w) : fmin(best, w);
    }
    int tied = 0;
    for (int base = f; base <= l; base += 32) {
        const int k = base + lane;
        bool t = false;
        if (k <= l && T[k].parent == x)
            t = (final ? __ddiv_rn((double)T[k].wins, (double)T[k].visits) : uct_value(T[k].wins, T[k].visits, c, ln_n)) == best;
        tied += __popc(__ballot_sync(FULL, t));
    }
    int r = 0;
    if (tied >= 2) r = (int)(philox(seed, env, 0x80000000u + j++) % (uint32_t)tied);
    for (int base = f; base <= l; base += 32) {
        const int k = base + lane;
        bool t = false;
        if (k <= l && T[k].parent == x)
            t = (final ? __ddiv_rn((double)T[k].wins, (double)T[k].visits) : uct_value(T[k].wins, T[k].visits, c, ln_n)) == best;
        const unsigned bal = __ballot_sync(FULL, t);
        if (r < __popc(bal)) return base + __fns(bal, 0, r + 1);
        r -= __popc(bal);
    }
    return -1;   // not reached: x has at least one child
}

// One playout played by the whole warp, for width 1 with pruned lists (otherwise one lane plays while 31 wait): every lane
// holds the same env, and a decision over a list of more than 10 moves takes entry u % count of the pruned list the warp
// builds with warp_mcts_list -- the move k_playout<true>'s single lane finds with pruned_pick.  Returns the winner (-1: not
// finished within kUctPlayoutSteps, which a game cannot reach).  Measured against the lane version in DESIGN.md 4; build
// with -DDDZ_UCT_LANE_PLAYOUT for that version.
DDZ_DEV int uct_warp_playout(Env e, uint64_t seed, uint64_t stream, uint64_t* moves, uint16_t* keys, uint64_t* list, int lane) {
    const int32_t zero_rewards[3] = {0, 0, 0};
    for (int t = 0; t < kUctPlayoutSteps && !e.done(); t++) {
        const uint64_t hand = hand_to_move(e), last = trick_of(e);
        const Masks m = masks_of(hand);
        const Rule ru = rule_of(last);
        const int n = count_legal(m, ru, last != 0);
        if (n <= 0) break;
        const uint32_t u = philox(seed, stream, (uint32_t)t);
        uint64_t mv;
        if (n > search::kPruneAbove) {
            int nfull;
            const int count = warp_mcts_list(hand, last, moves, keys, list, lane, nfull);
            __syncwarp();
            mv = list[u % (uint32_t)count];
            __syncwarp();                         // every lane has read the list before the next decision rebuilds it
        } else mv = select_legal(m, ru, last != 0, (int)(u % (uint32_t)n));
        const StepOut so = apply_move(e, mv, zero_rewards);
        if (so.done) return so.winner;
    }
    return -1;
}

__global__ void __launch_bounds__(kUctWarps * 32) k_uct(UctArgs a) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    __shared__ uint64_t s_moves[kUctWarps][DDZ_MAX_LEGAL];
    __shared__ uint16_t s_keys[kUctWarps][DDZ_MAX_LEGAL];
    __shared__ uint64_t s_list[kUctWarps][DDZ_MCTS_MAX_MOVES];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int b = blockIdx.x * kUctWarps + wib;
    if (b >= a.B) return;
    int32_t* nnodes = (int32_t*)a.ws + b;
    UctNode* T = (UctNode*)(a.ws + uct_header_bytes(a.B)) + (size_t)b * (size_t)(a.budget + 1);
    const Env e = load_env(view_of(const_cast<void*>(a.state), a.B), b);
    const bool live = !(a.mask && !a.mask[b]) && !e.done() &&
                      uct_entries(hand_to_move(e), trick_of(e), a.prune) > 0;
    if (!live) {                                  // masked out, finished, or nothing to play: sentinels, no draws
        if (lane == 0) {
            a.choice[b] = -1;
            if (a.move) a.move[b] = ~0ull;
            if (a.root_n) a.root_n[b] = 0;
            *nnodes = 0;
        }
        return;
    }
    const int me = e.cur();
    const uint64_t env = a.env0 + (uint64_t)b;
    const int32_t zero_rewards[3] = {0, 0, 0};
    uint32_t j = 0;                               // tree draws taken so far
    int nn = 1;
    uct_init(T, 0, e.hand, e.recent, me, -1, 0ull, -1, -1, a.prune, lane);
    __syncwarp();
    for (int it = 0; it < a.budget; it++) {
        // tree policy
        int x = 0;
        while (T[x].winner < 0) {
            const UctNode& X = T[x];
            const int remaining = X.remaining;
            if (remaining > 0) {                  // expand the i-th remaining entry (list.pop(i)) and stop
                const int i = (int)(philox(a.seed, env, 0x80000000u + j++) % (uint32_t)remaining);
                const uint32_t w = lane < 16 ? X.untried[lane] : 0u;
                const int pc = __popc(w);
                int incl = pc;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
                const bool mine = i >= incl - pc && i < incl;
                const int wl = __ffs(__ballot_sync(FULL, mine)) - 1;
                const int bit = mine ? (int)__fns(w, 0, i - (incl - pc) + 1) : 0;
                const int entry = __shfl_sync(FULL, wl * 32 + bit, wl);
                const int cur = X.cur;
                uint64_t hand[3] = {X.hand[0], X.hand[1], X.hand[2]}, recent[3] = {X.recent[0], X.recent[1], X.recent[2]};
                const uint64_t h = hand[cur], last = uct_trick(recent, cur);
                const Masks m = masks_of(h);
                const Rule ru = rule_of(last);
                const int n = count_legal(m, ru, last != 0);
                uint64_t mv;
                int index;
                if (a.prune && n > search::kPruneAbove) {
                    int nfull;
                    warp_mcts_list(h, last, s_moves[wib], s_keys[wib], s_list[wib], lane, nfull);
                    __syncwarp();
                    mv = s_list[wib][entry];
                    int idx = DDZ_MAX_LEGAL;
                    for (int k = lane; k < nfull; k += 32) if (s_moves[wib][k] == mv) idx = min(idx, k);
                    index = __reduce_min_sync(FULL, idx);
                    __syncwarp();
                } else {
                    mv = select_legal(m, ru, last != 0, entry);
                    index = entry;
                }
                __syncwarp();                     // every lane has read X before it changes
                if (lane == wl) T[x].untried[lane] = w & ~(1u << bit);
                if (lane == 0) {
                    T[x].remaining = (int16_t)(remaining - 1);
                    if (T[x].first_child < 0) T[x].first_child = nn;
                    T[x].last_child = nn;
                    T[x].nchild += 1;
                }
                hand[cur] -= mv;
                recent[cur] = mv;
                const int winner = (mv != 0 && hand[cur] == 0) ? cur : -1;
                uct_init(T, nn, hand, recent, (cur + 1) % 3, winner, mv, x, index, a.prune, lane);
                __syncwarp();
                x = nn++;
                break;
            }
            x = uct_best_child(T, x, X.cur == me, false, a.c, a.ln[X.visits], a.seed, env, j, lane);
        }
        // default policy
        int reward;
        const UctNode& L = T[x];
        if (L.winner >= 0) {
            reward = ((L.winner == 1) == (me == 1)) ? a.width : 0;
        }
#ifndef DDZ_UCT_LANE_PLAYOUT
        else if (a.prune && a.width == 1) {
            Env pe;
            for (int q = 0; q < 3; q++) { pe.hand[q] = L.hand[q]; pe.hist[q] = 0; pe.recent[q] = L.recent[q]; }
            pe.meta = (uint32_t)L.cur;
            const uint64_t stream = (a.env0 + (uint64_t)b) * (uint64_t)a.budget + (uint64_t)it;
            const int winner = uct_warp_playout(pe, a.seed, stream, s_moves[wib], s_keys[wib], s_list[wib], lane);
            reward = (winner >= 0 && ((winner == 1) == (me == 1))) ? 1 : 0;
        }
#endif
        else {
            int won = 0;
            for (int w = lane; w < a.width; w += 32) {
                Env pe;
                for (int q = 0; q < 3; q++) { pe.hand[q] = L.hand[q]; pe.hist[q] = 0; pe.recent[q] = L.recent[q]; }
                pe.meta = (uint32_t)L.cur;
                int steps = 0, passes = 0, over = 0, winner = 0;
                const uint64_t stream = ((a.env0 + (uint64_t)b) * (uint64_t)a.budget + (uint64_t)it) * (uint64_t)a.width + (uint64_t)w;
                if (a.prune) playout_env<true>(pe, kUctPlayoutSteps, a.seed, stream, 0, zero_rewards, steps, passes, over, winner);
                else playout_env<false>(pe, kUctPlayoutSteps, a.seed, stream, 0, zero_rewards, steps, passes, over, winner);
                won += (over && ((winner == 1) == (me == 1))) ? 1 : 0;
            }
            reward = __reduce_add_sync(FULL, won);
        }
        // back-up
        __syncwarp();
        if (lane == 0)
            for (int y = x; y >= 0; y = T[y].parent) { T[y].visits += a.width; T[y].wins += reward; }
        __syncwarp();
    }
    // answer: the root child with the best wins / visits; the root's children are nodes 1 .. nchild (the first
    // iterations expand the root until it is full)
    const int best = uct_best_child(T, 0, true, true, 0.0, 0.0, a.seed, env, j, lane);
    const int nroot = T[0].nchild;
    if (a.root_n) {
        for (int k = lane; k < min(nroot, a.root_stride); k += 32) {
            const size_t o = (size_t)b * (size_t)a.root_stride + (size_t)k;
            a.root_moves[o] = T[1 + k].move; a.root_visits[o] = T[1 + k].visits; a.root_wins[o] = T[1 + k].wins;
        }
    }
    if (lane == 0) {
        a.choice[b] = T[best].index;
        if (a.move) a.move[b] = T[best].move;
        if (a.root_n) a.root_n[b] = nroot;
        *nnodes = nn;
    }
}

// ------------------------------------------------------------------------------------------------
// Determinized search (PIMC): D full-information deals per root that agree with what the player to move has seen, searched
// by k_uct as B * D trees, their root statistics added up per canonical list index (the root list depends only on the
// mover's hand and the trick, so it is the same list in every determinization).
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kDeterminizeStep = 0xC0000000u;   // Philox step of draw 0; k_uct's tree draws start at 0x80000000
constexpr int kPoolWarps = 4;

// One thread per output env i = b * D + d.  Unseen cards = deck - hand[m] - hist[0..2], walked in rank order; card j goes
// to role a = (m+1)%3 with probability ra / (ra + rc) of the slots still open (selection sampling), else to c = (m+2)%3.
__global__ void __launch_bounds__(256) k_determinize(const void* state, const uint8_t* __restrict__ mask, int D, uint64_t seed,
                                                     uint64_t env0, void* out, int64_t* __restrict__ stats, int B) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)B * D) return;
    const int b = (int)(i / D), d = (int)(i % D);
    Env e = load_env(view_of(const_cast<void*>(state), B), b);
    if (!(mask && !mask[b]) && !e.done()) {
        const int m = e.cur(), a = (m + 1) % 3, c = (m + 2) % 3;
        const uint64_t own = pick3(m, e.hand[0], e.hand[1], e.hand[2]);
        const uint64_t ha = pick3(a, e.hand[0], e.hand[1], e.hand[2]), hc = pick3(c, e.hand[0], e.hand[1], e.hand[2]);
        int ra = card_count(ha), rc = card_count(hc), unseen = 0;
        bool bad = false;
        uint64_t un = 0;
        for (int r = 0; r < 15; r++) {
            const int u = (r < 13 ? 4 : 1) - (int)((own >> (4 * r)) & 15) - (int)((e.hist[0] >> (4 * r)) & 15) -
                          (int)((e.hist[1] >> (4 * r)) & 15) - (int)((e.hist[2] >> (4 * r)) & 15);
            bad |= u < 0;
            unseen += u;
            if (u > 0) un |= (uint64_t)u << (4 * r);
        }
        if (bad || unseen != ra + rc) {           // no deal agrees with this view: finished with a sticky error
            e.meta |= 4u | 32u;
            if (d == 0 && stats) atomicAdd((unsigned long long*)&stats[7], 1ull);
        } else {
            const uint64_t ctr = (env0 + (uint64_t)b) * (uint64_t)D + (uint64_t)d;
            uint64_t na = 0, nc = 0;
            uint32_t j = 0;
            for (int r = 0; r < 15; r++)
                for (int k = (int)((un >> (4 * r)) & 15); k > 0; k--) {
                    const uint32_t u = philox(seed, ctr, kDeterminizeStep + j++);
                    if ((int)(u % (uint32_t)(ra + rc)) < ra) { na += 1ull << (4 * r); ra--; }
                    else { nc += 1ull << (4 * r); rc--; }
                }
#pragma unroll
            for (int q = 0; q < 3; q++) e.hand[q] = q == a ? na : (q == c ? nc : e.hand[q]);
        }
    }
    store_env(view_of(out, B * D), (int)i, e);
}

// One warp per root b: the root children of trees b * D .. b * D + D - 1 (nodes first_child .. last_child whose parent is
// 0) add their visits and wins into shared counters keyed by canonical index; then the index with the best pooled
// wins / visits (exact 64-bit cross products, lowest index on ties).
__global__ void __launch_bounds__(kPoolWarps * 32) k_uct_pool(const char* __restrict__ ws, int budget, int D, int32_t* choice,
                                                              uint64_t* move, int32_t* pooled_visits, int32_t* pooled_wins, int B) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    __shared__ int32_t s_v[kPoolWarps][DDZ_MAX_LEGAL], s_w[kPoolWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int b = blockIdx.x * kPoolWarps + wib;
    if (b >= B) return;
    const int ntrees = B * D;
    const int32_t* nnodes = (const int32_t*)ws;
    const UctNode* base = (const UctNode*)(ws + uct_header_bytes(ntrees));
    for (int k = lane; k < DDZ_MAX_LEGAL; k += 32) { s_v[wib][k] = 0; s_w[wib][k] = 0; }
    __syncwarp();
    int root = -1;                                // the first tree of b that was searched
    for (int d = 0; d < D; d++) {
        const int t = b * D + d;
        if (nnodes[t] <= 0) continue;
        if (root < 0) root = t;
        const UctNode* T = base + (size_t)t * (size_t)(budget + 1);
        const int f = T[0].first_child, l = T[0].last_child;
        for (int k = f + lane; k >= 0 && k <= l; k += 32) {
            if (T[k].parent != 0) continue;
            const int idx = T[k].index;
            if ((unsigned)idx >= (unsigned)DDZ_MAX_LEGAL) continue;
            atomicAdd(&s_v[wib][idx], T[k].visits);
            atomicAdd(&s_w[wib][idx], T[k].wins);
        }
    }
    __syncwarp();
    int bi = -1;
    long long bv = 0, bw = 0;
    for (int k = lane; k < DDZ_MAX_LEGAL; k += 32) {
        const long long v = s_v[wib][k], w = s_w[wib][k];
        if (pooled_visits) pooled_visits[(size_t)b * DDZ_MAX_LEGAL + k] = (int32_t)v;
        if (pooled_wins) pooled_wins[(size_t)b * DDZ_MAX_LEGAL + k] = (int32_t)w;
        if (v > 0 && (bi < 0 || w * bv > bw * v)) { bi = k; bv = v; bw = w; }   // ascending k: ties keep the lower index
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const int oi = __shfl_xor_sync(FULL, bi, o);
        const long long ov = __shfl_xor_sync(FULL, bv, o), ow = __shfl_xor_sync(FULL, bw, o);
        if (oi >= 0 && (bi < 0 || ow * bv > bw * ov || (ow * bv == bw * ov && oi < bi))) { bi = oi; bv = ov; bw = ow; }
    }
    if (lane == 0) {
        uint64_t mv = ~0ull;
        if (root >= 0 && bi >= 0) {
            const UctNode& R = base[(size_t)root * (size_t)(budget + 1)];
            const uint64_t last = uct_trick(R.recent, R.cur);
            mv = select_legal(masks_of(R.hand[R.cur]), rule_of(last), last != 0, bi);
        }
        choice[b] = root >= 0 ? bi : -1;
        if (move) move[b] = root >= 0 ? mv : ~0ull;
    }
}

// Batched dqn.py:50-71: per env, the index of the best-scoring legal move (first maximum or first NaN, like torch.argmax), or with
// probability epsilon a uniformly random one (e_greedy_action).  One lane per env; segments are short (mean 5.6).
__global__ void __launch_bounds__(256) k_select_actions(const float* __restrict__ q, const int32_t* __restrict__ offsets,
                                                        float epsilon, uint64_t seed, uint64_t env0, uint32_t stepno,
                                                        int32_t* __restrict__ choice, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int lo = offsets[b], n = offsets[b + 1] - lo;
    int best = -1;
    if (n > 0) {
        bool explore = false;
        if (epsilon > 0.f) {
            // two independent Philox draws: counter word 3 distinguishes them from the env's move stream
            const uint32_t u = philox(seed ^ 0x9E3779B97F4A7C15ull, env0 + (uint64_t)b, stepno);
            explore = (float)(u >> 8) * (1.0f / 16777216.0f) < epsilon;
            if (explore) best = (int)(philox(seed ^ 0xD1B54A32D192ED03ull, env0 + (uint64_t)b, stepno) % (uint32_t)n);
        }
        if (!explore) {
            float bv = q[lo]; best = 0;
            // the first NaN wins, as in torch.argmax: a NaN beats every number, and nothing beats a NaN
            for (int i = 1; i < n; i++) { const float v = q[lo + i]; if (v > bv || (v != v && bv == bv)) { bv = v; best = i; } }
        }
    }
    choice[b] = best;
}

// Action ids (ddz_ids.cuh), one thread per element.
__global__ void __launch_bounds__(256) k_move_ids(const uint64_t* __restrict__ moves, long long n, int32_t* __restrict__ ids) {
    for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (long long)gridDim.x * 256) ids[i] = move_id(moves[i]);
}
__global__ void __launch_bounds__(256) k_moves_of_ids(const int32_t* __restrict__ ids, long long n, uint64_t* __restrict__ moves) {
    for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (long long)gridDim.x * 256) moves[i] = move_of_id(ids[i]);
}

// Legal-id mask rows, one warp per env.  The warp turns the env's stored list into ids in shared memory (they strictly
// increase), then every lane writes 16-byte pieces lane, lane + 32, ... of the row (coalesced), finding the ids of each piece
// by a merge walk that only moves forward.  Every byte of the row is stored once: no zero-fill pass, no atomics.
constexpr int kMaskWarps = 8;
DDZ_DEV bool has_id(const int16_t* ids, int n, int id) {
    int lo = 0, hi = n;                                    // first entry >= id
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ids[mid] < id) lo = mid + 1; else hi = mid; }
    return lo < n && ids[lo] == id;
}
template <bool BYTES>
__global__ void __launch_bounds__(kMaskWarps * 32) k_legal_mask(const int32_t* __restrict__ offsets,
                                                                const uint64_t* __restrict__ actions, long long cap,
                                                                void* out, int64_t* stats, int B) {
    __shared__ int16_t sids[kMaskWarps][DDZ_MAX_LEGAL];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * kMaskWarps + w;
    if (b >= B) return;
    int16_t* ids = sids[w];
    const long long lo = offsets[b], full = max(0ll, (long long)offsets[b + 1] - lo);
    const long long stored = max(0ll, min(full, cap - lo));
    if (lane == 0 && stored < full && stats) atomicAdd((unsigned long long*)&stats[7], 1ull);
    const int n = (int)min(stored, (long long)DDZ_MAX_LEGAL);
    for (int i = lane; i < n; i += 32) ids[i] = (int16_t)move_id(actions[lo + i]);
    __syncwarp();
    constexpr int kSpan = BYTES ? 16 : 128;                // ids per 16-byte piece
    int p = 0;
    auto piece = [&](int base) {                           // the 16 bytes of ids [base, base + kSpan)
        uint32_t v[4] = {0u, 0u, 0u, 0u};
        while (p < n && ids[p] < base) p++;
        for (; p < n && ids[p] < base + kSpan; p++) {
            const int d = ids[p] - base;                   // < 0 only for an entry that is not a move (-1)
            if (d >= 0) { if (BYTES) v[d >> 2] |= 1u << (8 * (d & 3)); else v[d >> 5] |= 1u << (d & 31); }
        }
        return make_uint4(v[0], v[1], v[2], v[3]);
    };
    if (!BYTES) {
        uint4* row = reinterpret_cast<uint4*>(out) + (size_t)b * (DDZ_MASK_WORDS / 4);
        for (int c = lane; c < DDZ_MASK_WORDS / 4; c += 32) row[c] = piece(c * kSpan);
    } else {
        uint8_t* row = reinterpret_cast<uint8_t*>(out) + (size_t)b * DDZ_NUM_ACTION_IDS;
        const int head = (int)((0u - (uint32_t)reinterpret_cast<uintptr_t>(row)) & 15u);   // bytes before a 16-byte boundary
        const int nmid = (DDZ_NUM_ACTION_IDS - head) >> 4, tail = head + 16 * nmid;
        if (lane < head) row[lane] = has_id(ids, n, lane);
        if (lane >= 16 && tail + lane - 16 < DDZ_NUM_ACTION_IDS) row[tail + lane - 16] = has_id(ids, n, tail + lane - 16);
        uint4* mid = reinterpret_cast<uint4*>(row + head);
        for (int c = lane; c < nmid; c += 32) mid[c] = piece(head + c * kSpan);
    }
}

}  // namespace ddz

// ------------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------------
using namespace ddz;

static thread_local char g_err[256] = "";
static std::atomic<int> g_tile_order{DDZ_TILES_AUTO};
static int cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString(e));
    return DDZ_E_CUDA;
}
#define DDZ_LAUNCH_CHECK(what)                                         \
    do {                                                               \
        cudaError_t e_ = cudaGetLastError();                           \
        if (e_ != cudaSuccess) return cuda_fail(e_, what);             \
    } while (0)

// CTAs of `kernel` (instantiation V, MODE, LEAN) that fit on the current device at once, cached per device (the shapes of
// the devices of a box may differ)
template <int V, int MODE, bool LEAN>
static int resident_ctas(const void* kernel, size_t smem, int& resident) {
    static std::atomic<int> resident_of[64];
    static std::once_flag once;
    std::call_once(once, [] { for (auto& r : resident_of) r.store(-1); });
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return cuda_fail(cudaGetLastError(), "cudaGetDevice");
    resident = dev < 64 ? resident_of[dev].load(std::memory_order_relaxed) : -1;
    if (resident < 0) {
        int per_sm = 0, sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem) != cudaSuccess)
            return cuda_fail(cudaGetLastError(), "occupancy query");
        resident = per_sm * sms;
        if (dev < 64) resident_of[dev].store(resident, std::memory_order_relaxed);
    }
    return 0;
}
template <int V, int MODE>
static int launch_env(void* state, const StepArgs& a, const OutArgs& o, void* workspace, int64_t* stats, int B, cudaStream_t st) {
    const size_t smem = (MODE == kStepOnly) ? 0 : kWarpsPerCta * sizeof(WarpSmem);
    Workspace ws = workspace ? ws_of(workspace) : Workspace{nullptr, nullptr};
    const int grid = (ntiles(B) + kWarpsPerCta - 1) / kWarpsPerCta;
    int resident = 0;
    if (int rc = resident_ctas<V, MODE, false>((const void*)k_env<V, MODE>, smem, resident)) return rc;
    // a step with a face whose grid fits at once at lean::k_step_observe's occupancy runs that kernel (more registers
    // per warp, no spills); a larger one runs k_env, which holds one wave of 131 072 envs
    bool lean_fits = false;
    if constexpr (MODE == kStepObserve && V >= 0) {
        int lean_resident = 0;
        if (int rc = resident_ctas<V, MODE, true>((const void*)lean::k_step_observe<V>, smem, lean_resident)) return rc;
        if (grid <= lean_resident) { lean_fits = true; resident = lean_resident; }
    }
    OutArgs oo = o;
    // tile = launch position needs every lower tile to be running or done when a tile waits on it: true when the whole grid
    // is resident at once (and CTAs are dispatched in launch order, as they are in practice).  A caller whose other kernels
    // share the GPU asks for tickets instead (ddz_set_tile_order): correct under any dispatch order.
    oo.static_tiles = (g_tile_order.load(std::memory_order_relaxed) == DDZ_TILES_AUTO && grid <= resident) ? 1 : 0;
    if constexpr (MODE == kStepObserve && V >= 0) {
        if (lean_fits) {
            lean::k_step_observe<V><<<grid, kThreads, smem, st>>>(state, a, oo, ws, stats, B);
            DDZ_LAUNCH_CHECK("lean::k_step_observe");
            return 0;
        }
    }
    k_env<V, MODE><<<grid, kThreads, smem, st>>>(state, a, oo, ws, stats, B);
    DDZ_LAUNCH_CHECK("k_env");
    return 0;
}
template <int V>
static int launch_q_features(const void* state, const int32_t* offsets, const uint64_t* actions, const uint8_t* env_mask,
                             const int32_t* dst_offsets, int env_begin, int env_count, long long row_base, const float* T,
                             const float* rank_bias, const float* L, const float* line_bias, int W, void* out, int out_bf16,
                             int B, cudaStream_t st) {
    const size_t smem = (size_t)5 * kQThreads * sizeof(float4);   // 20 KB
    const float4* T4 = reinterpret_cast<const float4*>(T);
    const float4* rb4 = reinterpret_cast<const float4*>(rank_bias);
#define DDZ_Q_LAUNCH(BF, WC_) k_q_features<V, BF, WC_><<<env_count, kQThreads, smem, st>>>(                        \
        state, offsets, actions, env_mask, dst_offsets, env_begin, row_base, T4, rb4, L, line_bias, W, out, B)
    if (W == 256) { if (out_bf16) DDZ_Q_LAUNCH(true, 256); else DDZ_Q_LAUNCH(false, 256); }
    else          { if (out_bf16) DDZ_Q_LAUNCH(true, 0); else DDZ_Q_LAUNCH(false, 0); }
#undef DDZ_Q_LAUNCH
    DDZ_LAUNCH_CHECK("k_q_features");
    return 0;
}
template <int MODE>
static int launch_env_v(int variant, bool want_face, void* state, const StepArgs& a, const OutArgs& o, void* workspace,
                        int64_t* stats, int B, cudaStream_t st) {
    if (!want_face) return launch_env<-1, MODE>(state, a, o, workspace, stats, B, st);
    switch (variant) {
        case 0: return launch_env<0, MODE>(state, a, o, workspace, stats, B, st);
        case 1: return launch_env<1, MODE>(state, a, o, workspace, stats, B, st);
        case 2: return launch_env<2, MODE>(state, a, o, workspace, stats, B, st);
        case 3: return launch_env<3, MODE>(state, a, o, workspace, stats, B, st);
    }
    return DDZ_E_ARG;
}

// driver entry points for the compressible row buffers (ddz_rows_alloc), fetched through the runtime
namespace {
struct DriverApi {
    CUresult (*getGranularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags);
    CUresult (*create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long);
    CUresult (*release)(CUmemGenericAllocationHandle);
    CUresult (*reserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long);
    CUresult (*addressFree)(CUdeviceptr, size_t);
    CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long);
    CUresult (*unmap)(CUdeviceptr, size_t);
    CUresult (*setAccess)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t);
    bool ok;
};
template <class Fn>
bool driver_fn(const char* name, Fn& fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult st;
    if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess || !p) {
        cudaGetLastError();
        return false;
    }
    fn = reinterpret_cast<Fn>(p);
    return true;
}
const DriverApi& driver_api() {
    static DriverApi d = [] {
        DriverApi a{};
        a.ok = driver_fn("cuMemGetAllocationGranularity", a.getGranularity) && driver_fn("cuMemCreate", a.create) &&
               driver_fn("cuMemRelease", a.release) && driver_fn("cuMemAddressReserve", a.reserve) &&
               driver_fn("cuMemAddressFree", a.addressFree) && driver_fn("cuMemMap", a.map) &&
               driver_fn("cuMemUnmap", a.unmap) && driver_fn("cuMemSetAccess", a.setAccess);
        return a;
    }();
    return d;
}
}  // namespace

template <int V>
static int launch_face_gather(const void* state, const int64_t* rows, int64_t n, const uint64_t* moves, float* face,
                              float* move_rows, int layout, int B, cudaStream_t st) {
    const unsigned grid = (unsigned)((n + kEnvs - 1) / kEnvs);
    if (layout == DDZ_ROWS_CONCAT)
        k_face_gather<V, true><<<grid, kEnvs, 0, st>>>(state, rows, n, moves, (float4*)face, nullptr, B);
    else
        k_face_gather<V, false><<<grid, kEnvs, 0, st>>>(state, rows, n, moves, (float4*)face, (float4*)move_rows, B);
    DDZ_LAUNCH_CHECK("k_face_gather");
    return 0;
}

// f(std::integral_constant<int, DT>) for the dtype code of a linear head
template <class F>
static void by_dtype(int dtype, F&& f) {
    if (dtype == DDZ_DTYPE_F32) f(std::integral_constant<int, DDZ_DTYPE_F32>{});
    else f(std::integral_constant<int, DDZ_DTYPE_BF16>{});
}
constexpr unsigned kLinearThreads = linear_head::kWarps * 32;

extern "C" {

#ifdef DDZ_TRACE
int ddz_debug_set_trace(unsigned long long* buf) {
    return cudaMemcpyToSymbol(g_trace, &buf, sizeof buf) == cudaSuccess ? 0 : DDZ_E_CUDA;
}
#endif
int ddz_abi_version(void) { return DDZ_ABI_VERSION; }
int ddz_prob_form(void) { return kProbForm; }
int ddz_set_tile_order(int mode) {
    if (mode != DDZ_TILES_AUTO && mode != DDZ_TILES_TICKET) return DDZ_E_ARG;
    return g_tile_order.exchange(mode);
}
int ddz_face_channels(int variant) {
    static const int C[4] = {4, 7, 9, 6};
    return (variant < 0 || variant > 3) ? DDZ_E_ARG : C[variant];
}
size_t ddz_state_bytes(int B) { return B <= 0 ? 0 : (size_t)B * (9 * 8 + 4); }
size_t ddz_workspace_bytes(int B) { return B <= 0 ? 0 : 256 + (size_t)ntiles(B) * 8; }
const char* ddz_last_error(void) { return g_err; }

int ddz_reset(void* state, const int8_t* perm, const int8_t* lord_pile, int pool_games, int only_done,
              int64_t* stats, int B, void* stream) {
    if (!state || !perm || B <= 0 || pool_games < 1) return DDZ_E_ARG;
    k_reset<<<nblocks(B), kEnvs, 0, (cudaStream_t)stream>>>(state, perm, lord_pile, pool_games, only_done, stats, B);
    DDZ_LAUNCH_CHECK("k_reset");
    return 0;
}

int ddz_observe(const void* state, void* workspace, int variant, int32_t* offsets, uint64_t* actions_u64,
                float* actions_f32, int64_t cap, float* face, int64_t* stats, int B, void* stream) {
    if (!state || !workspace || !offsets || !actions_u64 || B <= 0 || cap < 0) return DDZ_E_ARG;
    if (face && ddz_face_channels(variant) < 0) return DDZ_E_ARG;
    StepArgs a; memset(&a, 0, sizeof a);
    OutArgs o{offsets, actions_u64, (float4*)actions_f32, cap, (float4*)face, 0};
    return launch_env_v<kObserve>(variant, face != nullptr, const_cast<void*>(state), a, o, workspace, stats, B,
                                  (cudaStream_t)stream);
}

int ddz_legal_count(const void* state, int32_t* counts, int B, void* stream) {
    if (!state || !counts || B <= 0) return DDZ_E_ARG;
    k_legal_count<<<(B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(state, counts, B);
    DDZ_LAUNCH_CHECK("k_legal_count");
    return 0;
}

int ddz_legal_emit(const void* state, void* workspace, int32_t* offsets, uint64_t* actions_u64, int64_t cap,
                   int64_t* stats, int B, void* stream) {
    return ddz_observe(state, workspace, 0, offsets, actions_u64, nullptr, cap, nullptr, stats, B, stream);
}

static int fill_step_args(StepArgs& a, const int32_t* offsets, const uint64_t* actions, const void* choice, int mode,
                          uint64_t seed, uint64_t env0, uint32_t stepno, const int32_t rewards[3], int8_t* r,
                          uint8_t* done, int8_t* cat, float* reward) {
    static const int32_t defR[3] = {50, 100, 50};   // game.py:13-14 (up, lord, down)
    if (!offsets || !actions || mode < 0 || mode > 3) return DDZ_E_ARG;
    if (mode != DDZ_CHOICE_PHILOX && !choice) return DDZ_E_ARG;
    memset(&a, 0, sizeof a);
    a.offsets = offsets; a.actions = actions; a.choice = choice; a.mode = mode;
    a.seed = seed; a.env0 = env0; a.stepno = stepno;
    for (int i = 0; i < 3; i++) a.rewards[i] = rewards ? rewards[i] : defR[i];
    a.r = r; a.done = done; a.cat = cat; a.reward = reward;
    a.pool_games = 1;
    a.prev_cap = -1;   // ddz_step: complete lists (ddz_rollout_step sets the capacity)
    return 0;
}

int ddz_step(void* state, const int32_t* offsets, const uint64_t* actions_u64, const void* choice,
             int choice_mode, uint64_t seed, uint64_t env0, uint32_t stepno, const int32_t rewards[3],
             int8_t* r, uint8_t* done, int8_t* cat, float* reward, int64_t* stats, int B, void* stream) {
    if (!state || B <= 0) return DDZ_E_ARG;
    StepArgs a;
    int rc = fill_step_args(a, offsets, actions_u64, choice, choice_mode, seed, env0, stepno, rewards, r, done, cat, reward);
    if (rc) return rc;
    OutArgs o{nullptr, nullptr, nullptr, 0, nullptr, 0};
    return launch_env<-1, kStepOnly>(state, a, o, nullptr, stats, B, (cudaStream_t)stream);
}

int ddz_rollout_step(void* state, void* workspace, int variant,
                     const int32_t* prev_offsets, const uint64_t* prev_actions_u64,
                     const void* choice, int choice_mode, uint64_t seed, uint64_t env0, uint32_t stepno,
                     const int32_t rewards[3], const int8_t* perm, const int8_t* lord_pile, int pool_games,
                     int8_t* r, uint8_t* done, int8_t* cat, float* reward,
                     int32_t* out_offsets, uint64_t* out_actions_u64, float* out_actions_f32, int64_t cap,
                     float* face, int64_t* stats, int B, void* stream) {
    if (!state || !workspace || !out_offsets || !out_actions_u64 || B <= 0 || cap < 0) return DDZ_E_ARG;
    // at cap = 0 nothing is read from or written to the action lists, so they may alias (ddz_rollout_steps' slices do)
    if (out_offsets == prev_offsets || (cap > 0 && out_actions_u64 == prev_actions_u64)) return DDZ_E_ARG;
    if (face && ddz_face_channels(variant) < 0) return DDZ_E_ARG;
    if (perm && pool_games < 1) return DDZ_E_ARG;
    StepArgs a;
    int rc = fill_step_args(a, prev_offsets, prev_actions_u64, choice, choice_mode, seed, env0, stepno, rewards, r, done, cat, reward);
    if (rc) return rc;
    a.perm = perm; a.lord_pile = lord_pile; a.pool_games = perm ? pool_games : 1;
    a.prev_cap = cap;   // the ping-pong lists have the same capacity
    OutArgs o{out_offsets, out_actions_u64, (float4*)out_actions_f32, cap, (float4*)face, 0};
    return launch_env_v<kStepObserve>(variant, face != nullptr, state, a, o, workspace, stats, B, (cudaStream_t)stream);
}

int ddz_rollout_steps(void* state, void* workspace, int variant, int nsteps,
                      const int32_t* prev_offsets, const uint64_t* prev_actions_u64,
                      const void* choice, int choice_mode, uint64_t seed, uint64_t env0, uint32_t stepno,
                      const int32_t rewards[3], const int8_t* perm, const int8_t* lord_pile, int pool_games,
                      int8_t* r, uint8_t* done, int8_t* cat, float* reward,
                      int32_t* out_offsets, uint64_t* out_actions_u64, float* out_actions_f32, int64_t cap,
                      float* face, int64_t* stats, int B, void* stream) {
    if (nsteps < 1 || B <= 0 || cap < 0 || !out_offsets || !out_actions_u64) return DDZ_E_ARG;
    if (choice_mode != DDZ_CHOICE_PHILOX && choice_mode != DDZ_CHOICE_MOD) return DDZ_E_ARG;   // nobody sees the lists in between
    const int C = face ? ddz_face_channels(variant) : 0;
    if (C < 0) return DDZ_E_ARG;
    const size_t nB = (size_t)B;
    for (int s = 0; s < nsteps; s++) {
        const size_t k = (size_t)s;
        const int rc = ddz_rollout_step(
            state, workspace, variant, s ? out_offsets + (k - 1) * (nB + 1) : prev_offsets,
            s ? out_actions_u64 + (k - 1) * (size_t)cap : prev_actions_u64,
            choice ? (const char*)choice + k * nB * 4 : nullptr, choice_mode, seed, env0,
            stepno == DDZ_STEPNO_AUTO ? stepno : stepno + (uint32_t)s, rewards, perm, lord_pile, pool_games,
            r ? r + k * nB : nullptr, done ? done + k * nB : nullptr, cat ? cat + k * nB : nullptr,
            reward ? reward + k * nB * 3 : nullptr, out_offsets + k * (nB + 1), out_actions_u64 + k * (size_t)cap,
            out_actions_f32 ? out_actions_f32 + k * (size_t)cap * 60 : nullptr, cap,
            face ? face + k * nB * (size_t)C * 60 : nullptr, stats, B, stream);
        if (rc) return rc;
    }
    return 0;
}

// ---- host-buffer pipeline -------------------------------------------------------------------------
struct ddz_pipe {
    cudaStream_t h2d, d2h, refill;
    cudaEvent_t in_ready[2], in_free[2], kernel_done[2], out_done[DDZ_PIPE_DEPTH], stage_free, stage_full;
    unsigned long long step;
    bool stage_used;
    // a deal-pool upload that is on its way into the staging buffers: committed (device-to-device, between two steps) by
    // the first ddz_pipe_step that finds it complete, so that no step ever waits for a large host copy
    struct { int8_t *dst_perm, *dst_lord, *stage_perm, *stage_lord; size_t rows; bool active; } pending;
};
#define DDZ_CUDA(call, what)                                   \
    do {                                                       \
        cudaError_t e_ = (call);                               \
        if (e_ != cudaSuccess) return cuda_fail(e_, what);     \
    } while (0)

ddz_pipe* ddz_pipe_create(void) {
    ddz_pipe* p = new ddz_pipe();
    p->step = 0; p->stage_used = false; p->pending.active = false;
    bool ok = cudaStreamCreateWithFlags(&p->h2d, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->d2h, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->refill, cudaStreamNonBlocking) == cudaSuccess;
    cudaEvent_t* evs[] = {&p->in_ready[0], &p->in_ready[1], &p->in_free[0], &p->in_free[1], &p->kernel_done[0],
                          &p->kernel_done[1], &p->stage_free, &p->stage_full};
    for (cudaEvent_t* e : evs) ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
    for (cudaEvent_t& e : p->out_done) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { cuda_fail(cudaGetLastError(), "ddz_pipe_create"); delete p; return nullptr; }
    return p;
}
void ddz_pipe_destroy(ddz_pipe* p) {
    if (!p) return;
    cudaStreamDestroy(p->h2d); cudaStreamDestroy(p->d2h); cudaStreamDestroy(p->refill);
    cudaEvent_t evs[] = {p->in_ready[0], p->in_ready[1], p->in_free[0], p->in_free[1], p->kernel_done[0],
                         p->kernel_done[1], p->stage_free, p->stage_full};
    for (cudaEvent_t e : evs) cudaEventDestroy(e);
    for (cudaEvent_t e : p->out_done) cudaEventDestroy(e);
    delete p;
}
// replace the pool slot by the staged upload (device-to-device on the main stream, i.e. between two steps)
static int pipe_commit_refill(ddz_pipe* p, cudaStream_t main_s, bool wait) {
    if (!p->pending.active) return 0;
    if (!wait && cudaEventQuery(p->stage_full) != cudaSuccess) { cudaGetLastError(); return 0; }   // still uploading
    DDZ_CUDA(cudaStreamWaitEvent(main_s, p->stage_full, 0), "wait stage_full");
    DDZ_CUDA(cudaMemcpyAsync(p->pending.dst_perm, p->pending.stage_perm, p->pending.rows * 54, cudaMemcpyDeviceToDevice, main_s), "D2D perm");
    DDZ_CUDA(cudaMemcpyAsync(p->pending.dst_lord, p->pending.stage_lord, p->pending.rows, cudaMemcpyDeviceToDevice, main_s), "D2D lord");
    DDZ_CUDA(cudaEventRecord(p->stage_free, main_s), "record stage_free");
    p->pending.active = false;
    return 0;
}

int ddz_pipe_step(ddz_pipe* p, void* state, void* workspace, int variant,
                  const int32_t* prev_offsets, const uint64_t* prev_actions_u64,
                  const void* host_choice, void* dev_choice, uint64_t seed, uint64_t env0, uint32_t stepno,
                  const int32_t rewards[3], const int8_t* perm, const int8_t* lord_pile, int pool_games,
                  void* results_dev, void* results_host, size_t results_bytes,
                  int32_t* out_offsets, uint64_t* out_actions_u64, float* out_actions_f32, int64_t cap,
                  float* face, int64_t* stats, int B, void* stream) {
    if (!p || !host_choice || !dev_choice || !results_dev || !results_host || B <= 0) return DDZ_E_ARG;
    if (results_bytes < (size_t)B * 3) return DDZ_E_ARG;       // at least r | done | cat; the reward block is optional
    cudaStream_t main_s = (cudaStream_t)stream;
    if (int rc = pipe_commit_refill(p, main_s, false)) return rc;
    const int k = (int)(p->step & 1);
    const bool primed = p->step >= 2;                          // events of this parity were recorded two steps ago
    // H2D of this step's entropy, once the kernel that last read dev_choice (two steps ago) is done
    if (primed) DDZ_CUDA(cudaStreamWaitEvent(p->h2d, p->in_free[k], 0), "wait in_free");
    DDZ_CUDA(cudaMemcpyAsync(dev_choice, host_choice, (size_t)B * 4, cudaMemcpyHostToDevice, p->h2d), "H2D entropy");
    DDZ_CUDA(cudaEventRecord(p->in_ready[k], p->h2d), "record in_ready");
    DDZ_CUDA(cudaStreamWaitEvent(main_s, p->in_ready[k], 0), "wait in_ready");
    // results_dev alternates between two sets: the D2H that last read this set was issued two steps ago
    if (primed) DDZ_CUDA(cudaStreamWaitEvent(main_s, p->out_done[(p->step - 2) % DDZ_PIPE_DEPTH], 0), "wait out_done");
    char* rd = (char*)results_dev;
    const size_t off_reward = ((size_t)3 * B + 15) / 16 * 16;
    int rc = ddz_rollout_step(state, workspace, variant, prev_offsets, prev_actions_u64, dev_choice, DDZ_CHOICE_MOD, seed,
                              env0, stepno, rewards, perm, lord_pile, pool_games, (int8_t*)rd, (uint8_t*)rd + B,
                              (int8_t*)rd + 2 * (size_t)B, (float*)(rd + off_reward), out_offsets, out_actions_u64,
                              out_actions_f32, cap, face, stats, B, stream);
    if (rc) return rc;
    DDZ_CUDA(cudaEventRecord(p->kernel_done[k], main_s), "record kernel_done");
    DDZ_CUDA(cudaEventRecord(p->in_free[k], main_s), "record in_free");
    DDZ_CUDA(cudaStreamWaitEvent(p->d2h, p->kernel_done[k], 0), "wait kernel_done");
    DDZ_CUDA(cudaMemcpyAsync(results_host, results_dev, results_bytes, cudaMemcpyDeviceToHost, p->d2h), "D2H results");
    DDZ_CUDA(cudaEventRecord(p->out_done[p->step % DDZ_PIPE_DEPTH], p->d2h), "record out_done");
    p->step++;
    return 0;
}
int ddz_pipe_wait(ddz_pipe* p, int slot) {
    if (!p || slot < 0 || slot >= DDZ_PIPE_DEPTH) return DDZ_E_ARG;
    DDZ_CUDA(cudaEventSynchronize(p->out_done[slot]), "ddz_pipe_wait");
    return 0;
}
int ddz_pipe_refill(ddz_pipe* p, int8_t* pool_perm_slot, int8_t* pool_lord_slot, const int8_t* host_perm,
                    const int8_t* host_lord, int8_t* stage_perm, int8_t* stage_lord, int B, void* stream) {
    if (!p || !pool_perm_slot || !pool_lord_slot || !host_perm || !host_lord || !stage_perm || !stage_lord || B <= 0)
        return DDZ_E_ARG;
    cudaStream_t main_s = (cudaStream_t)stream;
    if (int rc = pipe_commit_refill(p, main_s, true)) return rc;          // an earlier upload still staged: commit it first
    if (p->stage_used) DDZ_CUDA(cudaStreamWaitEvent(p->refill, p->stage_free, 0), "wait stage_free");
    DDZ_CUDA(cudaMemcpyAsync(stage_perm, host_perm, (size_t)B * 54, cudaMemcpyHostToDevice, p->refill), "H2D perm");
    DDZ_CUDA(cudaMemcpyAsync(stage_lord, host_lord, (size_t)B, cudaMemcpyHostToDevice, p->refill), "H2D lord");
    DDZ_CUDA(cudaEventRecord(p->stage_full, p->refill), "record stage_full");
    p->pending.dst_perm = pool_perm_slot; p->pending.dst_lord = pool_lord_slot;
    p->pending.stage_perm = stage_perm; p->pending.stage_lord = stage_lord;
    p->pending.rows = (size_t)B; p->pending.active = true;
    p->stage_used = true;
    return 0;
}
int ddz_pipe_flush(ddz_pipe* p, void* stream) {
    if (!p) return DDZ_E_ARG;
    return pipe_commit_refill(p, (cudaStream_t)stream, true);
}

// ---- host-buffer pipeline over several env groups ---------------------------------------------------
// One native call per env-step of ALL groups of a GPU:
//   copy stream  : H2D of the step's pinned entropy (one copy for all groups)                      -> event in_ready
//   stream g     : wait in_ready; k_env of group g (its slice of the entropy; r|done|cat -> results_dev) -> event kdone[g]
//   copy stream 2: wait every kdone[g]; D2H of all groups' results (one copy)                       -> event out_done[slot]
// dev_choice / results_dev / results_host rotate through DDZ_PIPE_DEPTH buffers, and the step that reuses a slot first
// makes sure (on the HOST, normally a no-op) that the D2H of the step that used it before has landed -- so no stream ever
// waits for an older step: the groups stay unsynchronised, the only cross-stream edges are "entropy is there" and "this
// step's kernels are done".  4 G + 4 CUDA calls per step (12 G with ddz_pipe_step per group).
struct ddz_mpipe {
    int G;
    cudaStream_t h2d, d2h, refill;
    cudaEvent_t in_ready[DDZ_PIPE_DEPTH], out_done[DDZ_PIPE_DEPTH], stage_full;
    cudaEvent_t kdone[DDZ_PIPE_DEPTH][DDZ_MPIPE_MAX_GROUPS], committed[DDZ_MPIPE_MAX_GROUPS];
    bool out_pending[DDZ_PIPE_DEPTH];
    unsigned long long step;
    bool stage_used;
    // a deal-pool upload in progress: it goes up in chunks, one per step, so that a step's entropy copy never queues behind
    // megabytes of permutations on the host-to-device copy engine; `uploaded` < `bytes` while chunks are outstanding
    struct { int8_t *dst_perm[DDZ_MPIPE_MAX_GROUPS], *dst_lord[DDZ_MPIPE_MAX_GROUPS]; int8_t *stage_perm, *stage_lord;
             const int8_t *host_perm, *host_lord; size_t rows, uploaded, bytes; bool active; } pending;
};
constexpr size_t kRefillChunk = 384 * 1024;

ddz_mpipe* ddz_mpipe_create(int groups) {
    if (groups < 1 || groups > DDZ_MPIPE_MAX_GROUPS) { snprintf(g_err, sizeof g_err, "ddz_mpipe_create: 1..%d groups", DDZ_MPIPE_MAX_GROUPS); return nullptr; }
    ddz_mpipe* p = new ddz_mpipe();
    p->G = groups; p->step = 0; p->stage_used = false; p->pending.active = false;
    bool ok = cudaStreamCreateWithFlags(&p->h2d, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->d2h, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->refill, cudaStreamNonBlocking) == cudaSuccess;
    auto mk = [&](cudaEvent_t* e) { ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess; };
    mk(&p->stage_full);
    for (int k = 0; k < DDZ_PIPE_DEPTH; k++) { mk(&p->in_ready[k]); mk(&p->out_done[k]); p->out_pending[k] = false; }
    for (int g = 0; g < groups; g++) {
        mk(&p->committed[g]);
        for (int k = 0; k < DDZ_PIPE_DEPTH; k++) mk(&p->kdone[k][g]);
    }
    if (!ok) { cuda_fail(cudaGetLastError(), "ddz_mpipe_create"); delete p; return nullptr; }   // (a failed create leaks its few events)
    return p;
}
void ddz_mpipe_destroy(ddz_mpipe* p) {
    if (!p) return;
    cudaStreamDestroy(p->h2d); cudaStreamDestroy(p->d2h); cudaStreamDestroy(p->refill);
    cudaEventDestroy(p->stage_full);
    for (int k = 0; k < DDZ_PIPE_DEPTH; k++) { cudaEventDestroy(p->in_ready[k]); cudaEventDestroy(p->out_done[k]); }
    for (int g = 0; g < p->G; g++) {
        cudaEventDestroy(p->committed[g]);
        for (int k = 0; k < DDZ_PIPE_DEPTH; k++) cudaEventDestroy(p->kdone[k][g]);
    }
    delete p;
}
// next chunk(s) of a staged deal-pool upload (all of the rest when `all`); the last one records stage_full
static int mpipe_upload_chunk(ddz_mpipe* p, bool all) {
    auto& u = p->pending;
    while (u.active && u.uploaded < u.bytes) {
        const size_t n = all ? u.bytes - u.uploaded : (u.bytes - u.uploaded < kRefillChunk ? u.bytes - u.uploaded : kRefillChunk);
        DDZ_CUDA(cudaMemcpyAsync(u.stage_perm + u.uploaded, u.host_perm + u.uploaded, n, cudaMemcpyHostToDevice, p->refill), "H2D perm");
        u.uploaded += n;
        if (u.uploaded == u.bytes) {
            DDZ_CUDA(cudaMemcpyAsync(u.stage_lord, u.host_lord, u.rows, cudaMemcpyHostToDevice, p->refill), "H2D lord");
            DDZ_CUDA(cudaEventRecord(p->stage_full, p->refill), "record stage_full");
        }
        if (!all) break;
    }
    return 0;
}
// replace every group's pool slot by its part of the staged upload, each on the group's stream (between two of its steps)
static int mpipe_commit_refill(ddz_mpipe* p, const ddz_group_step* gs, bool wait) {
    if (!p->pending.active) return 0;
    if (p->pending.uploaded < p->pending.bytes) {
        if (int rc = mpipe_upload_chunk(p, wait)) return rc;
        if (p->pending.uploaded < p->pending.bytes) return 0;                                      // more chunks to go
    }
    if (!wait && cudaEventQuery(p->stage_full) != cudaSuccess) { cudaGetLastError(); return 0; }   // still uploading
    size_t row0 = 0;
    for (int g = 0; g < p->G; g++) {
        cudaStream_t st = (cudaStream_t)gs[g].stream;
        const size_t rows = (size_t)gs[g].B;
        DDZ_CUDA(cudaStreamWaitEvent(st, p->stage_full, 0), "wait stage_full");
        DDZ_CUDA(cudaMemcpyAsync(p->pending.dst_perm[g], p->pending.stage_perm + 54 * row0, rows * 54, cudaMemcpyDeviceToDevice, st), "D2D perm");
        DDZ_CUDA(cudaMemcpyAsync(p->pending.dst_lord[g], p->pending.stage_lord + row0, rows, cudaMemcpyDeviceToDevice, st), "D2D lord");
        DDZ_CUDA(cudaEventRecord(p->committed[g], st), "record committed");
        row0 += rows;
    }
    p->pending.active = false;
    return 0;
}

int ddz_mpipe_step(ddz_mpipe* p, const ddz_group_step* gs, int variant, const void* host_choice, void* dev_choice,
                   uint64_t seed, uint32_t stepno, const int32_t rewards[3], int pool_games,
                   void* results_dev, void* results_host, int64_t* stats) {
    if (!p || !gs || !host_choice || !dev_choice || !results_dev || !results_host) return DDZ_E_ARG;
    size_t total = 0;
    for (int g = 0; g < p->G; g++) { if (gs[g].B <= 0 || !gs[g].state) return DDZ_E_ARG; total += (size_t)gs[g].B; }
    if (int rc = mpipe_commit_refill(p, gs, false)) return rc;
    const int slot = (int)(p->step % DDZ_PIPE_DEPTH);
    // the buffers of this slot were last used DDZ_PIPE_DEPTH steps ago: that step's results must have left the device
    if (p->out_pending[slot]) { DDZ_CUDA(cudaEventSynchronize(p->out_done[slot]), "slot reuse"); p->out_pending[slot] = false; }
    DDZ_CUDA(cudaMemcpyAsync(dev_choice, host_choice, total * 4, cudaMemcpyHostToDevice, p->h2d), "H2D entropy");
    DDZ_CUDA(cudaEventRecord(p->in_ready[slot], p->h2d), "record in_ready");
    size_t off = 0;
    for (int g = 0; g < p->G; g++) {
        const ddz_group_step& q = gs[g];
        cudaStream_t st = (cudaStream_t)q.stream;
        const size_t B = (size_t)q.B;
        DDZ_CUDA(cudaStreamWaitEvent(st, p->in_ready[slot], 0), "wait in_ready");
        char* rd = (char*)results_dev + 3 * off;
        int rc = ddz_rollout_step(q.state, q.workspace, variant, q.prev_offsets, q.prev_actions_u64,
                                  (const char*)dev_choice + 4 * off, DDZ_CHOICE_MOD, seed, q.env0, stepno, rewards, q.perm,
                                  q.lord_pile, pool_games, (int8_t*)rd, (uint8_t*)rd + B, (int8_t*)rd + 2 * B, q.reward,
                                  q.out_offsets, q.out_actions_u64, q.out_actions_f32, q.cap, q.face, stats, q.B, q.stream);
        if (rc) return rc;
        DDZ_CUDA(cudaEventRecord(p->kdone[slot][g], st), "record kdone");
        DDZ_CUDA(cudaStreamWaitEvent(p->d2h, p->kdone[slot][g], 0), "wait kdone");
        off += B;
    }
    DDZ_CUDA(cudaMemcpyAsync(results_host, results_dev, 3 * total, cudaMemcpyDeviceToHost, p->d2h), "D2H results");
    DDZ_CUDA(cudaEventRecord(p->out_done[slot], p->d2h), "record out_done");
    p->out_pending[slot] = true;
    p->step++;
    return 0;
}
int ddz_mpipe_wait(ddz_mpipe* p, int slot) {
    if (!p || slot < 0 || slot >= DDZ_PIPE_DEPTH) return DDZ_E_ARG;
    if (!p->out_pending[slot]) return 0;
    DDZ_CUDA(cudaEventSynchronize(p->out_done[slot]), "ddz_mpipe_wait");
    p->out_pending[slot] = false;
    return 0;
}
int ddz_mpipe_refill(ddz_mpipe* p, const ddz_group_step* gs, int8_t* const* pool_perm_slot, int8_t* const* pool_lord_slot,
                     const int8_t* host_perm, const int8_t* host_lord, int8_t* stage_perm, int8_t* stage_lord) {
    if (!p || !gs || !pool_perm_slot || !pool_lord_slot || !host_perm || !host_lord || !stage_perm || !stage_lord) return DDZ_E_ARG;
    if (int rc = mpipe_commit_refill(p, gs, true)) return rc;             // an earlier upload still staged: commit it first
    size_t total = 0;
    for (int g = 0; g < p->G; g++) {
        if (p->stage_used) DDZ_CUDA(cudaStreamWaitEvent(p->refill, p->committed[g], 0), "wait committed");
        p->pending.dst_perm[g] = pool_perm_slot[g]; p->pending.dst_lord[g] = pool_lord_slot[g];
        total += (size_t)gs[g].B;
    }
    p->pending.stage_perm = stage_perm; p->pending.stage_lord = stage_lord;
    p->pending.host_perm = host_perm; p->pending.host_lord = host_lord;
    p->pending.rows = total; p->pending.bytes = total * 54; p->pending.uploaded = 0; p->pending.active = true;
    p->stage_used = true;
    return mpipe_upload_chunk(p, false);      // the first chunk now, one more with every step
}
int ddz_mpipe_join(ddz_mpipe* p, void* stream) {
    if (!p) return DDZ_E_ARG;
    if (p->step == 0) return 0;
    DDZ_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, p->out_done[(p->step - 1) % DDZ_PIPE_DEPTH], 0), "ddz_mpipe_join");
    return 0;
}
int ddz_mpipe_flush(ddz_mpipe* p, const ddz_group_step* gs) {
    if (!p || !gs) return DDZ_E_ARG;
    return mpipe_commit_refill(p, gs, true);
}

// ---- compressible row buffers ------------------------------------------------------------------------
// The one-hot / face rows are floats that are 0 or 1 (or 0 or a scale): lines of them compress well.  Memory created with
// CU_MEM_ALLOCATION_COMP_GENERIC is compressed by the L2 on its way to HBM (and expanded on the way back), which raises
// the bandwidth the row writer sees (profiles/r1u_compressible.json).  Driver entry points are fetched through the
// runtime (cudaGetDriverEntryPoint): the library does not link libcuda and still loads on a machine without a driver.

int ddz_rows_alloc(size_t bytes, int device, void** ptr, size_t* mapped_bytes) {
    if (!ptr || !mapped_bytes || bytes == 0 || device < 0) return DDZ_E_ARG;
    *ptr = nullptr; *mapped_bytes = 0;
    const DriverApi& d = driver_api();
    if (!d.ok) { snprintf(g_err, sizeof g_err, "ddz_rows_alloc: virtual memory management entry points not available"); return DDZ_E_CUDA; }
    CUmemAllocationProp prop; memset(&prop, 0, sizeof prop);
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    if (d.getGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0) {
        snprintf(g_err, sizeof g_err, "ddz_rows_alloc: compressible memory is not supported on device %d", device);
        return DDZ_E_CUDA;
    }
    const size_t size = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle h;
    if (d.create(&h, size, &prop, 0) != CUDA_SUCCESS) {
        snprintf(g_err, sizeof g_err, "ddz_rows_alloc: cuMemCreate(%zu bytes, compressible) failed", size);
        return DDZ_E_CUDA;
    }
    CUdeviceptr p = 0;
    if (d.reserve(&p, size, 0, 0, 0) != CUDA_SUCCESS) { d.release(h); snprintf(g_err, sizeof g_err, "ddz_rows_alloc: address reservation failed"); return DDZ_E_CUDA; }
    CUmemAccessDesc acc; memset(&acc, 0, sizeof acc);
    acc.location = prop.location; acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (d.map(p, size, 0, h, 0) != CUDA_SUCCESS || d.setAccess(p, size, &acc, 1) != CUDA_SUCCESS) {
        d.unmap(p, size); d.addressFree(p, size); d.release(h);
        snprintf(g_err, sizeof g_err, "ddz_rows_alloc: mapping failed");
        return DDZ_E_CUDA;
    }
    d.release(h);                      // the mapping keeps the memory alive until ddz_rows_free unmaps it
    *ptr = (void*)p; *mapped_bytes = size;
    return 0;
}

int ddz_rows_free(void* ptr, size_t mapped_bytes) {
    if (!ptr || mapped_bytes == 0) return DDZ_E_ARG;
    const DriverApi& d = driver_api();
    if (!d.ok) return DDZ_E_CUDA;
    if (d.unmap((CUdeviceptr)ptr, mapped_bytes) != CUDA_SUCCESS || d.addressFree((CUdeviceptr)ptr, mapped_bytes) != CUDA_SUCCESS) {
        snprintf(g_err, sizeof g_err, "ddz_rows_free: unmap failed");
        return DDZ_E_CUDA;
    }
    return 0;
}

int ddz_legal_moves(const uint64_t* hands, const uint64_t* lasts, void* workspace, int32_t* offsets,
                    uint64_t* actions_u64, int64_t cap, int64_t* stats, int n, void* stream) {
    if (!hands || !lasts || !workspace || !offsets || !actions_u64 || n <= 0 || cap < 0) return DDZ_E_ARG;
    if ((reinterpret_cast<uintptr_t>(actions_u64) & 15u) != 0) return DDZ_E_ARG;   // pairs of moves go out as 16-byte stores
    OutArgs o{offsets, actions_u64, nullptr, cap, nullptr, 0};
    const int grid = (ntiles(n) + kFlatWarps - 1) / kFlatWarps;
    k_legal_flat<<<grid, kFlatWarps * 32, 0, (cudaStream_t)stream>>>(hands, lasts, o, ws_of(workspace), stats, n);
    DDZ_LAUNCH_CHECK("k_legal_flat");
    return 0;
}

int ddz_encode_actions(const uint64_t* actions_u64, int64_t n, float* out, void* stream) {
    if (n < 0 || (n > 0 && (!actions_u64 || !out))) return DDZ_E_ARG;
    if (n == 0) return 0;
    long long nvec = (long long)n * 15;
    long long blocks = (nvec + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k_encode_actions<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(actions_u64, n, (float4*)out);
    DDZ_LAUNCH_CHECK("k_encode_actions");
    return 0;
}

int ddz_encode_state_actions(const void* state, int variant, const int32_t* offsets, const uint64_t* actions_u64,
                             const uint8_t* env_mask, const int32_t* dst_offsets, float* out, int B, void* stream) {
    if (!state || !offsets || !actions_u64 || !out || B <= 0) return DDZ_E_ARG;
    const int grid = (B + 3) / 4;
    cudaStream_t st = (cudaStream_t)stream;
    switch (variant) {
        case 0: k_state_actions<0><<<grid, 128, 0, st>>>(state, offsets, actions_u64, env_mask, dst_offsets, (float4*)out, B); break;
        case 1: k_state_actions<1><<<grid, 128, 0, st>>>(state, offsets, actions_u64, env_mask, dst_offsets, (float4*)out, B); break;
        case 2: k_state_actions<2><<<grid, 128, 0, st>>>(state, offsets, actions_u64, env_mask, dst_offsets, (float4*)out, B); break;
        case 3: k_state_actions<3><<<grid, 128, 0, st>>>(state, offsets, actions_u64, env_mask, dst_offsets, (float4*)out, B); break;
        default: return DDZ_E_ARG;
    }
    DDZ_LAUNCH_CHECK("k_state_actions");
    return 0;
}

int ddz_q_features(const void* state, int variant, const int32_t* offsets, const uint64_t* actions_u64,
                   const uint8_t* env_mask, const int32_t* dst_offsets, int env_begin, int env_count, int64_t row_base,
                   const float* rank_tables, const float* rank_bias, const float* line_weights, const float* line_bias,
                   int width, void* out, int out_bf16, int B, void* stream) {
    if (!state || !offsets || !actions_u64 || !rank_tables || !rank_bias || !line_weights || !line_bias || !out || B <= 0 ||
        env_begin < 0 || env_count <= 0 || env_begin + env_count > B || width <= 0 || width > kQThreads || (width & 3))
        return DDZ_E_ARG;
    const cudaStream_t st = (cudaStream_t)stream;
    switch (variant) {
        case 0: return launch_q_features<0>(state, offsets, actions_u64, env_mask, dst_offsets, env_begin, env_count, row_base, rank_tables, rank_bias, line_weights, line_bias, width, out, out_bf16, B, st);
        case 1: return launch_q_features<1>(state, offsets, actions_u64, env_mask, dst_offsets, env_begin, env_count, row_base, rank_tables, rank_bias, line_weights, line_bias, width, out, out_bf16, B, st);
        case 2: return launch_q_features<2>(state, offsets, actions_u64, env_mask, dst_offsets, env_begin, env_count, row_base, rank_tables, rank_bias, line_weights, line_bias, width, out, out_bf16, B, st);
        case 3: return launch_q_features<3>(state, offsets, actions_u64, env_mask, dst_offsets, env_begin, env_count, row_base, rank_tables, rank_bias, line_weights, line_bias, width, out, out_bf16, B, st);
    }
    return DDZ_E_ARG;
}

int ddz_kth_moves(const uint64_t* hands, const uint64_t* lasts, const int32_t* idx, uint64_t* moves, int32_t* counts,
                  int n, void* stream) {
    if (!hands || !lasts || !idx || !moves || n <= 0) return DDZ_E_ARG;
    k_kth_moves<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(hands, lasts, idx, moves, counts, n);
    DDZ_LAUNCH_CHECK("k_kth_moves");
    return 0;
}

int ddz_playout(void* state, int max_steps, uint64_t seed, uint64_t env0, uint32_t stepno0, const int32_t rewards[3],
                int32_t* steps_taken, int64_t* stats, int B, void* stream) {
    static const int32_t defR[3] = {50, 100, 50};
    if (!state || B <= 0 || max_steps < 0) return DDZ_E_ARG;
    const int32_t* R = rewards ? rewards : defR;
    k_playout<false><<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(state, max_steps, seed, env0, stepno0, R[0], R[1], R[2],
                                                                          steps_taken, stats, B);
    DDZ_LAUNCH_CHECK("k_playout");
    return 0;
}

int ddz_playout_pruned(void* state, int max_steps, uint64_t seed, uint64_t env0, uint32_t stepno0, const int32_t rewards[3],
                       int32_t* steps_taken, int64_t* stats, int B, void* stream) {
    static const int32_t defR[3] = {50, 100, 50};
    if (!state || B <= 0 || max_steps < 0) return DDZ_E_ARG;
    const int32_t* R = rewards ? rewards : defR;
    k_playout<true><<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(state, max_steps, seed, env0, stepno0, R[0], R[1], R[2],
                                                                         steps_taken, stats, B);
    DDZ_LAUNCH_CHECK("k_playout<pruned>");
    return 0;
}

int ddz_mcts_moves(const uint64_t* hands, const uint64_t* lasts, uint64_t* moves, int32_t* counts, int n, void* stream) {
    if (!hands || !lasts || !moves || !counts || n <= 0) return DDZ_E_ARG;
    k_mcts_moves<<<(n + kSearchWarps - 1) / kSearchWarps, kSearchWarps * 32, 0, (cudaStream_t)stream>>>(hands, lasts, moves,
                                                                                                        counts, n);
    DDZ_LAUNCH_CHECK("k_mcts_moves");
    return 0;
}

size_t ddz_uct_workspace_bytes(int B, int budget) {
    if (B <= 0 || budget < 1 || budget > DDZ_UCT_MAX_BUDGET) return 0;
    return uct_header_bytes(B) + (size_t)B * (size_t)(budget + 1) * sizeof(UctNode);
}

int ddz_uct_search(const void* state, const uint8_t* env_mask, void* workspace, int budget, int width, int prune, double c,
                   const double* ln_table, uint64_t seed, uint64_t env0, int32_t* choice, uint64_t* move,
                   int32_t* root_n, uint64_t* root_moves, int32_t* root_visits, int32_t* root_wins, int root_stride,
                   int B, void* stream) {
    if (!state || !workspace || !ln_table || !choice || B <= 0) return DDZ_E_ARG;
    if (budget < 1 || budget > DDZ_UCT_MAX_BUDGET || width < 1 || width > DDZ_UCT_MAX_WIDTH) return DDZ_E_ARG;
    if ((int64_t)budget * width > DDZ_UCT_MAX_PLAYOUTS || !(c == c) || c - c != 0.0) return DDZ_E_ARG;   // c finite
    if (root_n && (!root_moves || !root_visits || !root_wins || root_stride < 1)) return DDZ_E_ARG;
    UctArgs a;
    a.state = state; a.mask = env_mask; a.ws = (char*)workspace; a.ln = ln_table;
    a.budget = budget; a.width = width; a.prune = prune != 0; a.c = c; a.seed = seed; a.env0 = env0;
    a.choice = choice; a.move = move; a.root_n = root_n; a.root_moves = root_moves; a.root_visits = root_visits;
    a.root_wins = root_wins; a.root_stride = root_stride; a.B = B;
    k_uct<<<(B + kUctWarps - 1) / kUctWarps, kUctWarps * 32, 0, (cudaStream_t)stream>>>(a);
    DDZ_LAUNCH_CHECK("k_uct");
    return 0;
}

int ddz_determinize(const void* state, const uint8_t* env_mask, int D, uint64_t seed, uint64_t env0, void* out_state,
                    int64_t* stats, int B, void* stream) {
    if (!state || !out_state || B <= 0 || D < 1 || D > DDZ_PIMC_MAX_DETERMINIZATIONS) return DDZ_E_ARG;
    const long long n = (long long)B * D;
    if (n > INT_MAX) return DDZ_E_ARG;
    k_determinize<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(state, env_mask, D, seed, env0, out_state,
                                                                                 stats, B);
    DDZ_LAUNCH_CHECK("k_determinize");
    return 0;
}

int ddz_uct_pool(const void* workspace, int budget, int D, int32_t* choice, uint64_t* move, int32_t* pooled_visits,
                 int32_t* pooled_wins, int B, void* stream) {
    if (!workspace || !choice || B <= 0 || budget < 1 || budget > DDZ_UCT_MAX_BUDGET) return DDZ_E_ARG;
    if (D < 1 || D > DDZ_PIMC_MAX_DETERMINIZATIONS || (long long)B * D > INT_MAX || (long long)D * budget > INT_MAX)
        return DDZ_E_ARG;
    k_uct_pool<<<(B + kPoolWarps - 1) / kPoolWarps, kPoolWarps * 32, 0, (cudaStream_t)stream>>>(
        (const char*)workspace, budget, D, choice, move, pooled_visits, pooled_wins, B);
    DDZ_LAUNCH_CHECK("k_uct_pool");
    return 0;
}

int ddz_select_actions(const float* q, const int32_t* offsets, float epsilon, uint64_t seed, uint64_t env0,
                       uint32_t stepno, int32_t* choice, int B, void* stream) {
    if (!q || !offsets || !choice || B <= 0 || !(epsilon >= 0.f && epsilon <= 1.f)) return DDZ_E_ARG;
    k_select_actions<<<(B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(q, offsets, epsilon, seed, env0, stepno, choice, B);
    DDZ_LAUNCH_CHECK("k_select_actions");
    return 0;
}

int ddz_encode_face(const void* state, int variant, float* face, int B, void* stream) {
    if (!state || !face || B <= 0 || ddz_face_channels(variant) < 0) return DDZ_E_ARG;
    dim3 g(nblocks(B)), t(kEnvs);
    cudaStream_t st = (cudaStream_t)stream;
    switch (variant) {
        case 0: k_face<0><<<g, t, 0, st>>>(state, (float4*)face, B); break;
        case 1: k_face<1><<<g, t, 0, st>>>(state, (float4*)face, B); break;
        case 2: k_face<2><<<g, t, 0, st>>>(state, (float4*)face, B); break;
        default: k_face<3><<<g, t, 0, st>>>(state, (float4*)face, B); break;
    }
    DDZ_LAUNCH_CHECK("k_face");
    return 0;
}

int ddz_encode_face_gather(const void* state, int variant, const int64_t* rows, int64_t n, const uint64_t* moves,
                           float* face, float* move_rows, int layout, int B, void* stream) {
    if (n < 0 || B <= 0 || ddz_face_channels(variant) < 0) return DDZ_E_ARG;
    if (layout != DDZ_ROWS_SPLIT && layout != DDZ_ROWS_CONCAT) return DDZ_E_ARG;
    if (n > 0 && (!state || !rows || !face)) return DDZ_E_ARG;
    if (layout == DDZ_ROWS_CONCAT && (!moves || move_rows)) return DDZ_E_ARG;
    if (layout == DDZ_ROWS_SPLIT && move_rows && !moves) return DDZ_E_ARG;
    if ((n + kEnvs - 1) / kEnvs > INT_MAX) return DDZ_E_ARG;
    if (n == 0) return 0;
    const cudaStream_t st = (cudaStream_t)stream;
    switch (variant) {
        case 0: return launch_face_gather<0>(state, rows, n, moves, face, move_rows, layout, B, st);
        case 1: return launch_face_gather<1>(state, rows, n, moves, face, move_rows, layout, B, st);
        case 2: return launch_face_gather<2>(state, rows, n, moves, face, move_rows, layout, B, st);
        default: return launch_face_gather<3>(state, rows, n, moves, face, move_rows, layout, B, st);
    }
}

static unsigned elementwise_grid(int64_t n) { const int64_t g = (n + 255) / 256; return (unsigned)(g < 148 * 16 ? g : 148 * 16); }

int ddz_move_ids(const uint64_t* moves, int64_t n, int32_t* ids, void* stream) {
    if (n < 0 || (n > 0 && (!moves || !ids))) return DDZ_E_ARG;
    if (n == 0) return 0;
    k_move_ids<<<elementwise_grid(n), 256, 0, (cudaStream_t)stream>>>(moves, n, ids);
    DDZ_LAUNCH_CHECK("k_move_ids");
    return 0;
}

int ddz_moves_of_ids(const int32_t* ids, int64_t n, uint64_t* moves, void* stream) {
    if (n < 0 || (n > 0 && (!ids || !moves))) return DDZ_E_ARG;
    if (n == 0) return 0;
    k_moves_of_ids<<<elementwise_grid(n), 256, 0, (cudaStream_t)stream>>>(ids, n, moves);
    DDZ_LAUNCH_CHECK("k_moves_of_ids");
    return 0;
}

int ddz_legal_mask(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, int layout, void* out, int64_t* stats,
                   int B, void* stream) {
    if (!offsets || !out || B <= 0 || cap < 0 || (cap > 0 && !actions_u64)) return DDZ_E_ARG;
    if (layout != DDZ_MASK_BITS && layout != DDZ_MASK_BYTES) return DDZ_E_ARG;
    if (layout == DDZ_MASK_BITS && (reinterpret_cast<uintptr_t>(out) & 15u) != 0) return DDZ_E_ARG;   // 16-byte row stores
    const unsigned grid = (unsigned)((B + kMaskWarps - 1) / kMaskWarps);
    const cudaStream_t st = (cudaStream_t)stream;
    if (layout == DDZ_MASK_BITS) k_legal_mask<false><<<grid, kMaskWarps * 32, 0, st>>>(offsets, actions_u64, cap, out, stats, B);
    else k_legal_mask<true><<<grid, kMaskWarps * 32, 0, st>>>(offsets, actions_u64, cap, out, stats, B);
    DDZ_LAUNCH_CHECK("k_legal_mask");
    return 0;
}

static bool policy_args_ok(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* logits, int dtype,
                           int64_t ld, int B) {
    if (!offsets || !logits || B <= 0 || cap < 0 || (cap > 0 && !actions_u64) || ld < DDZ_NUM_ACTION_IDS) return false;
    if (dtype != DDZ_DTYPE_F32 && dtype != DDZ_DTYPE_BF16) return false;
    return (reinterpret_cast<uintptr_t>(logits) & (dtype == DDZ_DTYPE_F32 ? 3u : 1u)) == 0;
}
static unsigned policy_grid(int B) { return (unsigned)((B + policy_head::kWarps - 1) / policy_head::kWarps); }

int ddz_policy_sample(void* state, const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* logits,
                      int dtype, int64_t ld, float temperature, uint64_t seed, uint64_t env0, uint32_t stepno,
                      const uint8_t* env_mask, int32_t* choice, int32_t* ids, float* logp, float* entropy, int64_t* stats,
                      int B, void* stream) {
    if (!policy_args_ok(offsets, actions_u64, cap, logits, dtype, ld, B) || !choice || !ids || !logp || !entropy) return DDZ_E_ARG;
    if (!(temperature >= 0.f) || !(temperature <= FLT_MAX)) return DDZ_E_ARG;              // NaN, negative or infinite
    uint32_t* meta = state ? reinterpret_cast<uint32_t*>(reinterpret_cast<uint64_t*>(state) + 9 * (size_t)B) : nullptr;
    const cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = policy_grid(B), threads = policy_head::kWarps * 32;
    if (dtype == DDZ_DTYPE_F32)
        policy_head::k_policy_sample<DDZ_DTYPE_F32><<<grid, threads, 0, st>>>(offsets, actions_u64, cap, logits, ld, temperature, seed,
                                                                              env0, stepno, env_mask, meta, choice, ids, logp,
                                                                              entropy, stats, B);
    else
        policy_head::k_policy_sample<DDZ_DTYPE_BF16><<<grid, threads, 0, st>>>(offsets, actions_u64, cap, logits, ld, temperature, seed,
                                                                               env0, stepno, env_mask, meta, choice, ids, logp,
                                                                               entropy, stats, B);
    DDZ_LAUNCH_CHECK("k_policy_sample");
    return 0;
}

int ddz_policy_logprob(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* logits, int dtype,
                       int64_t ld, const int32_t* ids, float* logp, float* entropy, float* lse, int64_t* stats, int B,
                       void* stream) {
    if (!policy_args_ok(offsets, actions_u64, cap, logits, dtype, ld, B) || !ids || !logp || !entropy) return DDZ_E_ARG;
    const cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = policy_grid(B), threads = policy_head::kWarps * 32;
    if (dtype == DDZ_DTYPE_F32)
        policy_head::k_policy_logprob<DDZ_DTYPE_F32><<<grid, threads, 0, st>>>(offsets, actions_u64, cap, logits, ld, ids, logp,
                                                                               entropy, lse, stats, B);
    else
        policy_head::k_policy_logprob<DDZ_DTYPE_BF16><<<grid, threads, 0, st>>>(offsets, actions_u64, cap, logits, ld, ids, logp,
                                                                                entropy, lse, stats, B);
    DDZ_LAUNCH_CHECK("k_policy_logprob");
    return 0;
}

int ddz_policy_logprob_backward(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* logits,
                                int dtype, int64_t ld, const int32_t* ids, const float* lse, const float* grad_logp,
                                const float* grad_entropy, void* grad_logits, int64_t grad_ld, int B, void* stream) {
    if (!policy_args_ok(offsets, actions_u64, cap, logits, dtype, ld, B) || !ids || !lse || !grad_logits) return DDZ_E_ARG;
    if (grad_ld < DDZ_NUM_ACTION_IDS || (reinterpret_cast<uintptr_t>(grad_logits) & (dtype == DDZ_DTYPE_F32 ? 3u : 1u)) != 0)
        return DDZ_E_ARG;
    const cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = policy_grid(B), threads = policy_head::kWarps * 32;
    if (dtype == DDZ_DTYPE_F32)
        policy_head::k_policy_logprob_backward<DDZ_DTYPE_F32><<<grid, threads, 0, st>>>(
            offsets, actions_u64, cap, logits, ld, ids, lse, grad_logp, grad_entropy, grad_logits, grad_ld, B);
    else
        policy_head::k_policy_logprob_backward<DDZ_DTYPE_BF16><<<grid, threads, 0, st>>>(
            offsets, actions_u64, cap, logits, ld, ids, lse, grad_logp, grad_entropy, grad_logits, grad_ld, B);
    DDZ_LAUNCH_CHECK("k_policy_logprob_backward");
    return 0;
}

// linear heads: hidden / weight (16-byte rows, H and ld whole 16-byte pieces, H <= 1024) and bias (element-aligned) of one dtype
static bool linear_head_ok(const void* hidden, const void* weight, const void* bias, int dtype, int H, int64_t ld) {
    if (!hidden || !weight || (dtype != DDZ_DTYPE_F32 && dtype != DDZ_DTYPE_BF16)) return false;
    const int esz = dtype == DDZ_DTYPE_F32 ? 4 : 2, vec = 16 / esz;
    if (H <= 0 || H > linear_head::kMaxHidden || H % vec != 0 || ld < H || ld % vec != 0) return false;
    return ((reinterpret_cast<uintptr_t>(hidden) | reinterpret_cast<uintptr_t>(weight)) & 15u) == 0 &&
           (reinterpret_cast<uintptr_t>(bias) & (uintptr_t)(esz - 1)) == 0;
}
static bool linear_args_ok(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* hidden,
                           const void* weight, const void* bias, int dtype, int H, int64_t ld, int B) {
    if (!offsets || B <= 0 || cap < 0 || (cap > 0 && !actions_u64)) return false;
    return linear_head_ok(hidden, weight, bias, dtype, H, ld);
}

int ddz_policy_linear_logits(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* hidden,
                             const void* weight, const void* bias, int dtype, int H, int64_t ld, float* out, int64_t* stats,
                             int B, void* stream) {
    if (!linear_args_ok(offsets, actions_u64, cap, hidden, weight, bias, dtype, H, ld, B) || (cap > 0 && !out)) return DDZ_E_ARG;
    by_dtype(dtype, [&](auto dt) {
        constexpr int DT = decltype(dt)::value;
        linear_head::k_linear_logits<DT><<<policy_grid(B), kLinearThreads, 0, (cudaStream_t)stream>>>(
            offsets, actions_u64, cap, linear_head::Head<DT>{hidden, weight, bias, H, ld}, out, stats, B);
    });
    DDZ_LAUNCH_CHECK("k_linear_logits");
    return 0;
}

int ddz_policy_linear_sample(void* state, const int32_t* offsets, const uint64_t* actions_u64, int64_t cap,
                             const void* hidden, const void* weight, const void* bias, int dtype, int H, int64_t ld,
                             float temperature, uint64_t seed, uint64_t env0, uint32_t stepno, const uint8_t* env_mask,
                             int32_t* choice, int32_t* ids, float* logp, float* entropy, int64_t* stats, int B, void* stream) {
    if (!linear_args_ok(offsets, actions_u64, cap, hidden, weight, bias, dtype, H, ld, B) || !choice || !ids || !logp ||
        !entropy)
        return DDZ_E_ARG;
    if (!(temperature >= 0.f) || !(temperature <= FLT_MAX)) return DDZ_E_ARG;              // NaN, negative or infinite
    uint32_t* meta = state ? reinterpret_cast<uint32_t*>(reinterpret_cast<uint64_t*>(state) + 9 * (size_t)B) : nullptr;
    by_dtype(dtype, [&](auto dt) {
        constexpr int DT = decltype(dt)::value;
        linear_head::k_linear_sample<DT><<<policy_grid(B), kLinearThreads, 0, (cudaStream_t)stream>>>(
            offsets, actions_u64, cap, linear_head::Head<DT>{hidden, weight, bias, H, ld}, temperature, seed, env0, stepno,
            env_mask, meta, choice, ids, logp, entropy, stats, B);
    });
    DDZ_LAUNCH_CHECK("k_linear_sample");
    return 0;
}

int ddz_policy_linear_logprob(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* hidden,
                              const void* weight, const void* bias, int dtype, int H, int64_t ld, const int32_t* ids,
                              float* logp, float* entropy, float* lse, int64_t* stats, int B, void* stream) {
    if (!linear_args_ok(offsets, actions_u64, cap, hidden, weight, bias, dtype, H, ld, B) || !ids || !logp || !entropy)
        return DDZ_E_ARG;
    by_dtype(dtype, [&](auto dt) {
        constexpr int DT = decltype(dt)::value;
        linear_head::k_linear_logprob<DT><<<policy_grid(B), kLinearThreads, 0, (cudaStream_t)stream>>>(
            offsets, actions_u64, cap, linear_head::Head<DT>{hidden, weight, bias, H, ld}, ids, logp, entropy, lse, stats, B);
    });
    DDZ_LAUNCH_CHECK("k_linear_logprob");
    return 0;
}

int ddz_policy_linear_backward(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, const void* hidden,
                               const void* weight, const void* bias, int dtype, int H, int64_t ld, const int32_t* ids,
                               const float* lse, const float* grad_logp, const float* grad_entropy, float* grad_legal,
                               void* grad_hidden, int64_t ld_g, int B, void* stream) {
    if (!linear_args_ok(offsets, actions_u64, cap, hidden, weight, bias, dtype, H, ld, B) || !ids || !lse || !grad_hidden ||
        (cap > 0 && !grad_legal))
        return DDZ_E_ARG;
    if (ld_g < H || ld_g % (dtype == DDZ_DTYPE_F32 ? 4 : 8) != 0 || (reinterpret_cast<uintptr_t>(grad_hidden) & 15u) != 0)
        return DDZ_E_ARG;
    by_dtype(dtype, [&](auto dt) {
        constexpr int DT = decltype(dt)::value;
        linear_head::k_linear_backward<DT><<<policy_grid(B), kLinearThreads, 0, (cudaStream_t)stream>>>(
            offsets, actions_u64, cap, linear_head::Head<DT>{hidden, weight, bias, H, ld}, ids, lse, grad_logp, grad_entropy,
            grad_legal, grad_hidden, ld_g, B);
    });
    DDZ_LAUNCH_CHECK("k_linear_backward");
    return 0;
}

size_t ddz_policy_linear_workspace_bytes(int64_t n, int H) {
    if (n <= 0 || H <= 0 || H > linear_head::kMaxHidden) return 0;
    const int64_t chunks = (n + linear_head::kChunk - 1) / linear_head::kChunk;
    return (size_t)chunks * 2 * ((size_t)H + 4) * sizeof(float);
}

int ddz_policy_linear_grad_weight(const int32_t* offsets, int64_t n, const void* hidden, int dtype, int H, int64_t ld,
                                  const float* grad_legal, const int32_t* order, const int32_t* id_offsets,
                                  void* grad_weight, void* grad_bias, void* workspace, int B, void* stream) {
    if (!offsets || B <= 0 || n < 0 || !grad_weight) return DDZ_E_ARG;
    if (n > 0 && (!grad_legal || !order || !id_offsets || !workspace)) return DDZ_E_ARG;
    if (!linear_head_ok(hidden, grad_weight, grad_bias, dtype, H, ld) || (reinterpret_cast<uintptr_t>(workspace) & 15u) != 0)
        return DDZ_E_ARG;
    const int64_t per_cta = (int64_t)linear_head::kChunk * linear_head::kWarps;
    float* ws = reinterpret_cast<float*>(workspace);
    by_dtype(dtype, [&](auto dt) {
        constexpr int DT = decltype(dt)::value;
        const cudaStream_t st = (cudaStream_t)stream;
        // the head's weight and bias are not read: the id of every entry comes from id_offsets
        const linear_head::Head<DT> hd{hidden, nullptr, nullptr, H, ld};
        if (n > 0)
            linear_head::k_linear_grad_chunks<DT><<<(unsigned)((n + per_cta - 1) / per_cta), kLinearThreads, 0, st>>>(
                offsets, B, n, hd, grad_legal, order, id_offsets, grad_weight, grad_bias, ws);
        linear_head::k_linear_grad_combine<DT><<<(DDZ_NUM_ACTION_IDS + linear_head::kWarps - 1) / linear_head::kWarps,
                                                 kLinearThreads, 0, st>>>(H, n > 0 ? id_offsets : nullptr, grad_weight,
                                                                          grad_bias, ws);
    });
    DDZ_LAUNCH_CHECK("k_linear_grad_chunks / k_linear_grad_combine");
    return 0;
}

}  // extern "C"
