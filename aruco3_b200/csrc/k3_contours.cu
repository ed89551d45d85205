// K3 — border following and quad filtering on the GPU (SURVEY.md 8f-1), sm_100a.  Compile with -fmad=false.
//
// Replaces, with identical results, the host stage (host_quads.cpp) and therefore
//   imageproc::contours::find_contours::<u32>                    call site /root/reference/src/aruco.rs:64
//   contours_to_candidates / enforce_clockwise_corners / discard_too_near   /root/reference/src/aruco.rs:124-232
// for every frame it does not flag; flagged frames are redone by the host stage.
//
// The reference algorithm (Suzuki-Abe with imageproc's start guards) is sequential: whether a pixel starts a border
// depends on labels written by borders followed earlier in raster order.  tools/contour_parallel_proto.py restates
// it without that dependence and checks the restatement against the oracle on random masks:
//   * a border is a closed chain of cracks (foreground pixel + a side with a background 4-neighbour); following it
//     from any of its cracks gives the same cyclic pixel sequence, because the step function reads no labels;
//   * start candidates are west cracks with x > 0 (the reference's "outer" rule) and east cracks with x + 1 < w
//     ("hole" rule); a border is followed exactly once, from its raster-first ELIGIBLE candidate;
//   * eligibility can differ from "first candidate" only in frames that contain a border whose first candidate is a
//     west crack that is not the raster-first pixel of that border (its natural start lies in column 0, where the
//     outer rule is barred).  Such frames are FLAGGED and left to the sequential host stage.
// So on the GPU every candidate decides alone: it walks its own border and survives iff it meets no raster-earlier
// candidate crack of that border.  West candidates walk backwards (the pixel above on a left edge is an earlier
// candidate: one step), east candidates forwards; only the one survivor of each border walks the full loop.
//
// Kernels:  k3_candidates (one thread per 32-pixel word of the 1-bit mask; every candidate walks at most kBudget steps:
// almost all die within a few, short borders finish)  ->  k3_walkers (one thread per undecided candidate: the long
// borders, all in flight at once)  ->  the surviving long borders put in raster order of their starts (= the reference's
// discovery order): k3_order ranks them frame by frame, a radix sort takes over when a frame has more than its list holds
// ->  k3_emit (one thread per border writes its points)  ->  k3_rdp (one
// warp per border: Ramer-Douglas-Peucker, hull, edge test)  ->  k3_finalize (one warp per frame: ordered compaction,
// clockwise, discard_too_near).
// Calls of up to 16 frames walk differently (their time is the chain of the longest border, not throughput): every border that
// owns a candidate crack on a relay row (every 16th) is walked from ALL those cracks at once (k3_segments), the relays of a border
// are linked into a cycle whose smallest candidate key is the border's start (k3_jumps, k3_cycles, k3_spread), and the candidate walks above keep only
// the borders between two relay rows.  tools/relay_proto.py is the specification, tests/test_relay_proto.py checks it.
#include <cooperative_groups.h>
#include <cooperative_groups/scan.h>
#include <cub/device/device_radix_sort.cuh>

#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <optional>

#include "a3_internal.h"

namespace a3 {
namespace {

namespace cg = cooperative_groups;

constexpr int kDx[8] = {-1, -1, 0, 1, 1, 1, 0, -1};  // ring order w nw n ne e se s sw (screen clockwise)
constexpr int kDy[8] = {0, -1, -1, -1, 0, 1, 1, 1};

// step table entry: bits 0-2 direction of the next pixel, bit 3 west side examined, bit 4 east side examined,
// bits 5-6 dx + 1, bits 7-8 dy + 1, bits 10-12 state at the next pixel (direction back to this one): e & 0x1c00 is the byte
// offset of that state's row of 512 entries
struct StepTables {
    uint16_t fwd[8][512];  // [ring direction of the previous border pixel][3x3 neighbourhood]
    uint16_t bwd[8][512];  // [ring direction of the next border pixel][3x3 neighbourhood]
};

uint32_t ring_of_host(uint32_t hood9) {
    const uint32_t t = hood9 & 7u, m = (hood9 >> 3) & 7u, b = hood9 >> 6;
    return (m & 1u) | ((t & 1u) << 1) | ((t & 2u) << 1) | ((t & 4u) << 1) | ((m & 4u) << 2) | ((b & 4u) << 3) | ((b & 2u) << 5) | ((b & 1u) << 7);
}

void build_tables(StepTables &t) {
    for (int state = 0; state < 8; state++)
        for (int hood = 0; hood < 512; hood++) {
            const uint32_t nb = ring_of_host((uint32_t)hood);
            for (int back = 0; back < 2; back++) {
                int d = state;
                uint32_t examined = 0;
                for (int k = 1; k <= 7; k++) {
                    const int c = back ? (state + k) & 7 : (state - k) & 7;
                    if ((nb >> c) & 1) { d = c; break; }
                    examined |= 1u << c;
                }
                const uint16_t e = (uint16_t)(d | (((examined >> 0) & 1u) << 3) | (((examined >> 4) & 1u) << 4) | ((kDx[d] + 1) << 5) |
                                              ((kDy[d] + 1) << 7) | (((d + 4) & 7) << 10));
                (back ? t.bwd : t.fwd)[state][hood] = e;
            }
        }
}

__device__ __forceinline__ int ddx(int d) { return (d >= 3 && d <= 5) ? 1 : ((d == 2 || d == 6) ? 0 : -1); }
__device__ __forceinline__ int ddy(int d) { return (d >= 1 && d <= 3) ? -1 : ((d == 0 || d == 4) ? 0 : 1); }

struct Geo {
    const uint32_t *planes;  // guarded column-major bit planes: frame f at planes + f * frame_words, pixel (x, y) = bit x & 31 of
                             // word ((x >> 5) + 1) * Hp + (y + 1)
    uint32_t n, w, h, wpr, Hp;
    size_t frame_words;
};

// 3x3 neighbourhood of (x, y): bits 0-2 row y-1, 3-5 row y, 6-8 row y+1 (bit 0 of each = column x-1)
__device__ __forceinline__ uint32_t hood9(const uint32_t *plane, uint32_t Hp, int x, int y) {
    const int o = x + 31;                                   // column x-1 in guarded coordinates
    const uint32_t *p = plane + ((uint32_t)(o >> 5) * Hp + (uint32_t)y);  // word column of x-1, row y-1 (guarded row index y); < 2^28 words
    const int sh = o & 31;
    uint32_t t = __ldg(p) >> sh, m = __ldg(p + 1) >> sh, b = __ldg(p + 2) >> sh;
    if (sh > 29) {  // the three columns straddle two words
        const uint32_t *q = p + Hp;
        t |= __ldg(q) << (32 - sh); m |= __ldg(q + 1) << (32 - sh); b |= __ldg(q + 2) << (32 - sh);
    }
    return (t & 7u) | ((m & 7u) << 3) | ((b & 7u) << 6);
}
__device__ __forceinline__ uint32_t ring_of(uint32_t hood) {
    const uint32_t t = hood & 7u, m = (hood >> 3) & 7u, b = hood >> 6;
    return (m & 1u) | ((t & 1u) << 1) | ((t & 2u) << 1) | ((t & 4u) << 1) | ((m & 4u) << 2) | ((b & 4u) << 3) | ((b & 2u) << 5) | ((b & 1u) << 7);
}

// The same neighbourhood for k3_emit: a border moves one pixel per step, so the three words of the current word column
// (and, next to a 32-pixel boundary, of the following one) stay in registers; a step that keeps its row loads nothing,
// a step that changes row loads one word (two at a boundary).  A warp's lanes walk 32 different borders, so every load
// is 32 separate L1 wavefronts, and with one thread per segment k3_emit is bound by exactly those (measured: the first
// walks, which are bound by the latency of the longest chain instead, get slower with the extra branches).
struct Window {
    const uint32_t *plane;
    uint32_t Hp;
    int kc, yg;            // guarded word column of pixel x-1; guarded row of y-1 (== y)
    uint32_t t, m, b;      // column kc, rows y-1, y, y+1
    uint32_t t2, m2, b2;   // column kc+1, valid where v2 has bit 0 / 1 / 2
    uint32_t v2;
};
__device__ __forceinline__ void win_load(Window &w, int x, int y) {
    w.kc = (x + 31) >> 5; w.yg = y;
    const uint32_t *p = w.plane + (size_t)w.kc * w.Hp + y;
    w.t = __ldg(p); w.m = __ldg(p + 1); w.b = __ldg(p + 2);
    w.v2 = 0;
}
__device__ __forceinline__ uint32_t win_hood(Window &w, int x) {
    const int sh = (x + 31) & 31;
    uint32_t t = w.t >> sh, m = w.m >> sh, b = w.b >> sh;
    if (sh > 29) {
        if (w.v2 != 7u) {
            const uint32_t *q = w.plane + (size_t)(w.kc + 1) * w.Hp + w.yg;
            if (!(w.v2 & 1u)) w.t2 = __ldg(q);
            if (!(w.v2 & 2u)) w.m2 = __ldg(q + 1);
            if (!(w.v2 & 4u)) w.b2 = __ldg(q + 2);
            w.v2 = 7u;
        }
        t |= w.t2 << (32 - sh); m |= w.m2 << (32 - sh); b |= w.b2 << (32 - sh);
    }
    return (t & 7u) | ((m & 7u) << 3) | ((b & 7u) << 6);
}
// the walk moved to (x, y), at most one pixel away in each direction
__device__ __forceinline__ void win_move(Window &w, int x, int y) {
    const int kc = (x + 31) >> 5, dy = y - w.yg;
    if (kc != w.kc) {
        if (dy == 0 && kc == w.kc + 1 && w.v2 == 7u) {         // the following column becomes the current one
            w.t = w.t2; w.m = w.m2; w.b = w.b2; w.v2 = 0; w.kc = kc;
        } else if (dy == 0 && kc == w.kc - 1) {                // the current column becomes the following one
            w.t2 = w.t; w.m2 = w.m; w.b2 = w.b; w.v2 = 7u; w.kc = kc;
            const uint32_t *p = w.plane + (size_t)kc * w.Hp + y;
            w.t = __ldg(p); w.m = __ldg(p + 1); w.b = __ldg(p + 2);
        } else {
            win_load(w, x, y);
        }
    } else if (dy > 0) {
        w.t = w.m; w.m = w.b; w.b = __ldg(w.plane + (size_t)kc * w.Hp + y + 2);
        w.t2 = w.m2; w.m2 = w.b2; w.v2 >>= 1;
        w.yg = y;
    } else if (dy < 0) {
        w.b = w.m; w.m = w.t; w.t = __ldg(w.plane + (size_t)kc * w.Hp + y);
        w.b2 = w.m2; w.m2 = w.t2; w.v2 = (w.v2 << 1) & 7u;
        w.yg = y;
    }
}

constexpr uint32_t kBudget = 48;  // steps a candidate may walk inside k3_candidates before it is deferred to k3_walkers
// A walk is a chain of dependent loads: its time is its length.  The long walks (k3_walkers) are done by a PAIR of lanes
// that leave the start pixel in opposite directions and stop where they meet, which halves the chain; while they walk
// they drop a checkpoint every kSeg points, and k3_emit then writes the points with one thread per checkpoint: chains of
// kSeg steps instead of the longest border.
constexpr uint32_t kSeg = 64;
static_assert(kBudget < kSeg, "borders finished inside the budget must fit one emit segment");
// pos: forward index of the checkpoint's pixel, or (kCkptBackward set in `state`) its distance from the END of the border;
// state: the forward state there (direction of the previous border pixel)
struct Ckpt { uint32_t walker, pos, xy, state; };
constexpr uint32_t kCkptBackward = 0x80000000u;

enum { kDead = 0, kSurvivor = 1, kUndecided = 2 };
// slots of Lists::counters
constexpr uint32_t kNumWalkers = 0;    // entries of `walkers`
constexpr uint32_t kNumLong = 1;       // long borders
constexpr uint32_t kOverflow = 2;      // non-zero: a list overflowed
constexpr uint32_t kNumCands = 3;      // entries of `cands`
constexpr uint32_t kNumCkpts = 4;      // checkpoints
constexpr uint32_t kSpecFail = 5;      // the speculative finish gave up (k3_spec_prepare)
constexpr uint32_t kNumRelays = 6;     // relay cracks
constexpr uint32_t kMaxFrameLong = 7;  // most long borders in one frame

// Work lists shared by the kernels of one k3_quads call.
struct Lists {
    unsigned long long *cands;         // start candidates left after the word-level filter: ((word id * 32 + bit) << 1) | kind
    uint32_t cands_cap;
    unsigned long long *walkers;       // candidates undecided after kBudget steps: the same key
    unsigned long long *long_keys;     // surviving borders with >= min_points points: the same key ...
    uint32_t *long_n;                  // ... and their number of points
    uint32_t *counters;                // 8 words, slots kNumWalkers ... kMaxFrameLong
    uint32_t *long_slot;               // value array of the sort: the border's slot in long_keys / long_n
    uint32_t *walker_slot;             // per entry of `walkers`: slot of the border it survived as, or 0xffffffff
    Ckpt *ckpts;                       // checkpoints dropped by k3_walkers
    uint32_t ckpt_cap;
    unsigned long long *long_points;   // total points of the long borders
    uint32_t walkers_cap, long_cap;
    uint32_t *frame_contours;          // per frame: borders followed
    unsigned long long *frame_points;  // per frame: their points
    uint32_t *frame_flags;             // per frame: bit 0 barred start (host redo), bit 1 rdp stack overflow, bit 2 quad capacity
    uint32_t *long_off_slot;           // per slot of long_keys: where the border's points go (allocated with one atomic add)
    // the same long borders listed per frame, frame_cap entries each (0 = not kept): what k3_order ranks; counters[kMaxFrameLong] = the
    // largest number of long borders any frame has
    uint32_t frame_cap;
    uint32_t *frame_long_count;
    unsigned long long *frame_keys;
    uint32_t *frame_slots;
    // relays (tools/relay_proto.py is the spec): the west / east cracks on every (1 << relay_shift)-th row.  counters[kNumRelays] = how many
    uint2 *relays;                     // per relay crack: {x | y << 16, frame << 1 | side (0 west, 1 east)}
    struct Seg *segs;                  // per relay crack: its segment of the border (k3_segments), then its place in it (k3_cycles)
    uint32_t *relay_base;              // per (frame, relay row, word column): index of the word's first relay crack
    unsigned long long *seg_owner;     // per relay crack: (leader of its cycle << 32) | visits of the cycle before its segment (k3_cycles)
    struct Jump *jumps;                // per relay crack: the next `jump_hops` segments summed up (k3_jumps)
    unsigned long long *anchor_owner;  // per relay crack a walker of k3_cycles jumped from: (walker << 32) | visits so far (k3_spread hands it on)
    uint32_t jump_hops;
    uint32_t relay_cap;                // 0 = relays off
    uint32_t relay_shift, nrr;         // log2 of the row spacing; relay rows per frame
};
// One relay's segment: the visits from its own up to (not including) the next relay visit of the border.
struct __align__(16) Seg {
    uint32_t next;       // index of the relay crack that names the next relay visit
    uint32_t len;        // visits in the segment; 0 = not a relay (an isolated pixel, or an east crack whose visit owns a west crack too)
    uint32_t cand;       // smallest candidate key (pixel << 1 | kind) among the segment's visits, 0xffffffff = none
    uint32_t cand_pos;   // index of that visit within the segment
    uint32_t min_pix;    // raster-first pixel of the segment
    uint32_t slot;       // k3_cycles, in the record of the cycle's leader: slot of the border among the long borders, 0xffffffff = not recorded
    uint32_t off;        // k3_cycles, in the leader's record: index of the border's start visit, counted from the leader's own visit
    uint32_t state;      // state of the relay's own visit
};
// The next `hops` segments after a relay, summed up: a cycle of k segments is then followed in k / hops dependent steps.
struct __align__(16) Jump {
    uint32_t dest;       // the relay after them
    uint32_t len;        // their visits
    uint32_t cand;       // smallest candidate key among them, 0xffffffff = none
    uint32_t cand_off;   // index of that visit, counted from the first of them
    uint32_t min_pix;    // raster-first pixel among them
    uint32_t min_idx;    // smallest index among the relays landed on or passed (the start excluded, dest included)
    uint32_t pad0, pad1;
};
constexpr uint32_t kNone = 0xffffffffu;
constexpr uint32_t kRelayFlag = 0x80000000u;  // in long_n: the border's points come from relay segments


// 3x3 neighbourhood of the pixel at guarded column o = x + 31, row y, times two (the byte offset of its entry in a row of the
// step tables): three loads from one word column, the second column only when the three pixel columns straddle two words
__device__ __forceinline__ uint32_t hood2(const uint32_t *plane, uint32_t Hp, int o, int y) {
    const uint32_t *p = plane + ((uint32_t)(o >> 5) * Hp + (uint32_t)y);
    const int sh = o & 31;
    uint32_t t = __ldg(p), m = __ldg(p + 1), b = __ldg(p + 2), t2 = 0, m2 = 0, b2 = 0;
    if (sh > 29) {
        const uint32_t *q = p + Hp;
        t2 = __ldg(q); m2 = __ldg(q + 1); b2 = __ldg(q + 2);
    }
    t = __funnelshift_r(t, t2, sh); m = __funnelshift_r(m, m2, sh); b = __funnelshift_r(b, b2, sh);
    return ((t << 1) & 0x00eu) | ((m << 4) & 0x070u) | ((b << 7) & 0x380u);
}

// The candidate (x, y, kind) walks its border for at most `budget` steps.  kSurvivor: it is the raster-first candidate
// crack of the border (n = number of points of the border, first_pixel = it is also the border's raster-first pixel).
// rmask: a visit that owns a west or east crack on a row y & rmask == 0 is a relay visit — its border belongs to k3_segments /
// k3_cycles, so the candidate gives up (kDead) there (template relay_on: the batch route compiles none of it).
template <bool relay_on>
__device__ int walk_border(const uint32_t *plane, const Geo &g, const uint16_t (*fwd)[512], const uint16_t (*bwd)[512], int sx, int sy, int kind,
                           uint32_t budget, uint32_t &n, bool &first_pixel, uint32_t rmask) {
    const int w = (int)g.w, o_max = w + 30;
    const uint32_t start_pix = (uint32_t)(sy * w + sx);
    const uint32_t me = (start_pix << 1) | (uint32_t)kind;
    const uint32_t nb0 = ring_of(hood9(plane, g.Hp, sx, sy));
    const int adj = kind ? 4 : 0;
    int pred = -1;
    for (int k = 0; k < 8; k++) {  // clockwise from the zero neighbour: the previous pixel on the border
        const int d = (adj + k) & 7;
        if ((nb0 >> d) & 1) { pred = d; break; }
    }
    n = 1;
    first_pixel = true;
    if (pred < 0) return (kind == 0 || sx == 0) ? kSurvivor : kDead;  // isolated pixel: its west crack (if a candidate) comes first
    if (relay_on && ((uint32_t)sy & rmask) == 0u) return kDead;       // my own crack is a relay crack: a relay border
    // position as (o = x + 31, y, pix = y w + x), state as the byte offset of its table row (see k3_walkers)
    uint32_t min_pix = start_pix, pix = start_pix, state_off;
    int o = sx + 31, y = sy;
    if (kind) {  // forwards from the start pixel, previous pixel in direction `pred` (this is the reference's own trace)
        state_off = (uint32_t)pred << 10;
        n = 0;
    } else {     // backwards: the start pixel's own visit owns the west crack and nothing raster-earlier
        o += ddx(pred); y += ddy(pred); pix = (uint32_t)(y * w + o - 31); state_off = (uint32_t)((pred + 4) & 7) << 10;
    }
    const unsigned char *lut = reinterpret_cast<const unsigned char *>(kind ? &fwd[0][0] : &bwd[0][0]);
    // a candidate crack of a visit comes before me in raster order:  west  2 pix < me  <=>  pix < tw;  east  2 pix + 1 < me  <=>  pix < te
    const uint32_t tw = (me + 1u) >> 1, te = me >> 1, pred_off = (uint32_t)pred << 10;
    for (uint32_t steps = 0;; steps++) {
        const uint32_t e = *reinterpret_cast<const uint16_t *>(lut + state_off + hood2(plane, g.Hp, o, y));
        if (kind) {
            if (n && pix == start_pix && state_off == pred_off) break;  // back in the starting state
        } else {
            if (pix == start_pix && (e & 8u)) break;                     // back at the visit that owns the west crack
        }
        if (relay_on && ((uint32_t)y & rmask) == 0u && (((e & 8u) && o > 31) || ((e & 16u) && o < o_max))) return kDead;  // a relay border
        // candidate cracks of this visit that come before me in raster order (west needs x > 0, east x + 1 < w)
        if ((e & 8u) && o > 31 && pix < tw) return kDead;
        if ((e & 16u) && o < o_max && pix < te) return kDead;
        if (steps >= budget) return kUndecided;
        min_pix = min(min_pix, pix);
        n++;
        const int dx = (int)((e >> 5) & 3u) - 1, dy = (int)((e >> 7) & 3u) - 1;
        o += dx; y += dy;
        pix += (uint32_t)(dy * w + dx);
        state_off = e & 0x1c00u;
    }
    first_pixel = min_pix == start_pix;
    return kSurvivor;
}

__device__ __forceinline__ uint32_t record_survivor(const Lists &l, uint32_t frame, unsigned long long key, int kind, uint32_t n, bool first_pixel,
                                                    uint32_t min_points, bool relay = false) {
    atomicAdd(&l.frame_contours[frame], 1u);
    atomicAdd(&l.frame_points[frame], (unsigned long long)n);
    if (kind == 0 && !first_pixel) atomicOr(&l.frame_flags[frame], 1u);  // a west start below the top of its border: barred natural start
    if (n >= min_points && n >= 4) {
        const uint32_t slot = atomicAdd(&l.counters[kNumLong], 1u);
        if (slot < l.long_cap) {
            l.long_keys[slot] = key;
            l.long_n[slot] = relay ? (n | kRelayFlag) : n;
            l.long_slot[slot] = slot;
            l.long_off_slot[slot] = (uint32_t)atomicAdd(l.long_points, (unsigned long long)n);  // totals beyond 32 bits flag the whole call
            if (l.frame_cap) {
                const uint32_t j = atomicAdd(&l.frame_long_count[frame], 1u);
                if (j < l.frame_cap) {
                    l.frame_keys[(size_t)frame * l.frame_cap + j] = key;
                    l.frame_slots[(size_t)frame * l.frame_cap + j] = slot;
                }
                atomicMax(&l.counters[kMaxFrameLong], j + 1);
            }
            return slot;
        }
        atomicOr(&l.counters[kOverflow], 1u);
    }
    return 0xffffffffu;
}

template <bool RELAY>
__global__ void __launch_bounds__(256) k3_candidates(const Geo g, const StepTables *tables, const uint32_t min_points, const Lists l) {
    __shared__ uint16_t fwd[8][512];  // only for candidates that do not fit the list (walked right here)
    __shared__ uint16_t bwd[8][512];
    for (int i = threadIdx.x; i < 8 * 512; i += blockDim.x) {
        (&fwd[0][0])[i] = (&tables->fwd[0][0])[i];
        (&bwd[0][0])[i] = (&tables->bwd[0][0])[i];
    }
    __syncthreads();
    const uint32_t words_per_frame = g.h * g.wpr;
    // The scan is a stream of dependent loads with almost no work behind them (most words have no crack at all), so each
    // thread first issues the loads of kBatch words (the word and its two horizontal neighbours) and only then looks at them.
    // Index space without divisions: a block takes whole word columns k (blockIdx.x strides over them), its threads take
    // consecutive rows y of the column (consecutive words of the column-major plane), kBatch rows per thread and pass.
    constexpr int kBatch = 4;
    const uint32_t stride = blockDim.x;
    const uint32_t last_k = (g.w - 1) >> 5, last_bit = (g.w - 1) & 31;
    for (uint32_t frame = blockIdx.y; frame < g.n; frame += gridDim.y)
    for (uint32_t k = blockIdx.x; k < g.wpr; k += gridDim.x)
    for (uint32_t base0 = blockIdx.z * stride * kBatch; base0 < g.h; base0 += gridDim.z * stride * kBatch) {  // warp-uniform trip count: rows beyond h read as empty words
        const uint32_t base = base0 + threadIdx.x;
        const uint32_t *plane = g.planes + (size_t)frame * g.frame_words;
        const uint32_t *colk = plane + (size_t)(k + 1) * g.Hp + 1;  // row 0 of word column k
        uint32_t fv[kBatch], og[kBatch], hg[kBatch], av[kBatch], awv[kBatch], aev[kBatch];
        // phase 1: the word and its two horizontal neighbours -> west / east cracks that may start a border
        {
            uint32_t lv[kBatch], rv[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; u++) {
                const uint32_t y = base + (uint32_t)u * stride;
                fv[u] = 0; lv[u] = 0; rv[u] = 0;
                if (y < g.h) {
                    const uint32_t *col = colk + y;
                    fv[u] = __ldg(col); lv[u] = __ldg(col - g.Hp); rv[u] = __ldg(col + g.Hp);
                }
            }
#pragma unroll
            for (int u = 0; u < kBatch; u++) {
                const uint32_t f = fv[u];
                og[u] = f & ~((f << 1) | (lv[u] >> 31));
                hg[u] = f & ~((f >> 1) | (rv[u] << 31));
                if (k == 0) og[u] &= ~1u;                        // `x > 0`
                if (k == last_k) hg[u] &= ~(1u << last_bit);     // `x + 1 < w`
                // relay rows: every candidate crack of the row (west with x > 0, east with x + 1 < w) is listed; the entries of a word are
                // consecutive, in the order (bit, west before east), and the word's first index is kept for k3_segments' lookups
                const uint32_t y = base + (uint32_t)u * stride;
                if (RELAY && (og[u] | hg[u]) && (y & ((1u << l.relay_shift) - 1u)) == 0u) {
                    const uint32_t cnt = (uint32_t)(__popc(og[u]) + __popc(hg[u]));
                    uint32_t j = atomicAdd(&l.counters[kNumRelays], cnt);
                    l.relay_base[((size_t)frame * l.nrr + (y >> l.relay_shift)) * g.wpr + k] = j;
                    if (j + cnt <= l.relay_cap) {
                        for (uint32_t pending = og[u] | hg[u]; pending; pending &= pending - 1) {
                            const uint32_t bit = (uint32_t)__ffs(pending) - 1u, xy = (k * 32 + bit) | (y << 16);
                            if ((og[u] >> bit) & 1u) l.relays[j++] = make_uint2(xy, frame << 1);
                            if ((hg[u] >> bit) & 1u) l.relays[j++] = make_uint2(xy, (frame << 1) | 1u);
                        }
                    } else {
                        atomicOr(&l.counters[kOverflow], 1u);
                    }
                }
            }
        }
        // phase 2: the row above (three words) of the words that have such cracks, all loads first
#pragma unroll
        for (int u = 0; u < kBatch; u++) {
            av[u] = 0; awv[u] = 0; aev[u] = 0;
            if (og[u] | hg[u]) {
                const uint32_t *col = colk + (base + (uint32_t)u * stride);
                av[u] = __ldg(col - 1); awv[u] = __ldg(col - g.Hp - 1); aev[u] = __ldg(col + g.Hp - 1);   // row y-1 (guard row for y = 0)
            }
        }
        uint32_t mine = 0;
#pragma unroll
        for (int u = 0; u < kBatch; u++) {
            if (!(og[u] | hg[u])) continue;
            // Most candidates have a raster-earlier candidate crack of the same border right above them; word arithmetic
            // on the row above finds those without walking (each rule names a crack that is on the same border because
            // the background pixels involved are 4-connected and the foreground pixels 8-connected):
            //   west crack at (x, y):  (x, y-1) also has a west crack                       (straight left edge)
            //                          N and NW are background, NE is foreground: (x+1, y-1) has a west crack ('/' edge)
            //   east crack at (x, y):  (x, y-1) also has an east crack                      (straight right edge)
            //                          N and NE are background, NW is foreground: (x-1, y-1) has an east crack ('\' edge)
            const uint32_t f = fv[u], fa = av[u];
            const uint32_t fa_w = (fa << 1) | (awv[u] >> 31);                      // bit x = pixel (x-1, y-1)
            const uint32_t fa_e = (fa >> 1) | (aev[u] << 31);                      // bit x = pixel (x+1, y-1)
            og[u] &= ~((fa & ~fa_w) | (~fa & ~fa_w & fa_e));
            hg[u] &= ~((fa & ~fa_e) | (~fa & ~fa_e & fa_w));
            // The same two ideas over runs instead of single pixels (stair steps of shallow edges), inside this word; a run
            // that leaves the word is simply not used.  runs(P, S): all bits of the runs of ones of P whose lowest bit is in S
            // (the carry of P + S sweeps each such run).
            //   background run below foreground:  P  = above F, here B;  it ends (on one side) at a pixel that is B in both
            //     rows (T): the foreground pixel of the row above next to T has a west / east crack, and both background
            //     chains are 4-connected through the run.
            //   foreground run below background:  P2 = above B, here F;  it ends at a pixel whose upper neighbour is F: that
            //     pixel has a west / east crack towards the run (needs NW / NE background for the connection).
            auto runs = [](uint32_t P, uint32_t S) { return ((P + (S & P)) ^ P) & P; };
            const uint32_t valid = (k == last_k) ? (0xffffffffu >> (31 - last_bit)) : 0xffffffffu;  // real pixels of this word
            const uint32_t P = fa & ~f, T = ~fa & ~f & valid, P2 = ~fa & f;
            const uint32_t rP = __brev(P), rP2 = __brev(P2);
            og[u] &= ~(runs(P, T << 1) << 1);                                  // west crack right of a P run that starts right of a T
            og[u] &= ~(__brev(runs(rP2, __brev(fa) << 1)) & ~fa_w);            // west crack at the low end of a P2 run that ends below an F
            hg[u] &= ~(__brev(runs(rP, __brev(T) << 1)) >> 1);                 // east crack left of a P run that ends left of a T
            hg[u] &= ~(runs(P2, fa << 1) & ~fa_e);                             // east crack at the high end of a P2 run that starts below an F
            mine += __popc(og[u]) + __popc(hg[u]);
        }
        // what is left goes to the candidate list (one atomic per warp and batch); k3_walk_short gives every entry a thread.
        // Every lane of the warp is here (uniform trip counts, whole warps), so the prefix is a plain shuffle scan.
        __syncwarp();
        if (!__any_sync(0xffffffffu, mine != 0)) continue;
        const int lane = threadIdx.x & 31;
        uint32_t incl = mine;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t up = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += up;
        }
        uint32_t first = 0;
        if (lane == 31) first = atomicAdd(&l.counters[kNumCands], incl);
        first = __shfl_sync(0xffffffffu, first, 31);
        uint32_t slot = first + incl - mine;
        if (!mine) continue;
#pragma unroll
        for (int u = 0; u < kBatch; u++) {
            if (!(og[u] | hg[u])) continue;
            const uint32_t y = base + (uint32_t)u * stride;
            const unsigned long long gid = (unsigned long long)frame * words_per_frame + (unsigned long long)y * g.wpr + k;  // raster word id: the sort key
            // raster order inside the word: by bit, west before east
            for (uint32_t pending = og[u] | hg[u]; pending; pending &= pending - 1) {
                const uint32_t bit = (uint32_t)__ffs(pending) - 1u;
                for (uint32_t kind = 0; kind < 2; kind++) {
                    if (!(((kind ? hg[u] : og[u]) >> bit) & 1u)) continue;
                    const unsigned long long key = (((gid << 5) | bit) << 1) | kind;
                    if (slot < l.cands_cap) {
                        l.cands[slot] = key;
                    } else {  // list full (very dense noise): walk it here, same rules as k3_walk_short
                        uint32_t n;
                        bool first_pixel;
                        const int r = walk_border<RELAY>(plane, g, fwd, bwd, (int)(k * 32 + bit), (int)y, (int)kind, kBudget, n, first_pixel, (1u << l.relay_shift) - 1u);
                        if (r == kSurvivor) {
                            record_survivor(l, frame, key, (int)kind, n, first_pixel, min_points);
                        } else if (r == kUndecided) {
                            const uint32_t ws = atomicAdd(&l.counters[kNumWalkers], 1u);
                            if (ws < l.walkers_cap) l.walkers[ws] = key;
                            else atomicOr(&l.counters[kOverflow], 1u);
                        }
                    }
                    slot++;
                }
            }
        }
    }
}

__device__ __forceinline__ void decode_key(const Geo &g, unsigned long long key, uint32_t &frame, int &x, int &y, int &kind) {
    kind = (int)(key & 1ull);
    const unsigned long long v = key >> 1;
    const unsigned long long gid = v >> 5;
    const size_t words_per_frame = (size_t)g.h * g.wpr;
    uint32_t rem;
    if ((gid >> 32) == 0 && (words_per_frame >> 32) == 0) {  // the usual case: a 32-bit division instead of the 64-bit routine
        frame = (uint32_t)gid / (uint32_t)words_per_frame;
        rem = (uint32_t)gid - frame * (uint32_t)words_per_frame;
    } else {
        frame = (uint32_t)(gid / words_per_frame);
        rem = (uint32_t)(gid % words_per_frame);
    }
    y = (int)(rem / g.wpr);
    x = (int)((rem % g.wpr) * 32 + (uint32_t)(v & 31ull));
}

// One thread per listed candidate: walk at most kBudget steps.  Nearly all die within a few; short borders finish.
template <bool RELAY>
__global__ void __launch_bounds__(128) k3_walk_short(const Geo g, const StepTables *tables, const uint32_t min_points, const Lists l) {
    __shared__ uint16_t fwd[8][512];
    __shared__ uint16_t bwd[8][512];
    for (int i = threadIdx.x; i < 8 * 512; i += blockDim.x) {
        (&fwd[0][0])[i] = (&tables->fwd[0][0])[i];
        (&bwd[0][0])[i] = (&tables->bwd[0][0])[i];
    }
    __syncthreads();
    const uint32_t total = min(l.counters[kNumCands], l.cands_cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const unsigned long long key = l.cands[i];
        uint32_t frame, n;
        int x, y, kind;
        bool first_pixel;
        decode_key(g, key, frame, x, y, kind);
        const uint32_t *plane = g.planes + (size_t)frame * g.frame_words;
        const int r = walk_border<RELAY>(plane, g, fwd, bwd, x, y, kind, kBudget, n, first_pixel, (1u << l.relay_shift) - 1u);
        if (r == kSurvivor) {
            record_survivor(l, frame, key, kind, n, first_pixel, min_points);
        } else if (r == kUndecided) {
            const uint32_t slot = atomicAdd(&l.counters[kNumWalkers], 1u);
            if (slot < l.walkers_cap) l.walkers[slot] = key;
            else atomicOr(&l.counters[kOverflow], 1u);
        }
    }
}

// Index of the relay crack (x, y, side) of `frame`: the word's first index + the number of relay cracks before it in the word.
__device__ __forceinline__ uint32_t relay_index(const Lists &l, const Geo &g, const uint32_t *plane, uint32_t frame, int x, int y, uint32_t side) {
    const uint32_t k = (uint32_t)x >> 5, bit = (uint32_t)x & 31u;
    const uint32_t *p = plane + ((size_t)(k + 1) * g.Hp + (uint32_t)y + 1u);
    const uint32_t f = __ldg(p), lv = __ldg(p - g.Hp), rv = __ldg(p + g.Hp);
    uint32_t rw = f & ~((f << 1) | (lv >> 31)), re = f & ~((f >> 1) | (rv << 31));
    if (k == 0) rw &= ~1u;                                            // candidates only: west with x > 0,
    if (k == ((g.w - 1) >> 5)) re &= ~(1u << ((g.w - 1) & 31u));      // east with x + 1 < w
    const uint32_t below = (1u << bit) - 1u;
    return l.relay_base[((size_t)frame * l.nrr + ((uint32_t)y >> l.relay_shift)) * g.wpr + k] + (uint32_t)__popc(rw & below) + (uint32_t)__popc(re & below) +
           ((side && ((rw >> bit) & 1u)) ? 1u : 0u);
}

// Relay walks (spec and proof by test: tools/relay_proto.py).  A border's time used to be the chain of half its visits (a pair
// of lanes per border); with a walker per relay crack it is the longest stretch between two relay rows.  One thread per listed
// crack: find the visit that owns it (an east crack whose visit owns a west crack too is an alias and drops out), follow the
// border to the next relay visit and record where that is, how many visits lie between, the raster-first candidate crack among
// them and its position, and the raster-first pixel.
__global__ void __launch_bounds__(128) k3_segments(const Geo g, const StepTables *tables, const Lists l) {
    __shared__ uint16_t fwd[8][512];
    for (int i = threadIdx.x; i < 8 * 512; i += blockDim.x) (&fwd[0][0])[i] = (&tables->fwd[0][0])[i];
    __syncthreads();
    if (l.counters[kNumRelays] > l.relay_cap) return;  // the list overflowed: every frame of the call goes to the host stage
    const uint32_t total = l.counters[kNumRelays], rmask = (1u << l.relay_shift) - 1u;
    const unsigned char *lut = reinterpret_cast<const unsigned char *>(&fwd[0][0]);
    const int w = (int)g.w, o_max = w + 30;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const uint2 r = l.relays[i];
        const int sx = (int)(r.x & 0xffffu), sy = (int)(r.x >> 16);
        const uint32_t frame = r.y >> 1, side = r.y & 1u;
        const uint32_t *plane = g.planes + (size_t)frame * g.frame_words;
        asm volatile("" : "+l"(plane));
        const uint32_t nb0 = ring_of(hood9(plane, g.Hp, sx, sy));
        const int adj = side ? 4 : 0;
        int pred = -1;
        for (int k = 0; k < 8; k++) {  // clockwise from the crack's side: the state of the visit that owns it
            const int d = (adj + k) & 7;
            if ((nb0 >> d) & 1) { pred = d; break; }
        }
        Seg out;
        out.next = i; out.len = 0; out.cand = kNone; out.cand_pos = 0; out.min_pix = kNone; out.slot = kNone; out.off = 0; out.state = 0;
        l.seg_owner[i] = ~0ull;
        l.anchor_owner[i] = ~0ull;
        int o = sx + 31, y = sy;
        uint32_t pix = (uint32_t)(sy * w + sx), state_off = (uint32_t)(pred < 0 ? 0 : pred) << 10;
        uint32_t e = *reinterpret_cast<const uint16_t *>(lut + state_off + hood2(plane, g.Hp, o, y));
        if (pred < 0 || (side && (e & 8u) && o > 31)) {  // an isolated pixel has no visits; the west crack names a visit that owns both
            l.segs[i] = out;
            continue;
        }
        uint32_t t = 0, best = kNone, best_pos = 0, min_pix = kNone;
        for (;;) {
            if ((e & 8u) && o > 31 && (pix << 1) < best) { best = pix << 1; best_pos = t; }            // west candidate: x > 0
            if ((e & 16u) && o < o_max && ((pix << 1) | 1u) < best) { best = (pix << 1) | 1u; best_pos = t; }  // east: x + 1 < w
            min_pix = min(min_pix, pix);
            const int dx = (int)((e >> 5) & 3u) - 1, dy = (int)((e >> 7) & 3u) - 1;
            o += dx; y += dy;
            pix += (uint32_t)(dy * w + dx);
            state_off = e & 0x1c00u;
            t++;
            e = *reinterpret_cast<const uint16_t *>(lut + state_off + hood2(plane, g.Hp, o, y));
            // the next relay visit (my own, if the border has no other): it owns a candidate crack on a relay row
            if (((uint32_t)y & rmask) == 0u && (((e & 8u) && o > 31) || ((e & 16u) && o < o_max))) break;
        }
        out.next = relay_index(l, g, plane, frame, o - 31, y, ((e & 8u) && o > 31) ? 0u : 1u);
        out.len = t; out.cand = best; out.cand_pos = best_pos; out.min_pix = min_pix; out.state = (uint32_t)pred;
        l.segs[i] = out;
    }
}

// The relays of a border form a cycle of segments, and following a cycle is a chain of dependent loads: the largest border of the
// reference bench's noise frame has well over a thousand segments.  So first every relay sums up the `jump_hops` segments after it
// (all relays at once, jump_hops dependent steps).
__global__ void __launch_bounds__(256) k3_jumps(const Lists l) {
    if (l.counters[kNumRelays] > l.relay_cap) return;
    const uint32_t total = l.counters[kNumRelays];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        Seg q = l.segs[i];
        if (q.len == 0) continue;
        Jump out;
        out.len = 0; out.cand = kNone; out.cand_off = 0; out.min_pix = kNone; out.min_idx = kNone; out.pad0 = out.pad1 = 0;
        uint32_t j = i;
        for (uint32_t h = 0;;) {
            if (q.cand < out.cand) { out.cand = q.cand; out.cand_off = out.len + q.cand_pos; }
            out.min_pix = min(out.min_pix, q.min_pix);
            out.len += q.len;
            j = q.next;
            out.min_idx = min(out.min_idx, j);
            if (++h == l.jump_hops || j == i) break;
            q = l.segs[j];
        }
        out.dest = j;
        l.jumps[i] = out;
    }
}

// Every relay then follows its cycle: it jumps while every relay it would land on or pass has a larger index, leaving
// (its index << 32 | visits so far) at the relays it jumps from; when its own index is among the next jump_hops it closes the
// cycle segment by segment, leaving the same in each; when a smaller index is, it is not the leader and stops.  The leader — the
// smallest index of the cycle — so learns the border: its length, its start (the smallest candidate key on the way = the
// reference's discovery point) and its raster-first pixel, and records it like a surviving candidate does; its own record then
// holds the border's slot and the position of the start visit.  Everything left on the way is merged with an atomic minimum:
// the leader has the smallest index and passes everything, so its values are what remains.
__global__ void __launch_bounds__(256) k3_cycles(const Geo g, const uint32_t min_points, const Lists l) {
    if (l.counters[kNumRelays] > l.relay_cap) return;
    const uint32_t total = l.counters[kNumRelays];
    const size_t words_per_frame = (size_t)g.h * g.wpr;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        if (l.segs[i].len == 0) continue;
        uint32_t j = i, n = 0, best = kNone, best_off = 0, min_pix = kNone;
        bool leader = true;
        for (;;) {
            const Jump jp = l.jumps[j];
            if (jp.min_idx < i) { leader = false; break; }
            if (jp.min_idx == i) {  // the segments after j lead back to me
                for (;;) {
                    const Seg q = l.segs[j];
                    atomicMin(&l.seg_owner[j], ((unsigned long long)i << 32) | n);
                    if (q.cand < best) { best = q.cand; best_off = n + q.cand_pos; }
                    min_pix = min(min_pix, q.min_pix);
                    n += q.len;
                    j = q.next;
                    if (j == i) break;
                }
                break;
            }
            atomicMin(&l.anchor_owner[j], ((unsigned long long)i << 32) | n);
            if (jp.cand < best) { best = jp.cand; best_off = n + jp.cand_off; }
            min_pix = min(min_pix, jp.min_pix);
            n += jp.len;
            j = jp.dest;
        }
        if (!leader || best == kNone) continue;
        const uint32_t frame = l.relays[i].y >> 1, kind = best & 1u, spix = best >> 1;
        const uint32_t sy = spix / g.w, sx = spix - sy * g.w;
        const unsigned long long gid = (unsigned long long)frame * words_per_frame + (unsigned long long)sy * g.wpr + (sx >> 5);
        const unsigned long long key = (((gid << 5) | (sx & 31u)) << 1) | kind;
        l.segs[i].off = best_off;
        l.segs[i].slot = record_survivor(l, frame, key, (int)kind, n, min_pix == spix, min_points, true);
    }
}

// A relay that was jumped from hands (walker, visits so far) on to the jump_hops segments after it.
__global__ void __launch_bounds__(256) k3_spread(const Lists l) {
    if (l.counters[kNumRelays] > l.relay_cap) return;
    const uint32_t total = l.counters[kNumRelays];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const unsigned long long a = l.anchor_owner[i];
        if (a == ~0ull) continue;
        const unsigned long long owner = a & 0xffffffff00000000ull;
        uint32_t cum = (uint32_t)a, j = i;
        for (uint32_t h = 0; h < l.jump_hops; h++) {
            const Seg q = l.segs[j];
            atomicMin(&l.seg_owner[j], owner | cum);
            cum += q.len;
            j = q.next;
        }
    }
}

// The undecided candidates — mostly the one survivor of each long border — walk to the end, all at the same time, each
// as a pair of adjacent lanes: the even lane follows the border forwards from the start visit (index 0, 1, 2, ...), the odd
// lane backwards (index n-1, n-2, ...), in lockstep, and after every step they compare visits (pixel + direction of the
// previous border pixel identify a visit uniquely within the loop).  When the forward lane stands on the backward lane's
// current visit the border has 2s + 1 points, when it stands on the backward lane's previous visit it has 2s.  Every visit
// is examined by one of the two for raster-earlier candidate cracks (either finding one kills the candidate).
// (Measured before the pairing: fewer walkers per warp, software prefetch of the sector ahead and a register window all
// made this kernel slower: its time is the dependent chain of the longest border, about 750 cycles per step — which is
// why the per-step exchange and tests were moved off that chain, see the blocks of kBlk steps below.)
template <int kBlk, bool relay_on>
__global__ void __launch_bounds__(128) k3_walkers(const Geo g, const StepTables *tables, const uint32_t min_points, const Lists l) {
    __shared__ uint16_t fwd[8][512];
    __shared__ uint16_t bwd[8][512];
    for (int i = threadIdx.x; i < 8 * 512; i += blockDim.x) {
        (&fwd[0][0])[i] = (&tables->fwd[0][0])[i];
        (&bwd[0][0])[i] = (&tables->bwd[0][0])[i];
    }
    __syncthreads();
    const uint32_t total = min(l.counters[kNumWalkers], l.walkers_cap);
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, back = tid & 1u;
    const uint32_t pair_mask = 3u << (threadIdx.x & 30u);   // the two lanes of this pair: they never diverge from each other
    const unsigned char *lut = reinterpret_cast<const unsigned char *>(back ? &bwd[0][0] : &fwd[0][0]);
    const int w = (int)g.w, o_max = w + 30;
    const uint32_t rmask = (1u << l.relay_shift) - 1u;
    for (uint32_t i = tid >> 1; i < total; i += (gridDim.x * blockDim.x) >> 1) {
        const unsigned long long key = l.walkers[i];
        uint32_t frame;
        int sx, sy, kind;
        decode_key(g, key, frame, sx, sy, kind);
        const uint32_t *plane = g.planes + (size_t)frame * g.frame_words;
        asm volatile("" : "+l"(plane));  // keep the frame's base in registers: otherwise it is recomputed (64-bit) in every step
        const uint32_t start_pix = (uint32_t)(sy * w + sx);
        const uint32_t me = (start_pix << 1) | (uint32_t)kind;
        const uint32_t nb0 = ring_of(hood9(plane, g.Hp, sx, sy));
        const int adj = kind ? 4 : 0;
        int pred = -1;
        for (int k = 0; k < 8; k++) {  // clockwise from the zero neighbour: the previous pixel on the border
            const int d = (adj + k) & 7;
            if ((nb0 >> d) & 1) { pred = d; break; }
        }
        if (pred < 0) {  // isolated pixel (decided in k3_walk_short already; kept for completeness)
            if (!back) {
                uint32_t slot = 0xffffffffu;
                if (kind == 0 || sx == 0) slot = record_survivor(l, frame, key, kind, 1, true, min_points);
                l.walker_slot[i] = slot;
            }
            continue;
        }
        // The position is kept as (o = x + 31, y, pix = y w + x) and the state as the byte offset of its table row: a step is
        // three loads of one word column, three funnel shifts, the table entry, and four adds.
        int o = sx + 31, y = sy;
        uint32_t pix = start_pix, state_off = (uint32_t)pred << 10;  // forwards: the start visit
        if (back) {  // backwards: the visit before it
            o += ddx(pred); y += ddy(pred); pix = (uint32_t)(y * w + o - 31); state_off = (uint32_t)((pred + 4) & 7) << 10;
        }
        // a candidate crack of a visit comes before me in raster order:  west crack  2 pix < me  <=>  pix < tw;  east crack
        // 2 pix + 1 < me  <=>  pix < te
        const uint32_t tw = (me + 1u) >> 1, te = me >> 1;
        uint32_t min_pix = start_pix, n = 0, prev_back_id = 0xffffffffu, my_prev_id = 0xffffffffu;
        bool dead = false;
        // Blocks of kBlk steps: inside a block a lane only walks (load, table, move: the dependent chain), remembering its
        // visits; the exchange with the partner lane, the test for raster-earlier cracks and the meeting test follow once
        // per block, off that chain.  A lane may so walk up to kBlk - 1 visits past the meeting point; those are visits its
        // partner has examined already (same cracks, same verdict), checkpoints dropped there are valid positions of the
        // same border (a checkpoint needs 64 walked points, so n >= 122 and n / 2 + kBlk < n), and the meeting point itself
        // is taken from the remembered visit.
        uint32_t meet_id = 0;
        for (uint32_t s0 = 0;; s0 += kBlk) {
            uint32_t ids[kBlk];
            bool mine_dead = false;
#pragma unroll
            for (int k = 0; k < kBlk; k++) {
                const uint32_t h2 = hood2(plane, g.Hp, o, y);
                const uint32_t e = *reinterpret_cast<const uint16_t *>(lut + state_off + h2);
                const uint32_t fstate = back ? (e & 7u) : (state_off >> 10);      // direction of the previous border pixel at this visit
                ids[k] = (pix << 3) | fstate;
                // candidate cracks of this visit that come before me in raster order (west needs x > 0, east x + 1 < w); a relay
                // visit means the border belongs to k3_segments / k3_cycles
                mine_dead |= ((e & 8u) && o > 31 && pix < tw) || ((e & 16u) && o < o_max && pix < te) ||
                             (relay_on && ((uint32_t)y & rmask) == 0u && (((e & 8u) && o > 31) || ((e & 16u) && o < o_max)));
                min_pix = min(min_pix, pix);
                // checkpoints for k3_emit: forwards at index kSeg, 2 kSeg, ...; backwards kSeg, 2 kSeg, ... points before the end
                const uint32_t walked = back ? s0 + k + 1 : s0 + k;
                if (walked && walked % kSeg == 0) {
                    const uint32_t c = atomicAdd(&l.counters[kNumCkpts], 1u);
                    if (c < l.ckpt_cap) l.ckpts[c] = Ckpt{i, walked, (uint32_t)(o - 31) | ((uint32_t)y << 16), fstate | (back ? kCkptBackward : 0u)};
                    else atomicOr(&l.counters[kOverflow], 1u);
                }
                const int dx = (int)((e >> 5) & 3u) - 1, dy = (int)((e >> 7) & 3u) - 1;
                o += dx; y += dy;
                pix += (uint32_t)(dy * w + dx);
                state_off = e & 0x1c00u;
            }
            uint32_t oid[kBlk];
#pragma unroll
            for (int k = 0; k < kBlk; k++) oid[k] = __shfl_xor_sync(pair_mask, ids[k], 1);
            dead = __shfl_xor_sync(pair_mask, (int)mine_dead, 1) || mine_dead;
            if (dead) break;
            // the forward lane compares with the backward lane's visit of the same step and of the step before; the backward
            // lane mirrors it.  s is the step: forward visit index s, backward visit index n - 1 - s.
            bool met = false;
#pragma unroll
            for (int k = 0; k < kBlk; k++) {
                if (met) continue;
                const uint32_t s = s0 + k;
                const uint32_t fwd_id = back ? oid[k] : ids[k], back_id = back ? ids[k] : oid[k];
                const uint32_t back_prev = k == 0 ? (back ? my_prev_id : prev_back_id) : (back ? ids[k > 0 ? k - 1 : 0] : oid[k > 0 ? k - 1 : 0]);
                if (fwd_id == back_id) { n = 2 * s + 1; met = true; meet_id = ids[k]; }
                else if (s > 0 && fwd_id == back_prev) { n = 2 * s; met = true; meet_id = ids[k]; }
            }
            if (met) break;
            my_prev_id = ids[kBlk - 1];
            prev_back_id = oid[kBlk - 1];
        }
        min_pix = min(min_pix, __shfl_xor_sync(pair_mask, min_pix, 1));
        if (back) continue;
        uint32_t slot = 0xffffffffu;
        if (!dead) {
            // the meeting point is where the forward lane stands: one more checkpoint there closes the gap between the last
            // forward and the first backward segment (they may overlap: every segment writes the same values)
            if (n > kSeg) {
                const uint32_t c = atomicAdd(&l.counters[kNumCkpts], 1u);
                const uint32_t mp = meet_id >> 3, my = mp / (uint32_t)w, mx = mp - my * (uint32_t)w;
                if (c < l.ckpt_cap) l.ckpts[c] = Ckpt{i, n / 2, mx | (my << 16), meet_id & 7u};
                else atomicOr(&l.counters[kOverflow], 1u);
            }
            slot = record_survivor(l, frame, key, kind, n, min_pix == start_pix, min_points);
        }
        l.walker_slot[i] = slot;
    }
}

// after the radix sort: lengths and point offsets in sorted order and the sorted position of every slot
__global__ void __launch_bounds__(256) k3_rank(const uint32_t *slot_sorted, const uint32_t *long_n, const uint32_t *off_slot, uint32_t n_long,
                                               uint32_t *n_sorted, uint32_t *off_sorted, uint32_t *rank) {
    const uint32_t ci = blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= n_long) return;
    const uint32_t s = slot_sorted[ci];
    if (s == 0xffffffffu) {  // padding of a speculatively sized sort (k3_spec_prepare): sorts last, has no points
        n_sorted[ci] = 0;
        off_sorted[ci] = 0;
        return;
    }
    n_sorted[ci] = long_n[s];
    off_sorted[ci] = off_slot[s];
    rank[s] = ci;
}

// The order of the long borders without a global sort: the keys are frame-major, so a border's position is the number
// of long borders in earlier frames plus its rank among those of its own frame.  One CTA per frame: sums the counts of
// the frames before it, loads the frame's keys (at most frame_cap; the host takes the radix sort when a frame has more)
// into shared memory and ranks each by counting the smaller ones.  Replaces radix sort + k3_rank (seven launches).
constexpr uint32_t kOrderCap = 1024;
__global__ void __launch_bounds__(256) k3_order(const Lists l, uint32_t n_frames, unsigned long long *keys_sorted, uint32_t *n_sorted,
                                                uint32_t *off_sorted, uint32_t *rank, const uint32_t *dyn) {
    __shared__ unsigned long long keys[kOrderCap];
    __shared__ uint32_t partial[8];
    if (dyn && dyn[kSpecFail]) return;
    const uint32_t f = blockIdx.x, cap = l.frame_cap;
    uint32_t before = 0;
    for (uint32_t i = threadIdx.x; i < f; i += blockDim.x) before += min(l.frame_long_count[i], cap);
    for (int o = 16; o; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if ((threadIdx.x & 31) == 0) partial[threadIdx.x >> 5] = before;
    const uint32_t m = min(l.frame_long_count[f], cap);
    const unsigned long long *fk = l.frame_keys + (size_t)f * cap;
    for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) keys[i] = fk[i];
    __syncthreads();
    uint32_t base = 0;
    for (uint32_t i = 0; i < blockDim.x / 32; i++) base += partial[i];
    for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) {
        const unsigned long long k = keys[i];
        uint32_t r = 0;
        for (uint32_t j = 0; j < m; j++) r += keys[j] < k ? 1u : 0u;
        const uint32_t ci = base + r, slot = l.frame_slots[(size_t)f * cap + i];
        keys_sorted[ci] = k;
        n_sorted[ci] = l.long_n[slot];
        off_sorted[ci] = l.long_off_slot[slot];
        rank[slot] = ci;
    }
}

// Speculative finish (k3_finish_speculative): the second half of the stage is enqueued before the list sizes are known on
// the host, sized from the previous call.  counters[kSpecFail] = 1 when the real sizes do not fit (every later kernel of the chain
// then returns at once and the host, which sees the same counters after its next synchronisation, redoes the second half
// exactly); the sort input is padded to its speculated size with keys that sort last.
__global__ void __launch_bounds__(256) k3_spec_prepare(unsigned long long *long_keys, uint32_t *long_slot, uint32_t *counters,
                                                       const unsigned long long *long_points, uint32_t cap_long, uint32_t cap_ckpts,
                                                       unsigned long long cap_points, uint32_t cap_frame_long, uint32_t cap_relays) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_long = counters[kNumLong];
    if (i == 0)
        counters[kSpecFail] = (counters[kOverflow] || n_long > cap_long || counters[kNumCkpts] > cap_ckpts || *long_points > cap_points ||
                               counters[kMaxFrameLong] > cap_frame_long || counters[kNumRelays] > cap_relays) ? 1u : 0u;
    if (i >= n_long && i < cap_long) {
        long_keys[i] = ~0ull;
        long_slot[i] = 0xffffffffu;
    }
}

struct Contour {
    uint32_t frame, start, n, kind;     // start = x | y << 16
    unsigned long long point_off;
};

// Writes the points (x | y << 16) of the long borders (sorted by raster position of the start) in the reference's order,
// i.e. the forward trace from the start pixel, kSeg points per thread: thread ci < n_contours starts at the border's
// start pixel, the others at a checkpoint dropped by the border's walker.
template <bool LIGHT>
__global__ void __launch_bounds__(128) k3_emit(const Geo g, const StepTables *tables, const unsigned long long *keys, const uint32_t *lens,
                                               const uint32_t *offsets, uint32_t n_contours, const uint32_t *rank, const uint32_t *walker_slot,
                                               const Ckpt *ckpts, uint32_t n_ckpts, Contour *contours, uint32_t *points, const uint32_t *dyn,
                                               const uint2 *relays, const Seg *segs, const unsigned long long *seg_owner, uint32_t n_relays) {
    __shared__ uint16_t fwd[8][512];
    if (dyn) {  // speculative finish: the real sizes are on the device only
        if (dyn[kSpecFail]) return;
        n_contours = dyn[kNumLong]; n_ckpts = dyn[kNumCkpts]; n_relays = min(n_relays, dyn[kNumRelays]);
        if (blockIdx.x * blockDim.x >= n_contours + n_ckpts + n_relays) return;
    }
    for (int i = threadIdx.x; i < 8 * 512; i += blockDim.x) (&fwd[0][0])[i] = (&tables->fwd[0][0])[i];
    __syncthreads();
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_contours + n_ckpts + n_relays) return;
    uint32_t frame, ci, first, count, state;
    int x, y, sx, sy, kind;
    if (t >= n_contours + n_ckpts) {
        // a relay segment: its visits go to (off + i) mod n of the border's list; borders the reference never follows, or too
        // short to matter, were not recorded
        const uint32_t ri = t - n_contours - n_ckpts;
        const Seg sg = segs[ri];
        if (sg.len == 0) return;
        const unsigned long long own = seg_owner[ri];
        const uint32_t leader = (uint32_t)(own >> 32), cum = (uint32_t)own;
        const uint32_t slot = segs[leader].slot, start = segs[leader].off;
        if (slot == kNone) return;
        const uint2 r = relays[ri];
        ci = rank[slot];
        const uint32_t n = lens[ci] & ~kRelayFlag;
        uint32_t *out = points + offsets[ci];
        const uint32_t *plane = g.planes + (size_t)(r.y >> 1) * g.frame_words;
        asm volatile("" : "+l"(plane));
        const unsigned char *lut = reinterpret_cast<const unsigned char *>(&fwd[0][0]);
        int o = (int)(r.x & 0xffffu) + 31, yy = (int)(r.x >> 16);
        uint32_t state_off = sg.state << 10, pos = cum >= start ? cum - start : cum + n - start;
        for (uint32_t i = 0; i < sg.len; i++) {
            out[pos] = (uint32_t)(o - 31) | ((uint32_t)yy << 16);
            if (++pos == n) pos = 0;
            const uint32_t e = *reinterpret_cast<const uint16_t *>(lut + state_off + hood2(plane, g.Hp, o, yy));
            o += (int)((e >> 5) & 3u) - 1;
            yy += (int)((e >> 7) & 3u) - 1;
            state_off = e & 0x1c00u;
        }
        return;
    }
    if (t < n_contours) {
        ci = t;
        decode_key(g, keys[ci], frame, sx, sy, kind);
        const uint32_t *plane = g.planes + (size_t)frame * g.frame_words;
        const uint32_t nb0 = ring_of(hood9(plane, g.Hp, sx, sy));
        const int adj = kind ? 4 : 0;
        int pred = 0;
        for (int q = 0; q < 8; q++) {
            const int d = (adj + q) & 7;
            if ((nb0 >> d) & 1) { pred = d; break; }
        }
        const uint32_t n = lens[ci] & ~kRelayFlag;
        first = 0; count = (lens[ci] & kRelayFlag) ? 0u : min(kSeg, n);  // the rest is covered from the checkpoints (none for borders of at most kSeg points); a relay border's points all come from its segments
        x = sx; y = sy; state = (uint32_t)pred;
        Contour c;
        c.frame = frame; c.start = (uint32_t)sx | ((uint32_t)sy << 16); c.n = n; c.kind = (uint32_t)kind; c.point_off = offsets[ci];
        contours[ci] = c;
    } else {
        const Ckpt c = ckpts[t - n_contours];
        const uint32_t slot = walker_slot[c.walker];
        if (slot == 0xffffffffu) return;  // that walker did not survive (or its border is too short to matter)
        ci = rank[slot];
        decode_key(g, keys[ci], frame, sx, sy, kind);
        const uint32_t n = lens[ci] & ~kRelayFlag;
        first = (c.state & kCkptBackward) ? n - c.pos : c.pos;
        count = min(kSeg, n - first);
        x = (int)(c.xy & 0xffffu); y = (int)(c.xy >> 16); state = c.state & 7u;
    }
    Window win;
    win.plane = g.planes + (size_t)frame * g.frame_words; win.Hp = g.Hp;
    if constexpr (!LIGHT) win_load(win, x, y);
    uint32_t *out = points + offsets[ci] + first;
    // four points per 16-byte store where the destination allows it (points + offset is only 4-byte aligned in general)
    uint32_t i = 0;
    const uint32_t *plane = win.plane;
    asm volatile("" : "+l"(plane));
    const unsigned char *lut = reinterpret_cast<const unsigned char *>(&fwd[0][0]);
    int o = x + 31;
    uint32_t state_off = state << 10;
    auto step = [&]() {
        if constexpr (LIGHT) {  // the walkers' step: three loads, three funnel shifts, the table entry, three adds
            const uint32_t v = (uint32_t)(o - 31) | ((uint32_t)y << 16);
            const uint32_t e = *reinterpret_cast<const uint16_t *>(lut + state_off + hood2(plane, g.Hp, o, y));
            o += (int)((e >> 5) & 3u) - 1;
            y += (int)((e >> 7) & 3u) - 1;
            state_off = e & 0x1c00u;
            return v;
        } else {
            const uint32_t v = (uint32_t)x | ((uint32_t)y << 16);
            const uint32_t e = fwd[state][win_hood(win, x)];
            x += (int)((e >> 5) & 3u) - 1;
            y += (int)((e >> 7) & 3u) - 1;
            state = e >> 10;
            win_move(win, x, y);
            return v;
        }
    };
    while (i < count && ((uintptr_t)(out + i) & 15u)) out[i++] = step();
    for (; i + 4 <= count; i += 4) {
        uint4 v;
        v.x = step(); v.y = step(); v.z = step(); v.w = step();
        *reinterpret_cast<uint4 *>(out + i) = v;
    }
    while (i < count) out[i++] = step();
}

struct Pt { int x, y; };
__device__ __forceinline__ Pt unpack(uint32_t v) { return Pt{(int)(v & 0xffffu), (int)(v >> 16)}; }

__device__ __forceinline__ int orient(Pt p, Pt q, Pt r) {
    const long long v = (long long)(q.y - p.y) * (r.x - q.x) - (long long)(q.x - p.x) * (r.y - q.y);  // 64-bit: coordinates go up to 65535
    return v == 0 ? 0 : (v > 0 ? 1 : -1);
}
__device__ __forceinline__ double pdist(Pt p, Pt q) {
    const double dx = (double)p.x - (double)q.x, dy = (double)p.y - (double)q.y;
    return sqrt(dx * dx + dy * dy);
}
// imageproc::geometry::convex_hull on exactly four points (same steps as host_quads.cpp:hull4)
__device__ bool hull4(Pt q[4]) {
    int sp = 0;
    for (int i = 1; i < 4; i++)
        if (q[i].y < q[sp].y || (q[i].y == q[sp].y && q[i].x < q[sp].x)) sp = i;
    const Pt start = q[sp];
    Pt tmp[4] = {q[0], q[1], q[2], q[3]};
    { const Pt t = tmp[0]; tmp[0] = tmp[sp]; tmp[sp] = t; }
    Pt rest[3] = {tmp[1], tmp[2], tmp[3]};
    for (int i = 1; i < 3; i++) {  // insertion sort with the sort_by closure (never Equal)
        const Pt key = rest[i];
        int j = i;
        while (j > 0) {
            const int o = orient(start, key, rest[j - 1]);
            const bool less = o == 0 ? pdist(start, key) < pdist(start, rest[j - 1]) : o < 0;
            if (!less) break;
            rest[j] = rest[j - 1];
            j--;
        }
        rest[j] = key;
    }
    Pt rem[3];
    int nr = 0;
    for (int i = 0; i < 3;) {
        Pt p = rest[i++];
        while (i < 3 && orient(start, p, rest[i]) == 0) p = rest[i++];
        rem[nr++] = p;
    }
    Pt st[4];
    int ns = 0;
    st[ns++] = start;
    for (int k = 0; k < nr; k++) {
        while (ns > 1 && orient(st[ns - 2], st[ns - 1], rem[k]) != -1) ns--;
        st[ns++] = rem[k];
    }
    if (ns != 4) return false;
    for (int i = 0; i < 4; i++) q[i] = st[i];
    return true;
}

constexpr int kRdpStack = 64;

// One warp per contour: approximate_polygon_dp(points, n * eps, closed) -> exactly 4 vertices? -> hull -> edge test
// (src/aruco.rs:133-159).  Same span order and the same "first strict maximum" rule as host_quads.cpp:simplify_closed.
__global__ void __launch_bounds__(128) k3_rdp(const Contour *contours, const uint32_t *points, uint32_t n_contours, double eps_factor,
                                              uint32_t min_edge_length, uint32_t *quads, uint32_t *frame_flags, const uint32_t *dyn,
                                              const bool small_coords) {
    __shared__ uint2 stacks[4][kRdpStack];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t ci = blockIdx.x * 4 + wid;
    if (dyn) {
        if (dyn[kSpecFail]) return;
        n_contours = dyn[kNumLong];
    }
    if (ci >= n_contours) return;
    const Contour c = contours[ci];
    const uint32_t *pts = points + c.point_off;
    const double eps = (double)c.n * eps_factor;
    uint2 *stack = stacks[wid];
    int sp = 0;
    if (lane == 0) stack[0] = make_uint2(0u, c.n - 1);
    sp = 1;
    uint32_t nout = 0, nsplit = 0;
    Pt out[4];
    bool overflow = false;
    while (sp > 0) {
        __syncwarp();
        const uint2 s = stack[sp - 1];
        sp--;
        const Pt ps = unpack(pts[s.x]), pe = unpack(pts[s.y]);
        const long long a = (long long)ps.y - pe.y, b = (long long)pe.x - ps.x, cc = (long long)ps.x * pe.y - (long long)pe.x * ps.y;
        // pass 1: largest numerator and the first index that reaches it (per lane in index order, then across lanes)
        long long best = 0;
        uint32_t best_i = 0xffffffffu;
        // a x + b y + cc == a (x - xs) + b (y - ys): with coordinates below 2^14 both products and their sum fit 32 bits
        const int a32 = (int)a, b32 = (int)b, k32 = small_coords ? -(a32 * ps.x + b32 * ps.y) : 0;
        if (small_coords) {
            int best32 = 0;
            for (uint32_t i = s.x + 1 + lane; i <= s.y; i += 32) {
                const uint32_t pv = pts[i];
                const int v = abs(b32 * (int)(pv >> 16) + (a32 * (int)(pv & 0xffffu) + k32));
                if (v > best32) { best32 = v; best_i = i; }
            }
            const int wmax = __reduce_max_sync(0xffffffffu, best32);
            best_i = __reduce_min_sync(0xffffffffu, best32 == wmax ? best_i : 0xffffffffu);
            best = wmax;
        } else {
            for (uint32_t i = s.x + 1 + lane; i <= s.y; i += 32) {
                const Pt p = unpack(pts[i]);
                long long v = a * p.x + b * p.y + cc;
                v = v < 0 ? -v : v;
                if (v > best) { best = v; best_i = i; }
            }
            for (int off = 16; off; off >>= 1) {
                const long long other = __shfl_xor_sync(0xffffffffu, best, off);
                const uint32_t other_i = __shfl_xor_sync(0xffffffffu, best_i, off);
                if (other > best || (other == best && other_i < best_i)) { best = other; best_i = other_i; }
            }
        }
        // dmax > eps, where dmax = best / den in f64 as the reference computes it.  With small numerators the comparison of
        // the squares decides it without the square root and the division unless the two sides agree to 2^-40 (the f64
        // results carry relative errors below 2^-50, so outside that band the rounded quotient lies on the same side of
        // eps); and numerators below 2^40 are too far apart, relatively, for two of them to round to the same quotient, so
        // the first index of the largest numerator is the reference's index.
        bool split = false, decided = false;
        uint32_t index = 0;
        if (small_coords && best > 0) {
            const double d2 = (double)(a32 * a32 + b32 * b32);
            const double lhs = (double)best * (double)best, rhs = (eps * eps) * d2;
            if (lhs > rhs * 1.0000000000009095) { split = true; index = best_i; decided = true; }        // 1 + 2^-40
            else if (lhs < rhs * 0.9999999999990905) { decided = true; }                                // 1 - 2^-40
        }
        if (!decided && best > 0) {
            const double den = sqrt((double)a * (double)a + (double)b * (double)b);
            double dmax = 0.0;
            const double q = (double)best / den;
            if (q > 0.0) {
                long long t = best;  // smallest numerator whose quotient equals the maximum's
                while (t > 1 && (double)(t - 1) / den == q) t--;
                dmax = q;
                uint32_t first = best_i;
                if (t != best) {  // rare: a smaller numerator rounds to the same distance, and one of those may come earlier
                    first = 0xffffffffu;
                    for (uint32_t i = s.x + 1 + lane; i <= s.y && first == 0xffffffffu; i += 32) {
                        const Pt p = unpack(pts[i]);
                        long long v = a * p.x + b * p.y + cc;
                        v = v < 0 ? -v : v;
                        if (v >= t) first = i;
                    }
                    for (int off = 16; off; off >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, off));
                }
                index = first;
            }
            split = dmax > eps;
        }
        if (split) {
            // every split adds one vertex to the final polygon (vertices = splits + 1): the fourth split settles "not a quad"
            if (++nsplit >= 4) { nout = 5; break; }
            if (sp + 2 > kRdpStack) { overflow = true; break; }
            __syncwarp();
            if (lane == 0) {
                stack[sp] = make_uint2(index, s.y);
                stack[sp + 1] = make_uint2(s.x, index);
            }
            sp += 2;
        } else {
            if (nout < 4) out[nout] = ps;
            nout++;
            if (nout > 4) break;
        }
    }
    if (lane != 0) return;
    uint32_t *q = quads + (size_t)ci * 8;
    q[0] = 0xffffffffu;  // not a candidate
    if (overflow) { atomicOr(&frame_flags[c.frame], 2u); return; }
    if (nout != 4) return;
    if (!hull4(out)) return;
    uint32_t cmin = min_edge_length + 1;
    for (int i = 0; i < 4; i++) {
        const int j = (i + 1) & 3;
        const int dx = out[i].x - out[j].x, dy = out[i].y - out[j].y;
        cmin = min(cmin, (uint32_t)(dx * dx + dy * dy));
    }
    if (cmin < min_edge_length) return;  // squared vs unsquared on purpose (SURVEY Q1)
    for (int i = 0; i < 4; i++) { q[2 * i] = (uint32_t)out[i].x; q[2 * i + 1] = (uint32_t)out[i].y; }
}

__device__ __forceinline__ float perimeter(const uint32_t *q) {
    float p = 0.0f;
    for (int i = 0; i < 4; i++) {
        const int j = (i + 1) & 3;
        const float dx = (float)q[2 * i] - (float)q[2 * j], dy = (float)q[2 * i + 1] - (float)q[2 * j + 1];
        p += sqrtf((dx * dx) + (dy * dy));
    }
    return p;
}

// One warp per frame: the frame's quads in contour order, enforce_clockwise_corners, discard_too_near
// (src/aruco.rs:168-232).  frame_first[f] .. frame_first[f + 1] = the frame's range of contours.
__device__ __forceinline__ uint32_t lower_bound_key(const unsigned long long *keys, uint32_t n, unsigned long long v) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (keys[mid] < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(32) k3_finalize(const uint32_t *contour_quads, const unsigned long long *keys, size_t words_per_frame,
                                                  uint32_t total_contours, uint32_t n_frames, float min_corner_separation,
                                                  uint32_t quad_cap, uint32_t *out_quads, uint32_t *out_counts, uint32_t *out_before_discard,
                                                  uint32_t *frame_flags, uint8_t *dead_scratch, const uint32_t *dyn) {
    if (dyn) {
        if (dyn[kSpecFail]) return;
        total_contours = dyn[kNumLong];
    }
    extern __shared__ uint32_t sq[];  // quad_cap * 8 words of quads, then quad_cap floats of perimeters, then quad_cap dead bytes
    float *sper = reinterpret_cast<float *>(sq + (size_t)quad_cap * 8);
    uint8_t *dead = reinterpret_cast<uint8_t *>(sper + quad_cap);
    const uint32_t f = blockIdx.x;
    const int lane = threadIdx.x;
    // the frame's borders are a contiguous range of the sorted list: keys are (word id, bit, kind) with frame-major word ids
    const uint32_t c0 = lower_bound_key(keys, total_contours, ((unsigned long long)f * words_per_frame) << 6);
    const uint32_t c1 = lower_bound_key(keys, total_contours, ((unsigned long long)(f + 1) * words_per_frame) << 6);
    (void)n_frames; (void)dead_scratch;
    uint32_t nq = 0;
    bool over = false;
    // eight groups of 32 contours per round, their loads issued together: a frame of the noise workload has 17 k long borders
    // and one warp walks them all, so this loop was 525 dependent round trips to L2 (0.17 ms of a single-frame call)
    constexpr int kGroups = 8;
    for (uint32_t base = c0; base < c1; base += 32 * kGroups) {
        uint32_t first[kGroups];
#pragma unroll
        for (int u = 0; u < kGroups; u++) {
            const uint32_t ci = base + 32 * u + lane;
            first[u] = ci < c1 ? contour_quads[(size_t)ci * 8] : 0xffffffffu;
        }
#pragma unroll
        for (int u = 0; u < kGroups; u++) {
            const uint32_t ci = base + 32 * u + lane;
            const bool valid = first[u] != 0xffffffffu;
            const uint32_t m = __ballot_sync(0xffffffffu, valid);
            if (valid) {
                const uint32_t slot = nq + __popc(m & ((1u << lane) - 1));
                if (slot < quad_cap) {
                    const uint4 a = *reinterpret_cast<const uint4 *>(contour_quads + (size_t)ci * 8);
                    const uint4 b = *reinterpret_cast<const uint4 *>(contour_quads + (size_t)ci * 8 + 4);
                    uint32_t *p = sq + (size_t)slot * 8;
                    p[0] = a.x; p[1] = a.y; p[2] = a.z; p[3] = a.w; p[4] = b.x; p[5] = b.y; p[6] = b.z; p[7] = b.w;
                } else {
                    over = true;
                }
            }
            nq += __popc(m);
        }
    }
    over = __any_sync(0xffffffffu, over);
    if (over) nq = quad_cap;
    __syncwarp();
    for (uint32_t i = lane; i < nq; i += 32) {  // enforce_clockwise_corners, perimeters
        uint32_t *p = sq + (size_t)i * 8;
        const int dx1 = (int)p[2] - (int)p[0], dy1 = (int)p[3] - (int)p[1], dx2 = (int)p[4] - (int)p[0], dy2 = (int)p[5] - (int)p[1];
        if (dx1 * dy2 - dy1 * dx2 < 0) {
            const uint32_t sx = p[2], sy = p[3];
            p[2] = p[6]; p[3] = p[7]; p[6] = sx; p[7] = sy;
        }
        sper[i] = perimeter(p);
        dead[i] = 0;
    }
    __syncwarp();
    uint32_t *dst = out_quads + (size_t)f * quad_cap * 8;
    if (lane == 0) {
        if (over) atomicOr(&frame_flags[f], 4u);
        out_before_discard[f] = nq;
    }
    // discard_too_near: i is sequential as in the reference; for one i the lanes test 32 later quads at a time.  In the
    // reference's j loop, close quads with a perimeter <= perimeter(i) die until the first close quad with a larger one
    // kills i, after which nothing else happens for this i.
    for (uint32_t i = 0; i + 1 < nq; i++) {
        if (dead[i]) continue;  // warp-uniform (shared memory, synchronised below)
        const float per_i = sper[i];
        for (uint32_t j0 = i + 1; j0 < nq; j0 += 32) {
            const uint32_t j = j0 + lane;
            bool close = false;
            if (j < nq && !dead[j]) {
                float d = 0.0f;
                for (int c = 0; c < 4; c++) {
                    const float dx = (float)sq[(size_t)i * 8 + 2 * c] - (float)sq[(size_t)j * 8 + 2 * c];
                    const float dy = (float)sq[(size_t)i * 8 + 2 * c + 1] - (float)sq[(size_t)j * 8 + 2 * c + 1];
                    d += sqrtf((dx * dx) + (dy * dy));
                }
                close = (d / 4.0f) < min_corner_separation;
            }
            const bool killer = close && !(per_i >= sper[j]);
            const uint32_t mk = __ballot_sync(0xffffffffu, killer);
            const int first_killer = mk ? __ffs(mk) - 1 : 32;
            if (close && lane < first_killer) dead[j] = 1;
            if (mk) {
                if (lane == 0) dead[i] = 1;
                break;
            }
        }
        __syncwarp();
    }
    __syncwarp();
    if (lane == 0) {
        uint32_t kept = 0;
        for (uint32_t i = 0; i < nq; i++)
            if (!dead[i]) {
                for (int c = 0; c < 8; c++) dst[(size_t)kept * 8 + c] = sq[(size_t)i * 8 + c];
                kept++;
            }
        out_counts[f] = kept;
    }
}

}  // namespace

namespace {
// List sizes of one call, as k3_begin's counters report them.  The same struct carries the sizes a second half is enqueued
// with: the real ones (k3_finish) or capacities (k3_finish_speculative); frame_long above the per-frame lists' capacity
// orders the borders with the radix sort.
struct ListSizes {
    uint32_t n_long = 0, ckpts = 0, relays = 0, frame_long = 0;
    unsigned long long points = 0;
    bool overflow = false;  // a list overflowed: every frame of the call is flagged for the host stage
    // the test k3_spec_prepare makes on the device
    bool fits(const ListSizes &cap) const {
        return !overflow && n_long <= cap.n_long && ckpts <= cap.ckpts && points <= cap.points && frame_long <= cap.frame_long &&
               relays <= cap.relays;
    }
};
}  // namespace

struct K3Workspace::Impl {
    DevBuf<StepTables> tables;
    // work lists
    DevBuf<unsigned long long> cands, walkers, long_keys, long_keys_sorted, long_points, frame_points, frame_keys, seg_owner, anchor_owner;
    DevBuf<uint32_t> counters, walker_slot, long_n, long_n_sorted, long_off, long_slot, long_slot_sorted, long_rank, long_off_slot;
    DevBuf<uint32_t> frame_contours, frame_long_count, frame_slots, relay_base;
    DevBuf<Ckpt> ckpts;
    DevBuf<uint2> relays;
    DevBuf<Seg> segs;
    DevBuf<Jump> jumps;
    DevBuf<uint8_t> cub_tmp;
    DevBuf<Contour> contours;
    DevBuf<uint32_t> contour_quads, points;
    DevBuf<uint8_t> dead;
    PinBuf<unsigned long long> h_counts;  // [0..3] the eight 32-bit counters, [4] long_points
    Geo g;                                // state handed from k3_begin to the second half
    Lists l;
    // the previous call with this geometry: what k3_finish_speculative sizes its launches from
    struct History {
        uint32_t n = 0, w = 0, h = 0;
        ListSizes sizes;
        bool valid = false;
    } hist;
    std::optional<ListSizes> spec;        // capacities of the speculative finish in flight
};

K3Workspace::K3Workspace() : impl(new Impl()) {}
K3Workspace::~K3Workspace() = default;

#define K3_CUDA(expr)                              \
    do {                                           \
        cudaError_t e__ = (expr);                  \
        if (e__ != cudaSuccess) return e__;        \
    } while (0)

static __global__ void k3_flag_all(uint32_t *frame_flags, uint32_t n, const uint32_t *counters, int force) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && (force || counters[kOverflow])) frame_flags[i] |= 8u;  // a work list overflowed: every frame of this call goes to the host stage
}

// A3_K3_TIMING=1 in the environment: print the device time of every phase of a k3_quads call (debug aid)
struct PhaseTimer {
    bool on;
    cudaStream_t s;
    cudaEvent_t ev[16];
    const char *name[16];
    int n = 0;
    PhaseTimer(cudaStream_t stream) : on(getenv("A3_K3_TIMING") != nullptr), s(stream) {}
    void mark(const char *what) {
        if (!on || n >= 16) return;
        cudaEventCreate(&ev[n]);
        cudaEventRecord(ev[n], s);
        name[n++] = what;
    }
    ~PhaseTimer() {
        if (!on || n == 0) return;
        cudaEventSynchronize(ev[n - 1]);
        for (int i = 1; i < n; i++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
            fprintf(stderr, "k3 %-12s %8.3f ms\n", name[i], ms);
        }
        for (int i = 0; i < n; i++) cudaEventDestroy(ev[i]);
    }
};

cudaError_t k3_quads(K3Workspace &ws, const K3Params &p, cudaStream_t stream) {
    cudaError_t e = k3_begin(ws, p, stream);
    return e == cudaSuccess ? k3_finish(ws, p, stream) : e;
}

// First half: candidates and walks; ends with the asynchronous copy of the list counters to the host.
cudaError_t k3_begin(K3Workspace &ws, const K3Params &p, cudaStream_t stream) {
    K3Workspace::Impl &w = *ws.impl;
    if (p.n == 0) return cudaSuccess;
    PhaseTimer timer(stream);
    if (p.w > 65535 || p.h > 65535) return cudaErrorInvalidValue;  // points are packed 16 + 16
    if ((unsigned long long)p.w * p.h >= (1ull << 29)) return cudaErrorInvalidValue;  // pixel index << 3 | state must fit 32 bits
    Geo g;
    g.planes = p.planes; g.n = p.n; g.w = p.w; g.h = p.h; g.wpr = (p.w + 31) / 32; g.Hp = p.h + 2;
    g.frame_words = (size_t)(g.wpr + 2) * g.Hp;
    if (!w.tables.p) {
        StepTables *t = new StepTables();
        build_tables(*t);
        cudaError_t e = w.tables.reserve(1);
        if (e == cudaSuccess) e = cudaMemcpy(w.tables.p, t, sizeof(StepTables), cudaMemcpyHostToDevice);
        delete t;
        K3_CUDA(e);
        K3_CUDA(w.h_counts.reserve(8));
        K3_CUDA(w.counters.reserve(8));
        K3_CUDA(w.long_points.reserve(1));
    }
    // list capacities: generous per frame; an overflow sends the whole call to the host stage (flag 8), never a wrong answer
    const size_t pixels = (size_t)p.w * p.h;
    const size_t mp = p.min_points < 4 ? 4 : p.min_points;
    const size_t want_walkers = (size_t)p.n * (pixels / 32 + 4096), want_long = (size_t)p.n * (pixels / (4 * mp) + 1024);
    // what does not fit is walked inside k3_candidates (slow: one thread per word).  A pure-noise frame leaves about 0.22
    // candidates per pixel after the word filters, so calls of a few frames get room for a third of their pixels
    size_t want_cands = (size_t)p.n * (pixels / 8 + 4096);
    {
        const size_t roomy = (size_t)p.n * (pixels / 3), cap = (size_t)16 << 20;
        const size_t alt = roomy < cap ? roomy : cap;
        if (alt > want_cands) want_cands = alt;
    }
    K3_CUDA(w.cands.reserve(want_cands));
    K3_CUDA(w.walkers.reserve(want_walkers));
    K3_CUDA(w.walker_slot.reserve(want_walkers));
    const size_t want_ckpts = (size_t)p.n * (pixels / kSeg + 4096);  // one per kSeg walked points; an overflow flags the call (host stage)
    K3_CUDA(w.ckpts.reserve(want_ckpts));
    if (want_long > w.long_keys.cap) {
        for (DevBuf<uint32_t> *b : {&w.long_n, &w.long_n_sorted, &w.long_off, &w.long_slot, &w.long_slot_sorted, &w.long_rank, &w.long_off_slot})
            K3_CUDA(b->reserve(want_long));
        K3_CUDA(w.long_keys_sorted.reserve(want_long));
        size_t need = 0;
        K3_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need, w.long_keys.p, w.long_keys_sorted.p, w.long_slot.p, w.long_slot_sorted.p, (int)want_long, 0, 64, stream));
        K3_CUDA(w.cub_tmp.reserve(need));
        K3_CUDA(w.long_keys.reserve(want_long));  // last: its capacity says that the other lists and the sort's storage have grown
    }
    K3_CUDA(w.frame_points.reserve(p.n));
    K3_CUDA(w.frame_contours.reserve(p.n));
    K3_CUDA(w.frame_long_count.reserve(p.n));
    // per-frame lists of the long borders for k3_order: kOrderCap entries per frame, for calls of up to 4096 frames (48 MB of
    // lists; every CTA of k3_order also sums the counts of the frames before its own, which is quadratic in the frame count)
    const bool frame_lists = p.n <= 4096;
    if (frame_lists) {
        K3_CUDA(w.frame_keys.reserve((size_t)p.n * kOrderCap));
        K3_CUDA(w.frame_slots.reserve((size_t)p.n * kOrderCap));
    }
    K3_CUDA(w.dead.reserve((size_t)p.n * p.quad_cap));
    // relays: the candidate cracks of every 16th row (32nd above 1200 rows).  A pure-noise frame has about w / 2 of them per
    // row; the lists are sized for that, capped at 48 M entries (an overflow sends the call to the host stage like any other list).
    // Relay walks are for calls of up to 16 frames (one front-end chunk of host input), where the time of the stage is the chain of the longest border (the reference
    // bench's noise frame: walks 1.48 -> 0.10 ms, the call 2.3 -> 1.2 ms).  A batch has enough borders to fill the machine, and there the
    // lane pairs win: 256 x 1080p with relays 1.01 ms against 0.55 ms (segment lengths are very uneven - edges nearly parallel to the
    // rows - so a warp waits for its longest, the list allocation and the survivors' records are same-address atomics in short kernels).
    // On marker frames the two routes take the same time from 2 to 32 frames per call (0.28 ... 0.33 ms), at 64 the pairs win (0.36 against 0.41 ms).
    // A3_K3_RELAY_MAX_FRAMES overrides the threshold (0 = never, read at every call: tests drive both routes).
    const char *relay_env = getenv("A3_K3_RELAY_MAX_FRAMES");
    const bool relays_off = p.n > (relay_env ? (uint32_t)strtoul(relay_env, nullptr, 10) : 16u);
    const uint32_t relay_shift = p.h > 1200 ? 5u : 4u, nrr = (p.h + (1u << relay_shift) - 1) >> relay_shift;
    size_t want_relays = relays_off ? 0 : (size_t)p.n * nrr * (p.w / 2 + 64);
    if (want_relays > ((size_t)48 << 20)) want_relays = (size_t)48 << 20;
    if (const char *cap_env = getenv("A3_K3_RELAY_CAP")) {  // test hook: a list too small for the call (overflow -> host stage)
        const size_t c = strtoull(cap_env, nullptr, 10);
        if (want_relays > c) want_relays = c ? c : 1;
    }
    K3_CUDA(w.relays.reserve(want_relays));
    K3_CUDA(w.segs.reserve(want_relays));
    K3_CUDA(w.seg_owner.reserve(want_relays));
    K3_CUDA(w.anchor_owner.reserve(want_relays));
    K3_CUDA(w.jumps.reserve(want_relays));
    K3_CUDA(w.relay_base.reserve(relays_off ? 0 : (size_t)p.n * nrr * ((p.w + 31) / 32)));
    K3_CUDA(cudaMemsetAsync(w.frame_points.p, 0, (size_t)p.n * 8, stream));
    K3_CUDA(cudaMemsetAsync(w.frame_contours.p, 0, (size_t)p.n * 4, stream));
    K3_CUDA(cudaMemsetAsync(w.frame_long_count.p, 0, (size_t)p.n * 4, stream));
    K3_CUDA(cudaMemsetAsync(p.frame_flags, 0, (size_t)p.n * 4, stream));
    K3_CUDA(cudaMemsetAsync(w.counters.p, 0, 32, stream));
    K3_CUDA(cudaMemsetAsync(w.long_points.p, 0, 8, stream));

    timer.mark("begin");
    Lists l;
    l.cands = w.cands.p; l.cands_cap = (uint32_t)(w.cands.cap > 0xffffffffull ? 0xffffffffull : w.cands.cap);
    l.walkers = w.walkers.p; l.long_keys = w.long_keys.p; l.long_n = w.long_n.p; l.counters = w.counters.p; l.long_points = w.long_points.p;
    l.walkers_cap = (uint32_t)(w.walkers.cap > 0xffffffffull ? 0xffffffffull : w.walkers.cap);
    l.long_cap = (uint32_t)(w.long_keys.cap > 0x7fffffffull ? 0x7fffffffull : w.long_keys.cap);
    l.frame_contours = w.frame_contours.p; l.frame_points = w.frame_points.p; l.frame_flags = p.frame_flags;
    l.long_slot = w.long_slot.p; l.walker_slot = w.walker_slot.p; l.ckpts = w.ckpts.p;
    l.long_off_slot = w.long_off_slot.p; l.frame_cap = frame_lists ? kOrderCap : 0u; l.frame_long_count = w.frame_long_count.p;
    l.frame_keys = w.frame_keys.p; l.frame_slots = w.frame_slots.p;
    l.ckpt_cap = (uint32_t)(w.ckpts.cap > 0x7fffffffull ? 0x7fffffffull : w.ckpts.cap);
    l.relays = w.relays.p; l.segs = w.segs.p; l.seg_owner = w.seg_owner.p; l.relay_base = w.relay_base.p; l.relay_cap = (uint32_t)want_relays;
    l.relay_shift = relay_shift; l.nrr = nrr;
    l.jumps = w.jumps.p; l.anchor_owner = w.anchor_owner.p;
    {
        const char *jump_env = getenv("A3_K3_JUMP");  // test hook: short jumps exercise the multi-jump paths on small masks
        const unsigned long jh = jump_env ? strtoul(jump_env, nullptr, 10) : 32ul;
        l.jump_hops = jh < 1 ? 1u : (jh > 1024 ? 1024u : (uint32_t)jh);
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const StepTables *tables = w.tables.p;
    {
        // about 8 blocks of 256 threads per SM (measured best: more, smaller shares than one resident wave), split over the frames
        // (blockIdx.x strides over the word columns of a frame, blockIdx.y over frames)
        const uint32_t resident = (uint32_t)sms * 8;
        const uint32_t gy = p.n < resident ? p.n : resident;
        uint32_t gx = (resident + gy - 1) / gy;
        if (gx > g.wpr) gx = g.wpr;
        // threads per block so that whole passes over a column (4 rows per thread and pass) leave few idle lanes
        const uint32_t passes = (p.h + 1023) / 1024;
        uint32_t bd = ((p.h + 4 * passes - 1) / (4 * passes) + 31) & ~31u;
        if (bd < 64) bd = 64;
        if (bd > 256) bd = 256;
        // a call of a few frames (single-frame latency): columns x frames alone leave most SMs idle, so the rows of a column are
        // cut into chunks of 256 as well (blockIdx.z)
        uint32_t gz = 1;
        if ((uint64_t)gx * gy * 2 <= resident) {
            bd = 64;
            gz = (p.h + 4 * bd - 1) / (4 * bd);
            const uint32_t room = resident / (gx * gy);
            if (gz > room) gz = room;
            if (gz < 1) gz = 1;
        }
        if (l.relay_cap) k3_candidates<true><<<dim3(gx, gy, gz), bd, 0, stream>>>(g, tables, p.min_points, l);
        else k3_candidates<false><<<dim3(gx, gy, gz), bd, 0, stream>>>(g, tables, p.min_points, l);
    }
    K3_CUDA(cudaGetLastError());
    timer.mark("candidates");
    if (l.relay_cap) {
        k3_segments<<<(uint32_t)sms * 8, 128, 0, stream>>>(g, tables, l);
        K3_CUDA(cudaGetLastError());
        timer.mark("segments");
        k3_jumps<<<(uint32_t)sms * 4, 256, 0, stream>>>(l);
        k3_cycles<<<(uint32_t)sms * 4, 256, 0, stream>>>(g, p.min_points, l);
        k3_spread<<<(uint32_t)sms * 4, 256, 0, stream>>>(l);
        K3_CUDA(cudaGetLastError());
        timer.mark("cycles");
    }
    if (l.relay_cap) k3_walk_short<true><<<(uint32_t)sms * 8, 128, 0, stream>>>(g, tables, p.min_points, l);
    else k3_walk_short<false><<<(uint32_t)sms * 8, 128, 0, stream>>>(g, tables, p.min_points, l);
    K3_CUDA(cudaGetLastError());
    timer.mark("walk_short");
    // blocks of 2 / 4 / 6 / 8 steps measured: 0.207 / 0.188 / 0.186 / 0.184 ms (before the lighter step: 0.152 ms with 8)
    if (l.relay_cap) k3_walkers<8, true><<<(uint32_t)sms * 8, 128, 0, stream>>>(g, tables, p.min_points, l);
    else k3_walkers<8, false><<<(uint32_t)sms * 8, 128, 0, stream>>>(g, tables, p.min_points, l);
    K3_CUDA(cudaGetLastError());
    timer.mark("walkers");
    k3_flag_all<<<(p.n + 127) / 128, 128, 0, stream>>>(p.frame_flags, p.n, w.counters.p, 0);
    K3_CUDA(cudaGetLastError());
    K3_CUDA(cudaMemcpyAsync(&w.h_counts.p[0], w.counters.p, 32, cudaMemcpyDeviceToHost, stream));
    K3_CUDA(cudaMemcpyAsync(&w.h_counts.p[4], w.long_points.p, 8, cudaMemcpyDeviceToHost, stream));
    w.g = g; w.l = l;
    return cudaSuccess;
}

// k3_begin's list sizes, from the pinned copy of the counters (once the stream has been synchronised)
static ListSizes read_sizes(const K3Workspace::Impl &w) {
    const uint32_t *c = reinterpret_cast<const uint32_t *>(w.h_counts.p);
    ListSizes s;
    s.n_long = c[kNumLong]; s.ckpts = c[kNumCkpts]; s.relays = c[kNumRelays]; s.frame_long = c[kMaxFrameLong];
    s.points = w.h_counts.p[4];
    s.overflow = c[kOverflow] != 0;
    return s;
}

// the sizes of this call, for the speculative finish of the next call with the same geometry
static void record_history(K3Workspace::Impl &w, const K3Params &p, const ListSizes &s) {
    w.hist = {p.n, p.w, p.h, s, !s.overflow && s.points < 0xffffffffull};
}

// The second half: sort, emission, polygon simplification and the per-frame filters, launched for the sizes `s`.  k3_finish
// passes the real sizes; k3_finish_speculative passes capacities and dyn = counters, where every kernel reads the real sizes
// and where k3_spec_prepare stops the chain when they do not fit.
static cudaError_t enqueue_finish(K3Workspace::Impl &w, const K3Params &p, const ListSizes &s, const uint32_t *dyn, cudaStream_t stream) {
    const size_t fin_smem = (size_t)p.quad_cap * (32 + 4 + 1) + 16;
    if (fin_smem > 200 * 1024) return cudaErrorInvalidValue;
    const Geo &g = w.g;
    const Lists &l = w.l;
    const size_t words_per_frame = (size_t)g.h * g.wpr, nwords = words_per_frame * p.n;
    PhaseTimer timer(stream);
    timer.mark("begin");
    if (s.n_long) {  // (speculative capacities are never 0)
        if (s.n_long > w.contours.cap) {
            const size_t c = (size_t)s.n_long + s.n_long / 4 + 1024;
            K3_CUDA(w.contours.reserve(c));
            K3_CUDA(w.contour_quads.reserve(c * 8));
        }
        const size_t need = (size_t)s.points + 1;
        if (need > w.points.cap) K3_CUDA(w.points.reserve(need + need / 4 + 1024));
        if (dyn) {
            k3_spec_prepare<<<(s.n_long + 255) / 256, 256, 0, stream>>>(w.long_keys.p, w.long_slot.p, w.counters.p, w.long_points.p, s.n_long,
                                                                        s.ckpts, s.points, s.frame_long, s.relays);
            K3_CUDA(cudaGetLastError());
        }
        if (l.frame_cap && s.frame_long <= l.frame_cap) {
            k3_order<<<p.n, 256, 0, stream>>>(l, p.n, w.long_keys_sorted.p, w.long_n_sorted.p, w.long_off.p, w.long_rank.p, dyn);
            K3_CUDA(cudaGetLastError());
        } else {
            size_t tmp = w.cub_tmp.cap;
            const int end_bit = 64 - __builtin_clzll(((unsigned long long)nwords << 6) | 1ull);
            K3_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp.p, tmp, w.long_keys.p, w.long_keys_sorted.p, w.long_slot.p, w.long_slot_sorted.p,
                                                    (int)s.n_long, 0, end_bit, stream));
            k3_rank<<<(s.n_long + 255) / 256, 256, 0, stream>>>(w.long_slot_sorted.p, w.long_n.p, w.long_off_slot.p, s.n_long, w.long_n_sorted.p,
                                                               w.long_off.p, w.long_rank.p);
            K3_CUDA(cudaGetLastError());
        }
        timer.mark("order");
        // k3_emit's step: the register window when many segments are in flight (256 x 1080p: 0.094 ms against 0.115 ms), the
        // walkers' lighter step for calls of a few frames, where the chain of one segment is what is waited for (noise frame:
        // 0.025 against 0.040 ms)
        (p.n <= 4 ? k3_emit<true> : k3_emit<false>)<<<(s.n_long + s.ckpts + s.relays + 127) / 128, 128, 0, stream>>>(
            g, w.tables.p, w.long_keys_sorted.p, w.long_n_sorted.p, w.long_off.p, s.n_long, w.long_rank.p, w.walker_slot.p, w.ckpts.p, s.ckpts,
            w.contours.p, w.points.p, dyn, w.relays.p, w.segs.p, w.seg_owner.p, s.relays);
        K3_CUDA(cudaGetLastError());
        timer.mark("emit");
        k3_rdp<<<(s.n_long + 3) / 4, 128, 0, stream>>>(w.contours.p, w.points.p, s.n_long, p.eps_factor, p.min_edge_length, w.contour_quads.p,
                                                        p.frame_flags, dyn, p.w <= 16384 && p.h <= 16384);
        K3_CUDA(cudaGetLastError());
    }
    timer.mark("rdp");
    K3_CUDA(cudaFuncSetAttribute(k3_finalize, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));
    k3_finalize<<<p.n, 32, fin_smem, stream>>>(w.contour_quads.p, w.long_keys_sorted.p, words_per_frame, s.n_long, p.n, p.min_corner_separation,
                                               p.quad_cap, p.quads, p.quad_counts, p.before_discard, p.frame_flags, w.dead.p, dyn);
    K3_CUDA(cudaGetLastError());
    timer.mark("finalize");
    if (p.frame_contours) K3_CUDA(cudaMemcpyAsync(p.frame_contours, w.frame_contours.p, (size_t)p.n * 4, cudaMemcpyDeviceToDevice, stream));
    if (p.frame_points) K3_CUDA(cudaMemcpyAsync(p.frame_points, w.frame_points.p, (size_t)p.n * 8, cudaMemcpyDeviceToDevice, stream));
    return cudaSuccess;
}

// Second half, exactly: waits for the counters (the only host synchronisation of the stage) and launches for the real sizes.
cudaError_t k3_finish(K3Workspace &ws, const K3Params &p, cudaStream_t stream) {
    K3Workspace::Impl &w = *ws.impl;
    if (p.n == 0) return cudaSuccess;
    K3_CUDA(cudaStreamSynchronize(stream));
    const ListSizes s = read_sizes(w);
    if (getenv("A3_K3_TIMING")) {
        const uint32_t *hc = reinterpret_cast<const uint32_t *>(w.h_counts.p);
        fprintf(stderr, "k3 lists: %u candidates, %u walkers, %u long borders, %llu points, %u checkpoints, %u relay cracks\n", hc[kNumCands],
                hc[kNumWalkers], s.n_long, s.points, s.ckpts, s.relays);
    }
    record_history(w, p, s);
    w.spec.reset();
    const bool wide = s.points >= 0xffffffffull;
    if (wide && !s.overflow) {  // point offsets are 32-bit: hand the whole call to the host stage
        k3_flag_all<<<(p.n + 127) / 128, 128, 0, stream>>>(p.frame_flags, p.n, w.counters.p, 1);
        K3_CUDA(cudaGetLastError());
    }
    const Lists &l = w.l;
    ListSizes run = s;
    run.n_long = s.overflow || wide ? 0 : std::min(s.n_long, l.long_cap);  // every frame is flagged for the host stage
    run.ckpts = std::min(s.ckpts, l.ckpt_cap);
    run.relays = std::min(s.relays, l.relay_cap);
    return enqueue_finish(w, p, run, nullptr, stream);
}

// Second half without the host synchronisation: the same launches, sized from the previous call of this geometry plus
// headroom; the real sizes stay on the device (`counters`).  *speculated = false (nothing enqueued) when there is no such
// history.  The caller synchronises the stream later and asks k3_speculation_held(); when it did not hold, k3_finish redoes
// the second half exactly (k3_begin's lists are untouched by a failed speculation).
cudaError_t k3_finish_speculative(K3Workspace &ws, const K3Params &p, cudaStream_t stream, bool *speculated) {
    K3Workspace::Impl &w = *ws.impl;
    *speculated = false;
    w.spec.reset();
    const K3Workspace::Impl::History &h = w.hist;
    if (p.n == 0 || !h.valid || h.n != p.n || h.w != p.w || h.h != p.h) return cudaSuccess;
    const Lists &l = w.l;
    const ListSizes &last = h.sizes;
    ListSizes cap;
    cap.n_long = (uint32_t)std::min<unsigned long long>((unsigned long long)last.n_long + last.n_long / 8 + 256, l.long_cap);
    cap.ckpts = (uint32_t)std::min<unsigned long long>((unsigned long long)last.ckpts + last.ckpts / 8 + 1024, l.ckpt_cap);
    cap.relays = (uint32_t)std::min<unsigned long long>((unsigned long long)last.relays + last.relays / 8 + 1024, l.relay_cap);
    cap.points = std::min(last.points + last.points / 8 + 65536, 0xfffffffeull);
    // which ordering: the per-frame ranking when the previous call's fullest frame fits its lists with room to spare
    cap.frame_long = l.frame_cap && last.frame_long + last.frame_long / 4 + 16 <= l.frame_cap ? l.frame_cap : 0xffffffffu;
    K3_CUDA(enqueue_finish(w, p, cap, w.counters.p, stream));
    w.spec = cap;
    *speculated = true;
    return cudaSuccess;
}

// Device word that is non-zero when the speculative finish in flight gave up (for kernels queued behind it).
const uint32_t *k3_speculation_failed_flag(K3Workspace &ws) { return ws.impl->counters.p ? ws.impl->counters.p + kSpecFail : nullptr; }

// After the stream of a speculative finish has been synchronised: did the real list sizes fit?  Records the sizes for the
// next call either way.
bool k3_speculation_held(K3Workspace &ws, const K3Params &p) {
    K3Workspace::Impl &w = *ws.impl;
    if (!w.spec) return false;
    const ListSizes s = read_sizes(w);
    const bool held = s.fits(*w.spec);
    record_history(w, p, s);
    w.spec.reset();
    return held;
}

}  // namespace a3
