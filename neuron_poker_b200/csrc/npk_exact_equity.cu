// npk_exact_equity.cu -- exact equity of the hero against one or two UNKNOWN opponents, with any known opponent hands and dead
// cards (run_montecarlo's player_card_list beyond the hero and its ghost cards, montecarlo_python.py:132-163, 206-208), under
// uniform dealing or weighted by the reference's dealer (include/npk.h, npk_exact_equity_batch).
//
// R = the unseen cards (52 minus hero, known hands, board and dead cards) in ascending id order; slots are positions in R.
// Every completion of the board -- an m-subset of R, numbered in colexicographic order (c0 < c1 < ..., rank = sum C(c_i, i+1)) --
// is scored once for the hero and the known hands; the unknown hands are the pairs of slots the completion leaves free.
//   k = 1: a warp takes a completion and its lanes walk the hands (enum_kernel's fast path).  REFERENCE: hand a < b has weight
//          2 - [b = a+1], and its excluded slot (the highest slot left after its cards, enum_kernel's two-compare select) must
//          not be on the board.
//   k = 2: the CTA takes a completion, ranks the free hands into shared memory and walks the UNORDERED disjoint pairs once,
//          adding both orders' weights w(o1) w(o2|o1) + w(o2) w(o1|o2): w(o2|o1) = 2 - [every slot strictly between a2 and b2
//          belongs to o1].  Both orders share the excluded slot x = max(R minus the four cards): with T the completion's top
//          slot, x is on the board exactly when the four cards cover every slot above T, i.e. when the hands hold f = n-1-T
//          slots above T between them.
// The outcome is the hero against max(best known hand, unknown hands).  Counts are integers added per lane, reduced per warp and
// added to the spot's counters with one atomic per warp whenever the spot changes: they do not depend on the grid or the plan.
// With TYPES = 1 the kernel also fills win_types[9 s + t], the win + tie weight of the deals in which the hero's rank id has
// hand type t.  The hero's value is fixed for a whole completion, so each thread adds its win + tie weight of the completion
// to one of nine register bins (constant indices, selected by the type) once the completion's hands are walked, and the bins
// are flushed like the counts: at most one atomic per non-zero bin per warp and spot.
//
// Work split (npk_enum_plan.cuh): one global sequence of units over the batch, a completion is one unit with one unknown
// opponent and kEeUnitsK2 with two (about the ratio of their work); it belongs to the item that holds its first unit.  Items
// are taken per CTA.  Three kernels, all on the caller's stream and without a host round trip:
//   ee_prepare_kernel   per spot: units, zeroed outputs
//   ee_plan_kernel      one CTA: prefix of the units, item size, work counter reset
//   exact_equity_kernel<REF, TYPES>  persistent, one CTA per SM: tables staged once per CTA, CTAs pull items from the work counter
#include <algorithm>
#include "npk_enum_plan.cuh"
#include "npk_mc.cuh"

namespace npk {

constexpr int kEeThreads = 512;
constexpr int kEeWarps = kEeThreads / 32;
constexpr unsigned long long kEeUnitsK2 = 256;
// units per item: about four items per CTA, at least one completion per warp.  A lane then adds below 2^32: at most 2^16 + 1
// one-opponent completions of <= 42 hands of weight <= 2, or 2^12 two-opponent completions of <= 83 x 42 pairs of weight <= 8.
// A win-type bin holds part of the lane's win + tie, so it stays below 2^32 too.
constexpr unsigned long long kEeMinItem = kEeWarps, kEeMaxItem = 1ull << 20;
// dynamic shared memory behind the tables: descriptors [64] | pair list [1326] u16 | C(c, k) [6][64] u32 | R [64] u32 |
// free cards of the current completion, per warp and one for the CTA: descriptors [17][64] u32, R slots [17][64] u8 |
// ranked hands [1326] u32
constexpr uint32_t kEePairOff = kDescBytes, kEeBinomOff = kEePairOff + 2688, kEeDeckOff = kEeBinomOff + 6 * 64 * 4,
                   kEeFreeOff = kEeDeckOff + 256, kEeSlotOff = kEeFreeOff + (kEeWarps + 1) * 256,
                   kEeHandOff = kEeSlotOff + (kEeWarps + 1) * 64, kEeExtraBytes = kEeHandOff + 1326 * 4;

// workspace: the plan (npk_enum_plan.cuh), then the units of every spot
long long exact_equity_workspace_bytes(long long n) { return plan_workspace_bytes(n) + 8 * (n > 0 ? n : 0); }

__device__ __forceinline__ unsigned long long* ee_units(const ExactEquityParams& p)
{
    return reinterpret_cast<unsigned long long*>(p.workspace + plan_workspace_bytes(p.n));
}

struct EeSpot {
    uint64_t avail;    // R, one bit per id
    int n;             // |R|
    int missing;       // board cards to come
    int k;             // unknown opponents; 0 when n_known / n_random are out of range
    int nk;            // hands in `holes` that take part, hero included
};

// Ids are clamped to the 64-slot descriptor table and the dead mask to 52 bits: any bytes give a memory-safe spot.
__device__ __forceinline__ EeSpot ee_spot(const ExactEquityParams& p, long long s)
{
    EeSpot sp;
    const int nk = p.n_known[s], kr = p.n_random[s];
    const bool ok = nk >= 1 && nk <= p.maxk && (kr == 1 || kr == 2) && nk + kr <= 10;
    sp.nk = ok ? nk : 0;
    sp.k = ok ? kr : 0;
    uint64_t seen = p.dead ? p.dead[s] : 0ull;
    for (int i = 0; i < 2 * sp.nk; i++) seen |= 1ull << (p.holes[2 * p.maxk * s + i] & 63u);
    int nb = 0;
    for (int i = 0; i < 5; i++) {
        const uint32_t c = p.board[5 * s + i];
        if (c != 0xFFu) { seen |= 1ull << (c & 63u); nb++; }
    }
    sp.avail = ~seen & ((1ull << 52) - 1ull);
    sp.n = __popcll(sp.avail);
    sp.missing = 5 - nb;
    return sp;
}

__global__ void __launch_bounds__(256) ee_prepare_kernel(const ExactEquityParams p)
{
    unsigned long long* units = ee_units(p);
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < p.n; s += (long long)gridDim.x * blockDim.x) {
        const EeSpot sp = ee_spot(p, s);
        units[s] = sp.k && sp.n >= 2 * sp.k + sp.missing ? plan_binom(sp.n, sp.missing) * (sp.k == 2 ? kEeUnitsK2 : 1ull) : 0ull;
        p.win[s] = 0; p.tie[s] = 0; p.lose[s] = 0;
        if (p.win_types)
            for (int t = 0; t < 9; t++) p.win_types[9 * s + t] = 0;
    }
}

__global__ void __launch_bounds__(kPlanThreads) ee_plan_kernel(const ExactEquityParams p)
{
    plan_items(ee_units(p), p.n, p.workspace, 4ull * (unsigned long long)p.sm_count, kEeWarps, kEeMinItem, kEeMaxItem);
}

struct EeSmem {
    const uint32_t* desc;      // [64], ids 52..63 -> 0
    const uint16_t* pair;      // [1326] a | b << 8, number C(b,2) + a
    const uint32_t* binom;     // [k * 64 + c] = C(c, k), k = 0..5
    const uint32_t* deck;      // [52] descriptors of R
    uint32_t* free;            // [64] descriptors of the cards the completion leaves (this warp's, or the CTA's for k = 2)
    uint8_t* slot;             // [64] their slots in R
    uint32_t* hand;            // [1326] ranked hands (k = 2)
};

struct EeBoard {
    uint32_t sum, cnt, lo, hi; // known board cards: descriptor sum, suit counters biased by 5, suit-major rank masks
};

// completion number r -> its slots c[0..m-1], ascending
__device__ __forceinline__ void ee_unrank(const ExactEquityParams& p, const uint32_t* binom, int n, int m, uint32_t r, int (&c)[5])
{
#pragma unroll
    for (int i = 4; i >= 0; i--) {
        if (i < m) {
            int x = i + 1 < m ? c[i + 1 < 5 ? i + 1 : 4] - 1 : n - 1;
            while (x > i && binom[(i + 1) * 64 + x] > r) x--;
            c[i] = x;
            r -= binom[(i + 1) * 64 + x];
            NPK_CHECK(p.tables.check, x >= 0 && x < n, 12);
        }
    }
}

// the next completion in colexicographic order
__device__ __forceinline__ void ee_next(int n, int m, int (&c)[5])
{
    bool moved = false;
#pragma unroll
    for (int j = 0; j < 5; j++) {
        if (j < m && !moved) {
            const int ub = j + 1 < m ? c[j + 1 < 5 ? j + 1 : 4] : n;
            if (c[j] + 1 < ub) { c[j]++; moved = true; }
            else c[j] = j;
        }
    }
}

struct EeTable {
    uint32_t sum, field;
    BoardFlush bf;
};

// the complete board: the known cards plus the completion's slots of R
__device__ __forceinline__ EeTable ee_table(const EeBoard& kb, const uint32_t* deck, int m, const int (&c)[5])
{
    uint32_t sum = kb.sum, cnt = kb.cnt, lo = kb.lo, hi = kb.hi;
#pragma unroll
    for (int i = 0; i < 5; i++) {
        if (i < m) {
            const uint32_t d = deck[c[i] & 63];
            uint32_t l, h;
            card_bits(d, l, h);
            sum += d; cnt += suit_inc(d); lo |= l; hi |= h;
        }
    }
    EeTable t;
    t.bf = board_flush(cnt);
    t.sum = sum;
    t.field = prmt(lo, hi, t.bf.sel);
    return t;
}

__device__ __forceinline__ uint32_t ee_eval(const SmemAddr& st, const EeTable& t, uint32_t d0, uint32_t d1)
{
    return eval_player(st, t.sum + d0 + d1, t.field | flush_bit(d0, t.bf.fsx) | flush_bit(d1, t.bf.fsx), t.bf.thr);
}

// the hero's value and the best value of the known opponents (0 without any)
__device__ __forceinline__ void ee_known(const ExactEquityParams& p, const SmemAddr& st, const uint32_t* desc, const EeTable& t,
                                         long long s, int nk, uint32_t& hv, uint32_t& kv)
{
    const uint8_t* h = p.holes + 2 * p.maxk * s;
    hv = ee_eval(st, t, desc[h[0] & 63u], desc[h[1] & 63u]);
    kv = 0;
    for (int q = 1; q < nk; q++) kv = max(kv, ee_eval(st, t, desc[h[2 * q] & 63u], desc[h[2 * q + 1] & 63u]));
}

// sum the lanes' counts of spot s and add them to its outputs
__device__ __forceinline__ void ee_flush(const ExactEquityParams& p, long long s, uint32_t w, uint32_t t, uint32_t l, int lane)
{
    unsigned long long W = w, T = t, L = l;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        W += __shfl_down_sync(0xffffffffu, W, o);
        T += __shfl_down_sync(0xffffffffu, T, o);
        L += __shfl_down_sync(0xffffffffu, L, o);
    }
    if (lane == 0) {
        if (W) atomicAdd(&p.win[s], W);
        if (T) atomicAdd(&p.tie[s], T);
        if (L) atomicAdd(&p.lose[s], L);
    }
}

// the hand type of rank id v (0 high card .. 8 straight flush)
__device__ __forceinline__ uint32_t ee_type(const ExactEquityParams& p, uint32_t v)
{
    const uint32_t ty = hand_type(p.tables, v);
    NPK_CHECK(p.tables.check, ty < 9, 13);
    return ty;
}

// add d, a thread's win + tie weight of one completion, to the bin of the hero's type ty
__device__ __forceinline__ void ee_bin(uint32_t (&bins)[9], uint32_t ty, uint32_t d)
{
#pragma unroll
    for (int t = 0; t < 9; t++) bins[t] += t == (int)ty ? d : 0u;
}

// sum the lanes' win-type bins of spot s and add the non-zero ones to its outputs
__device__ __forceinline__ void ee_flush_types(const ExactEquityParams& p, long long s, const uint32_t (&bins)[9], int lane)
{
#pragma unroll
    for (int t = 0; t < 9; t++) {
        if (!__any_sync(0xffffffffu, bins[t])) continue;
        unsigned long long B = bins[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) B += __shfl_down_sync(0xffffffffu, B, o);
        if (lane == 0) atomicAdd(&p.win_types[9 * s + t], B);
    }
}

// the free cards of a completion (slot mask cm) into free / slot, by `count` threads starting at `t`
__device__ __forceinline__ void ee_free_cards(const EeSmem& sm, int n, uint64_t cm, int t, int count)
{
    for (int j = t; j < n; j += count) {
        if (!(cm >> j & 1ull)) {
            const int ci = j - __popcll(cm & ((1ull << j) - 1ull));
            sm.free[ci] = sm.deck[j];
            sm.slot[ci] = (uint8_t)j;
        }
    }
}

__device__ __forceinline__ uint64_t ee_mask(int m, const int (&c)[5])
{
    uint64_t cm = 0;
#pragma unroll
    for (int i = 0; i < 5; i++)
        if (i < m) cm |= 1ull << (c[i] & 63);
    return cm;
}

// One unknown opponent: completions r0..r1-1 of spot s, split over the warps (several warps share a completion when there
// are fewer completions than warps); the lanes walk the free hands.
template <int REF, int TYPES>
__device__ __forceinline__ void ee_one(const ExactEquityParams& p, const SmemAddr& st, const EeSmem& sm, const EeSpot& sp,
                                       const EeBoard& kb, long long s, uint32_t r0, uint32_t r1, int warp, int lane)
{
    const uint32_t nc = r1 - r0;
    const int wpc = nc >= (uint32_t)kEeWarps ? 1 : kEeWarps / (int)nc;    // warps sharing one completion
    const int groups = kEeWarps / wpc, g = warp / wpc, sub = warp % wpc;
    uint32_t win = 0, tie = 0, lose = 0;
    uint32_t bins[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (g < groups) {
        const uint32_t q0 = r0 + (uint32_t)((unsigned long long)nc * g / groups);
        const uint32_t q1 = r0 + (uint32_t)((unsigned long long)nc * (g + 1) / groups);
        const int n = sp.n, m = sp.missing, nf = n - m, H = nf * (nf - 1) / 2;
        int c[5] = {0, 0, 0, 0, 0};
        if (q0 < q1) ee_unrank(p, sm.binom, n, m, q0, c);
        for (uint32_t q = q0; q < q1; q++) {
            if (q > q0) ee_next(n, m, c);
            const uint64_t cm = ee_mask(m, c);
            __syncwarp();
            ee_free_cards(sm, n, cm, lane, 32);
            __syncwarp();
            const EeTable t = ee_table(kb, sm.deck, m, c);
            uint32_t hv, kv;
            ee_known(p, st, sm.desc, t, s, sp.nk, hv, kv);
            const uint32_t wt0 = win + tie;
            for (int ip = sub * 32 + lane; ip < H; ip += 32 * wpc) {
                NPK_CHECK(p.tables.check, ip < 1326, 12);
                const uint32_t pr = sm.pair[ip];
                const int a = pr & 255, b = pr >> 8;
                NPK_CHECK(p.tables.check, a < b && b < nf, 12);
                uint32_t w = 1;
                if (REF) {
                    const int A = sm.slot[a], B = sm.slot[b];
                    const int x = B != n - 1 ? n - 1 : (A != n - 2 ? n - 2 : n - 3);    // the hand's excluded slot
                    if (cm >> (x & 63) & 1ull) continue;
                    w = 2 - (B == A + 1);
                }
                const uint32_t best = max(kv, ee_eval(st, t, sm.free[a], sm.free[b]));
                win += hv > best ? w : 0u; tie += hv == best ? w : 0u; lose += hv < best ? w : 0u;
            }
            if (TYPES) ee_bin(bins, ee_type(p, hv), win + tie - wt0);
        }
    }
    ee_flush(p, s, win, tie, lose, lane);
    if (TYPES) ee_flush_types(p, s, bins, lane);
}

// Two unknown opponents: completions r0..r1-1 of spot s, one at a time on the whole CTA.
template <int REF, int TYPES>
__device__ __forceinline__ void ee_two(const ExactEquityParams& p, const SmemAddr& st, const EeSmem& sm, const EeSpot& sp,
                                       const EeBoard& kb, long long s, uint32_t r0, uint32_t r1, int warp, int lane)
{
    const int n = sp.n, m = sp.missing, nf = n - m, H = nf * (nf - 1) / 2;
    uint32_t win = 0, tie = 0, lose = 0;
    uint32_t bins[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int c[5] = {0, 0, 0, 0, 0};
    ee_unrank(p, sm.binom, n, m, r0, c);
    for (uint32_t r = r0; r < r1; r++) {
        if (r > r0) ee_next(n, m, c);
        const uint64_t cm = ee_mask(m, c);
        int top = n;                                           // the completion's top slot (n: no board card to come)
#pragma unroll
        for (int i = 0; i < 5; i++)
            if (i < m) top = c[i];
        const uint32_t f = m ? (uint32_t)(n - 1 - top) : 99u;  // slots above it: x is on the board iff the hands hold them all
        __syncthreads();                                       // the previous completion's pair walk is done
        ee_free_cards(sm, n, cm, threadIdx.x, kEeThreads);
        __syncthreads();
        const EeTable t = ee_table(kb, sm.deck, m, c);
        for (int h = threadIdx.x; h < H; h += kEeThreads) {
            NPK_CHECK(p.tables.check, h < 1326, 12);
            const uint32_t pr = sm.pair[h];
            const int a = pr & 255, b = pr >> 8;
            NPK_CHECK(p.tables.check, a < b && b < nf, 12);
            const uint32_t A = sm.slot[a], B = sm.slot[b];
            // value | slot a << 13 | slot b << 19 | cards above the top slot << 25 | adjacent << 27
            sm.hand[h] = ee_eval(st, t, sm.free[a], sm.free[b]) | A << 13 | B << 19 |
                         ((uint32_t)((int)A > top) + (uint32_t)((int)B > top)) << 25 | (uint32_t)(B == A + 1) << 27;
        }
        uint32_t hv, kv;
        ee_known(p, st, sm.desc, t, s, sp.nk, hv, kv);
        const uint32_t wt0 = win + tie;
        __syncthreads();
        for (int i1 = warp; i1 < H; i1 += kEeWarps) {
            const uint32_t h1 = sm.hand[i1];
            const int A1 = h1 >> 13 & 63, B1 = h1 >> 19 & 63;
            const uint32_t kv1 = max(kv, h1 & 8191u), hc1 = h1 >> 25 & 3u, w1 = 2 - (h1 >> 27 & 1u);
            for (int i2 = i1 + 1 + lane; i2 < H; i2 += 32) {
                NPK_CHECK(p.tables.check, i2 < 1326, 12);
                const uint32_t h2 = sm.hand[i2];
                const int A2 = h2 >> 13 & 63, B2 = h2 >> 19 & 63;
                // the list is ordered by the higher card, so a hand after h1 that shares no card has B2 > B1 (and A1 != B2)
                if (A2 == A1 || A2 == B1 || B2 == B1) continue;
                uint32_t w = 2;                                // UNIFORM: the two orders, once each
                if (REF) {
                    if (hc1 + (h2 >> 25 & 3u) == f) continue;
                    // o2 dealt after o1: o1's cards strictly between A2 and B2 are A1 if A2 < A1 and B1 if A2 < B1 (B1 < B2);
                    // o1 dealt after o2: only A2 can lie strictly between A1 and B1
                    const int btw12 = (A2 < A1) + (A2 < B1), btw21 = A1 < A2 && A2 < B1;
                    w = w1 * (2 - (B2 - A2 - 1 == btw12)) + (2 - (h2 >> 27 & 1u)) * (2 - (B1 - A1 - 1 == btw21));
                }
                const uint32_t best = max(kv1, h2 & 8191u);
                win += hv > best ? w : 0u; tie += hv == best ? w : 0u; lose += hv < best ? w : 0u;
            }
        }
        if (TYPES) ee_bin(bins, ee_type(p, hv), win + tie - wt0);
    }
    ee_flush(p, s, win, tie, lose, lane);
    if (TYPES) ee_flush_types(p, s, bins, lane);
}

template <int REF, int TYPES>
__global__ void __launch_bounds__(kEeThreads, 1) exact_equity_kernel(const ExactEquityParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ long long s_item;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemAddr st = smem_addr(stage_tables(p.tables, smem + 128, bar));
    uint8_t* extra = smem + 128 + p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes;
    uint32_t* s_desc = reinterpret_cast<uint32_t*>(extra);
    uint16_t* s_pair = reinterpret_cast<uint16_t*>(extra + kEePairOff);
    uint32_t* s_binom = reinterpret_cast<uint32_t*>(extra + kEeBinomOff);
    uint32_t* s_deck = reinterpret_cast<uint32_t*>(extra + kEeDeckOff);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 64) s_desc[threadIdx.x] = threadIdx.x < 52 ? p.tables.desc[threadIdx.x] : 0u;
    for (int i = threadIdx.x; i < 1326; i += blockDim.x) {
        int b = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)i)) * 0.5f);
        while (b * (b - 1) / 2 > i) b--;
        while ((b + 1) * b / 2 <= i) b++;
        s_pair[i] = (uint16_t)((i - b * (b - 1) / 2) | b << 8);
    }
    for (int i = threadIdx.x; i < 6 * 64; i += blockDim.x) s_binom[i] = (uint32_t)plan_binom(i & 63, i >> 6);
    EeSmem sm1, sm2;                                           // one opponent: this warp's free cards; two: the CTA's
    sm1.desc = sm2.desc = s_desc; sm1.pair = sm2.pair = s_pair; sm1.binom = sm2.binom = s_binom; sm1.deck = sm2.deck = s_deck;
    sm1.hand = sm2.hand = reinterpret_cast<uint32_t*>(extra + kEeHandOff);
    sm1.free = reinterpret_cast<uint32_t*>(extra + kEeFreeOff) + 64 * warp;
    sm1.slot = extra + kEeSlotOff + 64 * warp;
    sm2.free = reinterpret_cast<uint32_t*>(extra + kEeFreeOff) + 64 * kEeWarps;
    sm2.slot = extra + kEeSlotOff + 64 * kEeWarps;

    const unsigned long long* prefix = reinterpret_cast<const unsigned long long*>(p.workspace + kPlanWsPrefix);
    unsigned long long* counter = reinterpret_cast<unsigned long long*>(p.workspace + kPlanWsCounter);
    const unsigned long long total = prefix[p.n];
    const unsigned long long item_size = *reinterpret_cast<const uint32_t*>(p.workspace + kPlanWsItem);
    const long long n_items = (long long)((total + item_size - 1) / item_size);
    for (;;) {
        __syncthreads();                                       // tables staged / the previous item's readers of s_item done
        if (threadIdx.x == 0) s_item = (long long)atomicAdd(counter, 1ull);
        __syncthreads();
        const long long item = s_item;
        if (item >= n_items) break;
        unsigned long long g0 = (unsigned long long)item * item_size;
        const unsigned long long g1 = min(total, g0 + item_size);
        // the spot holding unit g0: the last s with prefix[s] <= g0, by a 32-way search (every warp finds the same)
        long long s = 0, hi = p.n;
        while (hi - s > 1) {
            const long long step = (hi - s + 31) / 32, idx = s + (long long)(lane + 1) * step;
            const unsigned int le = __ballot_sync(0xffffffffu, idx < hi && prefix[idx] <= g0);
            s += (long long)__popc(le) * step;
            hi = min(hi, s + step);
        }
        for (; g0 < g1; s++) {
            const unsigned long long a = prefix[s], b = prefix[s + 1];
            if (b <= g0) continue;                             // a spot without units
            const unsigned long long e = min(g1, b);
            const EeSpot sp = ee_spot(p, s);
            const unsigned long long u = sp.k == 2 ? kEeUnitsK2 : 1ull;
            // completion r starts at unit a + r u: this item holds those starting in [g0, e)
            const uint32_t r0 = (uint32_t)((g0 - a + u - 1) / u), r1 = (uint32_t)((e - a + u - 1) / u);
            g0 = e;
            if (r0 >= r1) continue;
            __syncthreads();                                   // the previous spot's readers of s_deck are done
            for (int c = threadIdx.x; c < 52; c += blockDim.x)
                if (sp.avail >> c & 1ull) s_deck[__popcll(sp.avail & ((1ull << c) - 1ull))] = s_desc[c];
            __syncthreads();
            EeBoard kb{0u, 0x5555u, 0u, 0u};
            for (int i = 0; i < 5; i++) {
                const uint32_t c = p.board[5 * s + i];
                if (c == 0xFFu) continue;
                const uint32_t d = s_desc[c & 63u];
                uint32_t l, h;
                card_bits(d, l, h);
                kb.sum += d; kb.cnt += suit_inc(d); kb.lo |= l; kb.hi |= h;
            }
            if (sp.k == 1) ee_one<REF, TYPES>(p, st, sm1, sp, kb, s, r0, r1, warp, lane);
            else ee_two<REF, TYPES>(p, st, sm2, sp, kb, s, r0, r1, warp, lane);
        }
    }
}

cudaError_t launch_exact_equity(const ExactEquityParams& p, int deal_mode, cudaStream_t s)
{
    const int prep_grid = (int)std::min<long long>((p.n + 255) / 256, 8ll * p.sm_count);
    ee_prepare_kernel<<<prep_grid, 256, 0, s>>>(p);
    ee_plan_kernel<<<1, kPlanThreads, 0, s>>>(p);
    const size_t smem = 128 + (size_t)p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes + kEeExtraBytes;
    auto k = p.win_types ? (deal_mode == 1 ? exact_equity_kernel<1, 1> : exact_equity_kernel<0, 1>)
                         : (deal_mode == 1 ? exact_equity_kernel<1, 0> : exact_equity_kernel<0, 0>);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<p.sm_count, kEeThreads, smem, s>>>(p);
    return cudaGetLastError();
}

}  // namespace npk
