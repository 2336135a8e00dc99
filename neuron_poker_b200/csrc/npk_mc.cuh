// npk_mc.cuh -- device code of the Monte-Carlo equity kernels (K1 uniform dealing, K1' the reference's dealer): work items,
// per-query constants, the evaluator on top of the staged tables, and one "item" function per dealer that runs a range of
// trials of one query on one warp.  Included by npk_kernels.cu (one kernel per shape) and npk_mixed.cu (all shapes in one
// persistent kernel).
#pragma once
#include "npk_device.cuh"
#include "npk_kernels.h"

namespace npk {

// ---------------------------------------------------------------------------------------------------------------------
// work items: (query, chunk of trials).  Warps pull items from a global counter (reset by the host before launch).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ long long next_item(unsigned long long* counter, int lane)
{
    unsigned long long it = 0;
    if (lane == 0) it = atomicAdd(counter, 1ull);
    return (long long)__shfl_sync(0xffffffffu, it, 0);
}

// item number -> (query slot, trial range [begin, end) relative to trial_offset)
__device__ __forceinline__ void item_range(const EquityParams& p, long long item, long long& qslot, long long& begin, long long& end)
{
    qslot = item / p.chunks;
    begin = (item - qslot * p.chunks) * p.chunk;
    end = min(p.trials, begin + (long long)p.chunk);
}

// Items of the range kernels.  PLAN = 1: a round of an adaptive range call, where p.plan = {chunk, chunks, queries} and the
// query slots p.qindex [queries] (the queries still active) are written on the device by the kernel that retired the previous
// round's queries.  PLAN = 0: queries 0..nq-1 as planned by the host.
template <int PLAN>
__device__ __forceinline__ long long range_items(const EquityParams& p)
{
    return PLAN ? (long long)p.plan[2] * p.plan[1] : p.nq * p.chunks;
}

template <int PLAN>
__device__ __forceinline__ void range_item(const EquityParams& p, long long item, long long& q, long long& begin, long long& end)
{
    if (PLAN) {
        const uint32_t chunk = p.plan[0], chunks = p.plan[1];
        const long long slot = item / chunks;
        begin = (item - slot * chunks) * chunk;
        end = min(p.trials, begin + (long long)chunk);
        NPK_CHECK(p.tables.check, slot < (long long)p.plan[2], 11);
        q = p.qindex[slot];
        NPK_CHECK(p.tables.check, q >= 0 && q < p.nq, 11);
    } else {
        item_range(p, item, q, begin, end);
    }
}

// Per-query constants shared by every trial of a work item.
struct QueryStatic {
    uint32_t hero_sum;    // desc(h0) + desc(h1)
    uint32_t hero_lo, hero_hi;     // suit-major rank masks (16 bits per suit) of the hero's cards
    uint32_t board_sum;   // sum of known board descriptors
    uint32_t board_lo, board_hi;   // suit-major rank masks of the known board cards
    uint32_t board_cnt;   // nibble-per-suit counters of known board cards, each biased by 5 (>= 8 <=> >= 3 cards)
    uint64_t known;       // bit per card id (rank-major) of hero + known board cards
};

__device__ __forceinline__ QueryStatic load_query(const EquityParams& p, const uint32_t* sdesc, long long q, int nb_known)
{
    QueryStatic s;
    const uint8_t h0 = p.hole ? p.hole[2 * q] : (uint8_t)p.inline_query;
    const uint8_t h1 = p.hole ? p.hole[2 * q + 1] : (uint8_t)(p.inline_query >> 8);
    uint32_t d0 = sdesc[h0], d1 = sdesc[h1], l, h;
    s.hero_sum = d0 + d1;
    card_bits(d0, s.hero_lo, s.hero_hi);
    card_bits(d1, l, h);
    s.hero_lo |= l; s.hero_hi |= h;
    s.known = (1ull << h0) | (1ull << h1);
    s.board_sum = 0; s.board_lo = 0; s.board_hi = 0; s.board_cnt = 0x5555u;
    for (int i = 0; i < nb_known; i++) {
        const uint8_t c = p.hole ? p.board[5 * q + i] : (uint8_t)(p.inline_query >> (16 + 8 * i));
        uint32_t d = sdesc[c];
        card_bits(d, l, h);
        s.board_sum += d; s.board_lo |= l; s.board_hi |= h; s.board_cnt += suit_inc(d);
        s.known |= 1ull << c;
    }
    return s;
}

// One-query fast path: the last warp of the grid to get here hands the counters to the host and resets them.
__device__ __forceinline__ void finish_single_call(const EquityParams& p, int lane)
{
    SingleCall* sc = p.single;
    if (!sc) return;
    __syncwarp();
    unsigned int last = 0;
    if (lane == 0) {
        __threadfence();                                              // this warp's atomics before its ticket
        const unsigned int total = gridDim.x * (blockDim.x >> 5);
        last = atomicAdd(&sc->ticket, 1u) == total - 1u;
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence();
    unsigned long long v = 0;
    if (lane < 12) {
        unsigned long long* src = &sc->wins;                           // wins, ties, win_types[9], passes are contiguous
        v = atomicExch(src + lane, 0ull);                             // read and reset for the next call
    }
    if (lane == 0) { sc->work_counter = 0; sc->ticket = 0; }
    if (lane < 12) (&sc->host->wins)[lane] = v;
    __threadfence_system();
    __syncwarp();
    if (lane == 0) *reinterpret_cast<volatile unsigned long long*>(&sc->host->seq) = p.single_seq;   // the host spins on this word
}

// Trial-sharded job: the last warp of this rank's grid exchanges the counters with the other ranks over NVLink-mapped
// peer memory and leaves the reduced totals in p.peer_totals (see PeerCall in npk_kernels.h).
static __device__ __noinline__ void finish_peer(PeerCall* pc, unsigned long long epoch, unsigned long long* totals, uint32_t words,
                                         int lane)
{
    __syncwarp();
    unsigned int last = 0;
    if (lane == 0) {
        __threadfence();                                              // this warp's atomics before its ticket
        const unsigned int total = gridDim.x * (blockDim.x >> 5);
        last = atomicAdd(&pc->ticket, 1u) == total - 1u;
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence();
    const uint32_t world = pc->world, me = pc->rank;
    const uint32_t parity = (uint32_t)(epoch & 1ull);
    const size_t my_slot = ((size_t)parity * world + me) * pc->stride;
    // push: four words per lane and batch, the reads (and resets) of the local counters first, then the peer stores --
    // independent memory operations in flight instead of one dependent round trip after the other
    for (uint32_t base = 0; base < words; base += 128) {
        unsigned long long v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t i = base + 32u * k + lane;
            v[k] = i < words ? atomicExch(&pc->acc[i], 0ull) : 0ull;                // read and reset for the next step
        }
        for (uint32_t r = 0; r < world; r++) {
            unsigned long long* dst = pc->slots[r] + my_slot;                       // NVLink for r != me
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t i = base + 32u * k + lane;
                if (i < words) dst[i] = v[k];
            }
        }
    }
    __threadfence_system();
    __syncwarp();
    if (lane < world)
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(pc->flags[lane] + parity * kMaxPeers + me), "l"(epoch) : "memory");
    if (lane < world) {
        const unsigned long long* f = pc->flags[me] + parity * kMaxPeers + lane;
        const long long t0 = clock64();
        unsigned long long seen;
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(f) : "memory");
            if (seen >= epoch) break;
            if (clock64() - t0 > (4ll << 30)) { pc->error = 1u; break; }           // ~2 s: a peer never arrived
        }
    }
    __syncwarp();
    // sum the ranks' slots of this buffer (L2 is the point of coherence for the peers' writes: ld.cg after the acquire)
    const unsigned long long* mine = pc->slots[me] + (size_t)parity * world * pc->stride;
    for (uint32_t base = 0; base < words; base += 128) {
        unsigned long long sum[4] = {0, 0, 0, 0};
#pragma unroll 4
        for (uint32_t r = 0; r < world; r++) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t i = base + 32u * k + lane;
                if (i < words) sum[k] += __ldcg(mine + (size_t)r * pc->stride + i);
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t i = base + 32u * k + lane;
            if (i < words) totals[i] = sum[k];
        }
    }
    if (lane == 0) { pc->work_counter = 0; pc->ticket = 0; }
}

// What a complete board says about flushes: at most one suit (the one holding >= 3 board cards) can still flush.
struct BoardFlush {
    uint32_t fsx;     // that suit << 4 (meaningless when thr == 64)
    uint32_t sel;     // PRMT selector of its 16-bit field
    uint32_t thr;     // 5 if a flush is possible on this board, else 64 (= never)
};

__device__ __forceinline__ BoardFlush board_flush(uint32_t board_cnt)
{
    BoardFlush b;
    const uint32_t f = board_cnt & 0x8888u;
    const uint32_t fs = ((31u - __clz(f)) >> 2) & 3u;     // & 3 keeps selector and shift legal when f == 0
    b.fsx = fs << 4;
    b.sel = field_selector(fs);
    b.thr = f ? 5u : 64u;
    return b;
}

// Flush-aware rank id: `total` = wrapped descriptor sum of the 7 cards, `field` = rank mask of the candidate flush suit.
__device__ __forceinline__ uint32_t eval_player(const SmemAddr& a, uint32_t total, uint32_t field, uint32_t thr)
{
    uint32_t v = lookup_nonflush(a, total);
    NPK_CHECK(a.check, 2u * field + 2u <= a.flush_bytes, 3);
    if ((uint32_t)__popc(field) >= thr) v = max(v, lds_u16(a.flush + 2u * field));
    return v;
}

// =====================================================================================================================
// K1: uniform dealing.  NOPP opponents, NB board cards still to come (known board = 5 - NB), two trials per lane and
// loop iteration.
//
// Dealing = partial Fisher-Yates over the N = 50 - (5 - NB) unseen cards.  Each warp owns a private copy of the deck in
// shared memory, interleaved so that lane l only ever touches bank l (element j of lane l at word j*32 + l): every
// LDS/STS of the shuffle is conflict-free whatever the random indices are.  Elements are the 32-bit card descriptors
// themselves, so a draw yields everything the evaluator needs with no decode table.  After the D = 2*NOPP + NB draws
// the D overwritten slots are restored in reverse order from registers, which leaves the deck in its canonical order
// for the next trial: the outcome of a trial depends only on (seed, query, trial), not on how trials are partitioned.
//
// Random numbers: Philox4x32-10, key = seed.  Each 32-bit word serves two draws by multiply-shift with remainder reuse:
// x*m -> (index, x'), x'*(m-1) -> index; the first draw of a word is uniform to within 2^-26, the second to within
// 2^-20 (the remainder takes 2^32/m equally spaced values).  A trial needs NW = ceil(D/2) words.  Trials are generated
// in PAIRS so that no word of a block is thrown away: pair P = trial >> 1 draws ceil(2*NW/4) blocks with counter
// (P_lo, P_hi, query, block), trial 2P reads words [0, NW), trial 2P+1 words [NW, 2*NW).  For the six-player flop
// (D = 12) that is three blocks per two trials instead of four (-20 instructions per trial, +5.6 % measured), and the
// two trials of a lane interleave in the instruction stream.  Pairs are numbered by ABSOLUTE trial number
// (trial_offset included), so the outcome of a trial still depends only on (seed, query, trial).
// A 64-bit fraction serving six draws (one Philox block for D <= 12) was built and measured in round 1: the two extra
// multiply-adds per draw cost as much as the half-pruned second block saves, so the 32-bit form stayed.
// =====================================================================================================================
__device__ __forceinline__ uint32_t lds_u32(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_u32(uint32_t saddr, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}

// What a warp of the Monte-Carlo kernels works with: the staged tables and its private deck in shared memory.
struct WarpCtx {
    SmemAddr st;
    const uint32_t* sdesc;     // [52] card descriptors (shared memory)
    uint32_t* scratch;         // 64 words of staging + the lane-interleaved deck (N * 32 words)
    uint32_t fy_addr;          // shared address of this lane's deck element 0
    int lane;
};

// Stage the tables (whole CTA) and carve this warp's deck out of the dynamic shared memory behind them.
__device__ __forceinline__ WarpCtx warp_context(const EquityParams& p, uint8_t* smem, int words_per_warp)
{
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemTables stab = stage_tables(p.tables, smem + 128, bar);
    const uint32_t table_bytes = 128 + p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes + kDescBytes;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpCtx cx;
    cx.st = smem_addr(stab);
    cx.sdesc = stab.desc;
    cx.scratch = reinterpret_cast<uint32_t*>(smem + table_bytes) + warp * words_per_warp;
    cx.fy_addr = smem_u32(cx.scratch + 64 + lane);
    cx.lane = lane;
    return cx;
}

template <int NOPP, int NB>
__device__ __forceinline__ void uniform_item(const EquityParams& p, const WarpCtx& cx, long long q, long long t_begin,
            long long t_end)
{
    constexpr int KNOWN = 5 - NB;
    constexpr int N = 50 - KNOWN;
    constexpr int D = 2 * NOPP + NB;
    constexpr int NW = (D + 1) / 2;
    constexpr int NBLK2 = (2 * NW + 3) / 4;   // Philox blocks per trial PAIR
    static_assert(D <= N, "not enough cards");

    const SmemAddr& st = cx.st;
    const int lane = cx.lane;
    uint32_t* scratch = cx.scratch;
    uint32_t* fy = scratch + 64 + lane;
    const uint32_t fy_addr = cx.fy_addr;
    const QueryStatic qs = load_query(p, cx.sdesc, q, KNOWN);

    __syncwarp();
    {
        const uint64_t avail = ~qs.known & ((1ull << 52) - 1ull);
        for (int c = lane; c < 52; c += 32)
            if (avail >> c & 1ull) scratch[__popcll(avail & ((1ull << c) - 1ull))] = cx.sdesc[c];
    }
    __syncwarp();
#pragma unroll 4
    for (int j = 0; j < N; j++) fy[j * 32] = scratch[j];
    __syncwarp();

    // absolute trial numbers [a_begin, a_end) of this item; lanes walk over absolute trial PAIRS
    const unsigned long long a_begin = (unsigned long long)(p.trial_offset + t_begin);
    const unsigned long long a_end = (unsigned long long)(p.trial_offset + t_end);
    uint32_t wins = 0, ties = 0;
    unsigned long long wt_pack = 0;

    // trial = 2 * pair + u is inside the item iff (trial - a_begin) < (a_end - a_begin) as UNSIGNED 32-bit numbers
    // (an item holds at most 2,048 trials; a trial just below a_begin wraps around to a huge value)
    const uint32_t span = (uint32_t)(a_end - a_begin);
    uint32_t rel = (uint32_t)(2ull * (a_begin >> 1) - a_begin) + 2u * (uint32_t)lane;     // 2 * pair - a_begin
    for (unsigned long long pb = a_begin >> 1; pb <= (a_end - 1) >> 1; pb += 32, rel += 64u) {
        const unsigned long long pair = pb + lane;
        uint32_t w[NBLK2 > 0 ? NBLK2 * 4 : 1];
#pragma unroll
        for (int b = 0; b < NBLK2; b++)
            philox4x32_10((uint32_t)pair, (uint32_t)(pair >> 32), (uint32_t)q + p.query_offset, (uint32_t)b,
                          p.seed_lo, p.seed_hi, &w[4 * b]);
        uint32_t dv[2][D > 0 ? D : 1];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            uint32_t slot[D > 0 ? D : 1];
            uint32_t rem = 0;
#pragma unroll
            for (int k = 0; k < D; k++) {
                const uint32_t x = (k & 1) ? rem : w[u * NW + (k >> 1)];
                const uint32_t idx = __umulhi(x, (uint32_t)(N - k));
                rem = x * (uint32_t)(N - k);
                slot[k] = fy_addr + idx * 128u;
                dv[u][k] = lds_u32(slot[k]);
                sts_u32(slot[k], lds_u32(fy_addr + (uint32_t)(N - 1 - k) * 128u));
            }
#pragma unroll
            for (int k = D - 1; k >= 0; k--) sts_u32(slot[k], dv[u][k]);
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const bool active = rel + (uint32_t)u < span;
            uint32_t bsum = qs.board_sum, bcnt = qs.board_cnt;
#pragma unroll
            for (int k = 2 * NOPP; k < D; k++) { bsum += dv[u][k]; bcnt += suit_inc(dv[u][k]); }
            const BoardFlush bf = board_flush(bcnt);
            uint32_t bfield = prmt(qs.board_lo, qs.board_hi, bf.sel);
#pragma unroll
            for (int k = 2 * NOPP; k < D; k++) bfield |= flush_bit(dv[u][k], bf.fsx);
            const uint32_t hv = eval_player(st, bsum + qs.hero_sum, bfield | prmt(qs.hero_lo, qs.hero_hi, bf.sel), bf.thr);
            uint32_t best = 0;
#pragma unroll
            for (int o = 0; o < NOPP; o++) {
                const uint32_t d0 = dv[u][2 * o], d1 = dv[u][2 * o + 1];
                best = max(best, eval_player(st, bsum + d0 + d1, bfield | flush_bit(d0, bf.fsx) | flush_bit(d1, bf.fsx), bf.thr));
            }
            const bool win = active && (NOPP == 0 || hv > best), tie = active && NOPP > 0 && hv == best;
            wins += win; ties += tie;
            if (p.win_types && (win || tie)) {
                uint32_t ty = 0;
#pragma unroll
                for (int i = 1; i < 9; i++) ty += hv >= p.tables.type_start[i];
                wt_pack += 1ull << (7 * ty);
            }
        }
    }
#ifdef NPK_CHECKED
    __syncwarp();
    for (int j = 0; j < N; j++) NPK_CHECK(st.check, fy[j * 32] == scratch[j], 7);      // every trial put its cards back
#endif
    wins = __reduce_add_sync(0xffffffffu, wins);
    ties = __reduce_add_sync(0xffffffffu, ties);
    if (lane == 0) {
        atomicAdd(&p.wins[q], (unsigned long long)wins);
        atomicAdd(&p.ties[q], (unsigned long long)ties);
    }
    if (p.win_types) {
#pragma unroll
        for (int i = 0; i < 9; i++) {
            uint32_t c = __reduce_add_sync(0xffffffffu, (uint32_t)(wt_pack >> (7 * i)) & 127u);
            if (lane == 0 && c) atomicAdd(&p.win_types[9 * q + i], (unsigned long long)c);
        }
    }
}


// =====================================================================================================================
// K1': the Python reference's dealer (tools/montecarlo_python.py:165-189), shape-specialised like K1, REJECTION-FREE.
//
// What the reference does, on the ORDERED list R of unseen cards (n of them, ascending card id):
//   opponent: i1 ~ U[0,n), i2 ~ U[0,n-1), retry while i1 == i2;  c1 = R.pop(i1); c2 = R.pop(i2)                  (:169-179)
//   board:    j ~ U[0, n-1);  c = R.pop(j)  -- the last element of R never reaches the board                      (:188)
// The accepted (i1, i2) are uniform over {i1 in [0,n), i2 in [0,n-1), i1 != i2}: (n-1)^2 pairs.  For a fixed i2 = b the
// admissible i1 are [0,n) without b, so  (a, b) uniform in [0,n-1)^2  ->  (i1, i2) = (a + (a >= b), b)  is a bijection
// onto the accepted set: the retry loop disappears and a trial is D = 2*NOPP + NB pops at known indices -- a Lehmer code.
// Decoding it needs no ordered list either.  Walking the pops BACKWARDS, un-popping pop k shifts every later pop whose
// index is >= i_k up by one; after the sweep every index is a slot of the CANONICAL (ascending, never modified) deck.
// The sweep is SIMD inside registers: four 8-bit indices per register, and for bytes x, t < 64 bit 7 of x + (0x80 - t)
// says x >= t, so  tmp = x4 + C_k;  x4 += (tmp & H) >> 7  bumps up to four later pops with three instructions
// (IADD3, LOP3, IMAD.HI -- C_k = 0x80808080 - i_k * 0x01010101 from the raw index, H = 0x80 in the bytes j > k).
// The card descriptors are then read from the warp's lane-interleaved copy of the canonical deck: ONE conflict-free LDS
// per card, no STS, no restore (K1's shuffle needs two LDS + two STS per card), no card ids, no availability mask, no
// divergence.  Round 1 drew from K1's shuffled deck and rejected on card ids: 830 executed instructions per trial, lane
// efficiency 25 of 32 (profiles/r01_ncu_refdeal_v1.txt).
//
// Random numbers: Philox4x32-10, key = seed.  A trial needs NWR = NOPP + ceil(NB/2) words: word o gives opponent o's
// (a, b) by multiply-shift with remainder reuse (a = hi32(w*(n-1)), b = hi32(lo32(w*(n-1))*(n-1))), a board word serves two
// board cards the same way.  Trials are generated in PAIRS like K1's: pair P = trial >> 1 draws ceil(2*NWR/4) blocks with
// counter (P_lo, P_hi, query, 0x80000000 + block); trial 2P reads words [0, NWR), trial 2P+1 words [NWR, 2*NWR).
// `passes` (the reference's count of draw attempts, :167) is a by-product of ITS rejection loop: an attempt fails with
// probability 1/n, independently of the pair finally dealt.  When the caller asks for it, it is drawn from that law
// (1 + a geometric number of failures per opponent) out of a separate block (counter 0x40000000 + ...), so the joint
// distribution of (cards, passes) is the reference's.
// =====================================================================================================================
struct WordStream {
    uint32_t c0, c1, c2, k0, k1, blk, have;
    uint32_t w[4];
    __device__ __forceinline__ uint32_t next()
    {
        if (have == 0) { philox4x32_10(c0, c1, c2, blk++, k0, k1, w); have = 4; }
        const uint32_t r = w[0];                 // words leave in order; the rest moves up (no dynamic indexing: the
        w[0] = w[1]; w[1] = w[2]; w[2] = w[3];   // block stays in registers instead of local memory)
        have--;
        return r;
    }
};

// k-th (0-based) set bit of a 52-bit mask, by halving on popcounts
__device__ __forceinline__ int select_bit(uint64_t m, int k)
{
    uint32_t lo = (uint32_t)m, hi = (uint32_t)(m >> 32);
    int c = __popc(lo), base = 0;
    uint32_t w = lo;
    if (k >= c) { k -= c; w = hi; base = 32; }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const uint32_t lowmask = (1u << s) - 1u;
        const int cl = __popc(w & lowmask);
        if (k >= cl) { k -= cl; w >>= s; base += s; } else { w &= lowmask; }
    }
    return base;
}

// x4 + (((x4 + c) & h) >> 7): the byte-wise "bump" of the Lehmer sweep
__device__ __forceinline__ uint32_t bump4(uint32_t x4, uint32_t c, uint32_t h)
{
    const uint32_t t = (x4 + c) & h;
    return x4 + (t >> 7);
}

// Decode D pop indices (raw[k] < 64, pop k taken from the list shortened by pops 0..k-1) into canonical slots, packed
// four per register.
template <int D>
__device__ __forceinline__ void lehmer_decode(const uint32_t (&raw)[D > 0 ? D : 1], uint32_t (&x4)[(D + 3) / 4 > 0 ? (D + 3) / 4 : 1])
{
    constexpr int G = (D + 3) / 4;
#pragma unroll
    for (int g = 0; g < G; g++) {
        uint32_t v = raw[4 * g];
#pragma unroll
        for (int b = 1; b < 4; b++)
            if (4 * g + b < D) v += raw[4 * g + b] << (8 * b);
        x4[g] = v;
    }
#pragma unroll
    for (int k = D - 2; k >= 0; k--) {
        const uint32_t c = 0x80808080u - raw[k] * 0x01010101u;       // IMAD
#pragma unroll
        for (int g = (k + 1) / 4; g < G; g++) {
            uint32_t h = 0;
#pragma unroll
            for (int b = 0; b < 4; b++)
                if (4 * g + b > k && 4 * g + b < D) h |= 0x80u << (8 * b);
            x4[g] = bump4(x4[g], c, h);
        }
    }
}

// shared address of slot j's descriptor in a lane-interleaved deck: base + 128 * byte (j & 3) of x4
__device__ __forceinline__ uint32_t slot_addr(uint32_t x4, int b, uint32_t base)
{
    const uint32_t f = x4 & (0xFFu << (8 * b));
    return b == 0 ? base + f * 128u : base + (f >> (8 * b - 7));
}

template <int NOPP, int NB>
__device__ __forceinline__ void refdeal_item(const EquityParams& p, const WarpCtx& cx, long long q, long long t_begin,
            long long t_end)
{
    constexpr int KNOWN = 5 - NB;
    constexpr int N = 50 - KNOWN;          // unseen cards
    constexpr int D = 2 * NOPP + NB;       // cards dealt per trial
    constexpr int NWR = NOPP + (NB + 1) / 2;       // Philox words per trial
    constexpr int NBLK2 = (2 * NWR + 3) / 4;       // Philox blocks per trial PAIR
    constexpr int G = (D + 3) / 4;
    static_assert(D <= N, "not enough cards");

    const SmemAddr& st = cx.st;
    const int lane = cx.lane;
    uint32_t* scratch = cx.scratch;
    uint32_t* fy = scratch + 64 + lane;
    const uint32_t fy_addr = cx.fy_addr;
    const QueryStatic qs = load_query(p, cx.sdesc, q, KNOWN);

    __syncwarp();
    {
        const uint64_t avail = ~qs.known & ((1ull << 52) - 1ull);
        for (int c = lane; c < 52; c += 32)
            if (avail >> c & 1ull) scratch[__popcll(avail & ((1ull << c) - 1ull))] = cx.sdesc[c];
    }
    __syncwarp();
#pragma unroll 4
    for (int j = 0; j < N; j++) fy[j * 32] = scratch[j];       // read-only from here on: the canonical deck
    __syncwarp();

    const unsigned long long a_begin = (unsigned long long)(p.trial_offset + t_begin);
    const unsigned long long a_end = (unsigned long long)(p.trial_offset + t_end);
    uint32_t wins = 0, ties = 0, passes = 0;        // passes <= 64 iterations * 2 * 9 opponents * a few attempts
    unsigned long long wt_pack = 0;

    const uint32_t span = (uint32_t)(a_end - a_begin);
    uint32_t rel = (uint32_t)(2ull * (a_begin >> 1) - a_begin) + 2u * (uint32_t)lane;     // 2 * pair - a_begin
    for (unsigned long long pb = a_begin >> 1; pb <= (a_end - 1) >> 1; pb += 32, rel += 64u) {
        const unsigned long long pair = pb + lane;
        uint32_t w[NBLK2 > 0 ? NBLK2 * 4 : 1];
#pragma unroll
        for (int b = 0; b < NBLK2; b++)
            philox4x32_10((uint32_t)pair, (uint32_t)(pair >> 32), (uint32_t)q + p.query_offset, 0x80000000u + (uint32_t)b,
                          p.seed_lo, p.seed_hi, &w[4 * b]);
        uint32_t dv[2][D > 0 ? D : 1];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            uint32_t raw[D > 0 ? D : 1];
#pragma unroll
            for (int o = 0; o < NOPP; o++) {
                const uint32_t m = (uint32_t)(N - 2 * o - 1);              // n - 1
                const uint32_t x = w[u * NWR + o];
                const uint32_t a = __umulhi(x, m), b = __umulhi(x * m, m);
                raw[2 * o] = a + (a >= b ? 1u : 0u);
                raw[2 * o + 1] = b;
            }
            uint32_t rem = 0;
#pragma unroll
            for (int c = 0; c < NB; c++) {
                const uint32_t m = (uint32_t)(N - 2 * NOPP - c - 1);       // n - 1: never the last element
                const uint32_t x = (c & 1) ? rem : w[u * NWR + NOPP + (c >> 1)];
                raw[2 * NOPP + c] = __umulhi(x, m);
                rem = x * m;
            }
            uint32_t x4[G > 0 ? G : 1];
            lehmer_decode<D>(raw, x4);
#pragma unroll
            for (int k = 0; k < D; k++) dv[u][k] = lds_u32(slot_addr(x4[k >> 2], k & 3, fy_addr));
        }
        if (p.passes) {
            // the reference's attempt counter: every opponent costs 1 + Geometric(1/n) attempts
            constexpr int NPB = (2 * NOPP + 3) / 4;
#pragma unroll
            for (int b = 0; b < NPB; b++) {
                uint32_t pw[4];
                philox4x32_10((uint32_t)pair, (uint32_t)(pair >> 32), (uint32_t)q + p.query_offset, 0x40000000u + (uint32_t)b,
                              p.seed_lo, p.seed_hi, pw);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int s = 4 * b + i;                                   // word s: trial s / NOPP, opponent s % NOPP
                    if (s < 2 * NOPP) {
                        const uint32_t n = (uint32_t)(N - 2 * (s % (NOPP > 0 ? NOPP : 1)));
                        uint32_t x = pw[i], tries = 1;
                        while (x < 0xFFFFFFFFu / n && tries < kMaxRangeAttempts) { tries++; x *= n; }   // x < 2^32 / n with probability 1/n
                        if (rel + (uint32_t)(s / (NOPP > 0 ? NOPP : 1)) < span) passes += tries;
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const bool active = rel + (uint32_t)u < span;
            uint32_t bsum = qs.board_sum, bcnt = qs.board_cnt;
#pragma unroll
            for (int k = 2 * NOPP; k < D; k++) { bsum += dv[u][k]; bcnt += suit_inc(dv[u][k]); }
            const BoardFlush bf = board_flush(bcnt);
            uint32_t bfield = prmt(qs.board_lo, qs.board_hi, bf.sel);
#pragma unroll
            for (int k = 2 * NOPP; k < D; k++) bfield |= flush_bit(dv[u][k], bf.fsx);
            const uint32_t hv = eval_player(st, bsum + qs.hero_sum, bfield | prmt(qs.hero_lo, qs.hero_hi, bf.sel), bf.thr);
            uint32_t best = 0;
#pragma unroll
            for (int o = 0; o < NOPP; o++) {
                const uint32_t d0 = dv[u][2 * o], d1 = dv[u][2 * o + 1];
                best = max(best, eval_player(st, bsum + d0 + d1, bfield | flush_bit(d0, bf.fsx) | flush_bit(d1, bf.fsx), bf.thr));
            }
            const bool win = active && (NOPP == 0 || hv > best), tie = active && NOPP > 0 && hv == best;
            wins += win; ties += tie;
            if (p.win_types && (win || tie)) {
                uint32_t ty = 0;
#pragma unroll
                for (int i = 1; i < 9; i++) ty += hv >= p.tables.type_start[i];
                wt_pack += 1ull << (7 * ty);
            }
        }
    }

    wins = __reduce_add_sync(0xffffffffu, wins);
    ties = __reduce_add_sync(0xffffffffu, ties);
    if (lane == 0) {
        atomicAdd(&p.wins[q], (unsigned long long)wins);
        atomicAdd(&p.ties[q], (unsigned long long)ties);
    }
    if (p.passes) {
        const uint32_t plo = __reduce_add_sync(0xffffffffu, passes & 0xffffu);
        const uint32_t phi = __reduce_add_sync(0xffffffffu, passes >> 16);
        if (lane == 0) atomicAdd(&p.passes[q], (unsigned long long)plo + ((unsigned long long)phi << 16));
    }
    if (p.win_types) {
#pragma unroll
        for (int i = 0; i < 9; i++) {
            uint32_t c = __reduce_add_sync(0xffffffffu, (uint32_t)(wt_pack >> (7 * i)) & 127u);
            if (lane == 0 && c) atomicAdd(&p.win_types[9 * q + i], (unsigned long long)c);
        }
    }
}


}  // namespace npk
