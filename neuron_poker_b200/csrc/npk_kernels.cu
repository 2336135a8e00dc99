// npk_kernels.cu -- hand-written sm_100a kernels for neuron_poker's Monte-Carlo equity hot path.
//
//   equity_uniform_kernel<NOPP,NB>  K1  batched (query x trial) Monte-Carlo, uniform dealing
//                                       replaces MonteCarlo.run_montecarlo's loop (reference montecarlo_python.py:210-239)
//                                       with the C++ sibling's dealing semantics (Montecarlo.cpp:293-312)
//   equity_refdeal_kernel<NOPP,NB>  K1' same loop with the Python reference's own (biased) dealer
//                                       (montecarlo_python.py:165-189)
//   equity_ranges_kernel<MODE,PLAN> K1'' generic dealer with opponent / hero ranges and ghost cards (the reference's attempt
//                                       loop played literally; the pair-list sampler lives in npk_ranges.cu, the persistent
//                                       all-shapes kernel for mixed batches in npk_mixed.cu, the per-trial code in npk_mc.cuh)
//   rank7_kernel / rank7_colex      K2  batched 7-card rank ids (hand_evaluator.py:27-119 `_calc_score` ordering)
//   enum_headsup_kernel             K3  exact heads-up enumeration of opponents and missing board cards
//   showdown_kernel                 K4  batched get_winner (hand_evaluator.py:9-17)
//
// Everything is integer work on 32-bit lanes: no tensor cores, no floating point.  Two trials per lane and iteration; the rank
// tables (about 129 KB) are staged once per CTA into shared memory by the bulk-copy engine and gathered with 16-bit
// LDS; win / tie counts are reduced with warp REDUX and one 64-bit RED per (warp, work item).
#include <atomic>
#include <cstdlib>
#include "npk_mc.cuh"

namespace npk {

// One kernel per shape and dealer: the warps pull the (query, trial range) items of queries 0..nq-1.  A rank of a sharded job
// without trials runs one CTA without items, which still takes part in the peer exchange.
template <int NOPP, int NB, int REF>
__device__ __forceinline__ void shape_kernel_body(const EquityParams& p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const WarpCtx cx = warp_context(p, smem, 64 + (45 + NB) * 32);
    const int lane = cx.lane;
    const long long n_items = p.nq * p.chunks;
    for (long long item = next_item(p.work_counter, lane); item < n_items; item = next_item(p.work_counter, lane)) {
        long long q, t_begin, t_end;
        item_range(p, item, q, t_begin, t_end);
        if (REF) refdeal_item<NOPP, NB>(p, cx, q, t_begin, t_end);
        else uniform_item<NOPP, NB>(p, cx, q, t_begin, t_end);
    }
    finish_single_call(p, lane);
    if (p.peer) finish_peer(p.peer, p.peer_epoch, p.peer_totals, p.peer_words, lane);
}

template <int NOPP, int NB>
__global__ void __launch_bounds__(kEquityMaxThreads, 1) equity_uniform_kernel(const EquityParams p)
{
    shape_kernel_body<NOPP, NB, 0>(p);
}

template <int NOPP, int NB>
__global__ void __launch_bounds__(kEquityMaxThreads, 1) equity_refdeal_kernel(const EquityParams p)
{
    shape_kernel_body<NOPP, NB, 1>(p);
}

// =====================================================================================================================
// K1'': dealing with ranges (SURVEY 8f-2).  Opponents -- and optionally the hero -- hold only hands whose starting-hand
// class is in a 169-bit mask; ghost cards are removed from the deck first.  Reference: montecarlo_python.py:24-34
// (class of two cards), :136-148 (hero drawn from a range), :165-181 (opponent range test), :206-208 (ghost cards).
//   REFERENCE (MODE 1): i1 = hi32(w*n), i2 = hi32(lo32(w*n)*(n-1)); retry while i1 == i2 or the class of
//       (deck[i1], deck[i2]) -- both read BEFORE anything is popped (:173-174) -- is not allowed.  A hero keeps exactly
//       those two cards (:146-148); an opponent receives deck.pop(i1) and then deck.pop(i2) from the SHORTENED list
//       (:178-179), so for i2 >= i1 the tested and the dealt second card differ (reference quirk, kept).
//       Board card j = hi32(w*(n-1)) (:188).  With a full mask and a fixed hero this samples the distribution of K1' (index-based instead of shuffle-based).
//   UNIFORM (MODE 0): c1 = deck[i1], c2 = (deck without c1)[i2], retry while their class is not allowed; board uniform.
// One Philox word per attempt, blocks from 0x80000000 (REFERENCE) / 0xC0000000 (UNIFORM).  A draw that needs more than
// kMaxRangeAttempts attempts raises p.abort_flag; every warp then stops at its next trial (the host reports the error).
// =====================================================================================================================
__device__ __forceinline__ bool class_allowed(const uint32_t (&mask)[6], int c1, int c2)
{
    const int r1 = c1 >> 2, r2 = c2 >> 2, hi = max(r1, r2), lo = min(r1, r2);
    const int k = ((c1 ^ c2) & 3) == 0 ? hi * 13 + lo : lo * 13 + hi;
    return (mask[k >> 5] >> (k & 31)) & 1u;
}

// PLAN = 1: a round of an adaptive call (npk_equity_ranges_batch_adaptive), whose items are planned on the device.
template <int MODE, int PLAN>
__global__ void __launch_bounds__(kRefThreads, 1) equity_ranges_kernel(const EquityParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemAddr st = smem_addr(stage_tables(p.tables, smem + 128, bar));
    const int lane = threadIdx.x & 31;

    const long long n_items = range_items<PLAN>(p);

    for (long long item = next_item(p.work_counter, lane); item < n_items; item = next_item(p.work_counter, lane)) {
        long long q, t_begin, t_end;
        range_item<PLAN>(p, item, q, t_begin, t_end);
        int known = 0;
        for (int i = 0; i < 5; i++) known += p.board[5 * q + i] != 0xFF;
        // opponents dealt at random; the others' cards are known (montecarlo_python.py:132-163: removed from the deck like the
        // hero's, part of the showdown like any opponent)
        const int nknown = (int)p.n_known;
        const int nopp = max(0, (int)p.n_players[q] - 1 - nknown);

        // static part of the query: the known board, the cards nobody can receive
        uint64_t taken = 0;
        uint32_t board_sum = 0, board_lo = 0, board_hi = 0, board_cnt = 0x5555u;
        for (int i = 0; i < known; i++) {
            const uint8_t c = p.board[5 * q + i];
            const uint32_t d = p.tables.desc[c];
            uint32_t l, h;
            card_bits(d, l, h);
            board_sum += d; board_lo |= l; board_hi |= h; board_cnt += suit_inc(d);
            taken |= 1ull << c;
        }
        if (p.ghost)
            for (int i = 0; i < 2; i++) { const uint8_t c = p.ghost[2 * q + i]; if (c < 52) taken |= 1ull << c; }
        int h0 = 0, h1 = 0;
        if (!p.hero_range) { h0 = p.hole[2 * q]; h1 = p.hole[2 * q + 1]; taken |= (1ull << h0) | (1ull << h1); }
        for (int f = 0; f < 2 * nknown; f++) taken |= 1ull << (p.known_opp[2 * q * nknown + f] & 63u);
        const uint64_t avail0 = ~taken & ((1ull << 52) - 1ull);
        const int n0 = __popcll(avail0);

        uint32_t wins = 0, ties = 0;
        unsigned long long passes = 0;
        unsigned long long wt_pack = 0;

        for (long long tb = t_begin; tb < t_end; tb += 32) {
            if (*reinterpret_cast<volatile uint32_t*>(p.abort_flag)) break;
            const long long t_local = tb + lane;
            bool active = t_local < t_end;
            const unsigned long long trial = (unsigned long long)(p.trial_offset + t_local);
            WordStream rs;
            rs.c0 = (uint32_t)trial; rs.c1 = (uint32_t)(trial >> 32); rs.c2 = (uint32_t)q + p.query_offset;
            rs.k0 = p.seed_lo; rs.k1 = p.seed_hi; rs.blk = MODE == 1 ? 0x80000000u : 0xC0000000u; rs.have = 0;

            uint64_t avail = avail0;
            int n = n0;
            uint32_t hd0 = 0, hd1 = 0, best = 0;
            uint32_t oc1[9], oc2[9];
            if (active) {
                // hand 0 = the hero when drawn from a range, hands 1.. = the opponents
                for (int o = p.hero_range ? -1 : 0; o < nopp && active; o++) {
                    const bool is_hero = o < 0;
                    int c1 = 0, c2 = 0;
                    uint32_t tries = 0;
                    for (;;) {
                        if (++tries > kMaxRangeAttempts) { atomicExch(p.abort_flag, 1u); active = false; break; }
                        passes++;
                        const uint64_t prod = (uint64_t)rs.next() * (uint32_t)n;
                        const uint32_t i1 = (uint32_t)(prod >> 32);
                        const uint32_t i2 = __umulhi((uint32_t)prod, (uint32_t)(n - 1));
                        if (MODE == 1 && i1 == i2) continue;
                        c1 = select_bit(avail, (int)i1);
                        if (MODE == 1) {
                            const int ct = select_bit(avail, (int)i2);           // tested BEFORE popping c1
                            if (!(is_hero ? class_allowed(p.hero_mask, c1, ct) : class_allowed(p.opp_mask, c1, ct))) continue;
                            c2 = is_hero ? ct : select_bit(avail & ~(1ull << c1), (int)i2);
                        } else {
                            c2 = select_bit(avail & ~(1ull << c1), (int)i2);
                            if (!(is_hero ? class_allowed(p.hero_mask, c1, c2) : class_allowed(p.opp_mask, c1, c2))) continue;
                        }
                        break;
                    }
                    avail &= ~((1ull << c1) | (1ull << c2));
                    n -= 2;
                    if (is_hero) { h0 = c1; h1 = c2; }
                    else { oc1[o] = p.tables.desc[c1]; oc2[o] = p.tables.desc[c2]; }
                }
            }
            hd0 = p.tables.desc[h0]; hd1 = p.tables.desc[h1];
            uint32_t bsum = board_sum, bcnt = board_cnt;
            uint32_t bd[5];
            int nbd = 0;
            if (active) {
                for (int k = known; k < 5; k++) {
                    const uint32_t j = __umulhi(rs.next(), (uint32_t)(MODE == 1 ? n - 1 : n));
                    const int c = select_bit(avail, (int)j);
                    avail &= ~(1ull << c);
                    n--;
                    const uint32_t d = p.tables.desc[c];
                    bd[nbd++] = d;
                    bsum += d; bcnt += suit_inc(d);
                }
            }
            const BoardFlush bf = board_flush(bcnt);
            uint32_t bfield = prmt(board_lo, board_hi, bf.sel);
            for (int k = 0; k < nbd; k++) bfield |= flush_bit(bd[k], bf.fsx);
            const uint32_t hv = eval_player(st, bsum + hd0 + hd1, bfield | flush_bit(hd0, bf.fsx) | flush_bit(hd1, bf.fsx), bf.thr);
            if (active) {
                for (int o = 0; o < nopp; o++)
                    best = max(best, eval_player(st, bsum + oc1[o] + oc2[o],
                                                 bfield | flush_bit(oc1[o], bf.fsx) | flush_bit(oc2[o], bf.fsx), bf.thr));
                for (int f = 0; f < nknown; f++) {
                    const uint32_t k1 = p.tables.desc[p.known_opp[2 * (q * nknown + f)] & 63u];
                    const uint32_t k2 = p.tables.desc[p.known_opp[2 * (q * nknown + f) + 1] & 63u];
                    best = max(best, eval_player(st, bsum + k1 + k2, bfield | flush_bit(k1, bf.fsx) | flush_bit(k2, bf.fsx), bf.thr));
                }
            }
            const int nrivals = nopp + nknown;
            const bool win = active && (nrivals == 0 || hv > best), tie = active && nrivals > 0 && hv == best;
            wins += win; ties += tie;
            if (p.win_types && (win || tie)) {
                uint32_t ty = 0;
#pragma unroll
                for (int i = 1; i < 9; i++) ty += hv >= p.tables.type_start[i];
                wt_pack += 1ull << (7 * ty);
            }
        }
        wins = __reduce_add_sync(0xffffffffu, wins);
        ties = __reduce_add_sync(0xffffffffu, ties);
        if (lane == 0) {
            atomicAdd(&p.wins[q], (unsigned long long)wins);
            atomicAdd(&p.ties[q], (unsigned long long)ties);
        }
        if (p.passes) {
            // 64-bit warp sum in three 21-bit slices (a lane makes at most 64 * 10 * 65536 < 2^26 attempts per item)
            unsigned long long tot = 0;
#pragma unroll
            for (int sft = 0; sft < 63; sft += 21)
                tot += (unsigned long long)__reduce_add_sync(0xffffffffu, (uint32_t)(passes >> sft) & 0x1fffffu) << sft;
            if (lane == 0) atomicAdd(&p.passes[q], tot);
        }
        if (p.win_types) {
#pragma unroll
            for (int i = 0; i < 9; i++) {
                uint32_t c = __reduce_add_sync(0xffffffffu, (uint32_t)(wt_pack >> (7 * i)) & 127u);
                if (lane == 0 && c) atomicAdd(&p.win_types[9 * q + i], (unsigned long long)c);
            }
        }
    }
}

// =====================================================================================================================
// K2: rank ids of 7-card hands
// =====================================================================================================================
// Four consecutive hands per thread: their 28 bytes are seven aligned 32-bit words (a warp reads 896 contiguous bytes),
// all seven loads are issued before the first use, and the four rank ids leave as one 8-byte store.  HBM traffic is the
// algorithmic 9 B per hand.  Round 1's kernel was bound by the alu pipe (87 %) and by shared-memory wavefronts (28 per 32
// hands in 33 SM cycles): per card a byte extract, a gather from a 52-word descriptor table (about 3 wavefronts, random
// banks), an add into the key sum and three instructions to turn the suit into a counter increment
// (profiles/r02_ncu_rank7_before.txt).  Now the card table holds {descriptor, suit-counter increment} as 8-byte entries,
// replicated per lane ([64 cards][32 lanes], 16 KB): one conflict-free LDS.64 per card (2 wavefronts, the minimum for
// 256 B), no suit arithmetic, and the byte extract is one mask (alu) plus one multiply-high that shifts the id into the
// address and adds the lane's base (fma pipe, idle in this kernel).
__global__ void __launch_bounds__(kRank7Threads, 1) rank7_kernel(const DeviceTables tables, const uint8_t* __restrict__ cards,
                                                               long long n, uint16_t* __restrict__ out)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemAddr st = smem_addr(stage_tables(tables, smem + 128, bar));
    uint8_t* extra = smem + 128 + tables.value_bytes + tables.rowoff_bytes + tables.flush_bytes + kDescBytes;
    uint2* s_card = reinterpret_cast<uint2*>(extra);                  // [64][32] {descriptor, 1 << 4*suit}; ids 52..63 -> {0, 0}
    for (int i = threadIdx.x; i < 64 * 32; i += blockDim.x) {
        const int c = i >> 5;
        const uint32_t d = c < 52 ? tables.desc[c] : 0u;
        s_card[i] = make_uint2(d, c < 52 ? suit_inc(d) : 0u);
    }
    __syncthreads();
    const uint32_t lane_base = smem_u32(s_card) + 8u * (threadIdx.x & 31);
    // entry of the card in byte k of word w (id clamped to 64 slots: an id >= 52 is the caller's error, reported by
    // NPK_FLAG_VALIDATE, and ranks as garbage, never out of bounds): shared address = lane_base + id * 256
    auto card_entry = [&](uint32_t w, int k) {
        const uint32_t f = w & (0x3Fu << (8 * k));
        uint32_t addr;
        if (k == 0) addr = f * 256u + lane_base;
        else if (k == 1) addr = f + lane_base;
        else asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(f), "r"(1u << (32 - (8 * k - 8))), "r"(lane_base));
        uint2 e;
        asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "r"(addr));
        return e;
    };
    auto eval7 = [&](const uint2 (&e)[7]) {
        const uint32_t total = (e[0].x + e[1].x + e[2].x) + (e[3].x + e[4].x + e[5].x) + e[6].x;
        const uint32_t cnt = (0x3333u + e[0].y + e[1].y) + (e[2].y + e[3].y + e[4].y) + (e[5].y + e[6].y);
        uint32_t v = lookup_nonflush(st, total);
        const uint32_t f = cnt & 0x8888u;                 // nibble >= 8  <=>  that suit holds >= 5 cards
        if (f) {
            const uint32_t fsx = (((31u - __clz(f)) >> 2) & 3u) << 4;
            uint32_t field = 0;
#pragma unroll
            for (int i = 0; i < 7; i++) field |= shr_clamp(0x1000u, (e[i].x ^ fsx) & 63u);
            NPK_CHECK(st.check, 2u * field + 2u <= st.flush_bytes, 3);
            v = lds_u16(st.flush + 2u * field);           // a flush excludes full house / quads in 7 cards
        }
        return v;
    };
    const bool aligned = ((reinterpret_cast<uintptr_t>(cards) & 3u) == 0) && ((reinterpret_cast<uintptr_t>(out) & 7u) == 0);
    const long long quads = aligned ? n / 4 : 0;
    const uint32_t* __restrict__ words = reinterpret_cast<const uint32_t*>(cards);
    // software pipeline: the seven words of the NEXT quad are in flight while this one is evaluated (one CTA of 32 warps
    // per SM cannot hide HBM latency by occupancy alone)
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t nxt[7];
    if (g < quads) {
#pragma unroll
        for (int k = 0; k < 7; k++) nxt[k] = __ldg(words + 7 * g + k);
    }
    for (; g < quads; g += stride) {
        uint32_t w[7];
#pragma unroll
        for (int k = 0; k < 7; k++) w[k] = nxt[k];
        if (g + stride < quads) {
#pragma unroll
            for (int k = 0; k < 7; k++) nxt[k] = __ldg(words + 7 * (g + stride) + k);
        }
        uint32_t r[4];
#pragma unroll
        for (int h = 0; h < 4; h++) {
            uint2 e[7];
#pragma unroll
            for (int k = 0; k < 7; k++) {
                const int byte = 7 * h + k;
                e[k] = card_entry(w[byte >> 2], byte & 3);
            }
            r[h] = eval7(e);
        }
        uint2 packed;
        packed.x = r[0] | (r[1] << 16);
        packed.y = r[2] | (r[3] << 16);
        *reinterpret_cast<uint2*>(out + 4 * g) = packed;
    }
    for (long long i = 4 * quads + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint2 e[7];
#pragma unroll
        for (int k = 0; k < 7; k++) e[k] = card_entry(cards[7 * i + k], 0);
        out[i] = (uint16_t)eval7(e);
    }
}

// Hands enumerated in colexicographic order: c0 < c1 < ... < c6, index = sum_i C(c_i, i+1).  `first`..`first+count`.
__device__ __forceinline__ unsigned long long binom(int n, int k)
{
    if (k < 0 || k > n) return 0;
    unsigned long long r = 1;
    for (int i = 1; i <= k; i++) r = r * (unsigned long long)(n - k + i) / (unsigned long long)i;
    return r;
}

__global__ void __launch_bounds__(kAuxThreads, 1) rank7_colex_kernel(const DeviceTables tables, long long first,
                                                                     long long count, uint16_t* __restrict__ out)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemAddr st = smem_addr(stage_tables(tables, smem + 128, bar));
    uint32_t* s_desc = reinterpret_cast<uint32_t*>(smem + 128 + tables.value_bytes + tables.rowoff_bytes + tables.flush_bytes);
    if (threadIdx.x < 52) s_desc[threadIdx.x] = tables.desc[threadIdx.x];
    __syncthreads();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
        unsigned long long r = (unsigned long long)(first + i);
        uint32_t d[7];
        int hi = 51;
#pragma unroll
        for (int k = 7; k >= 1; k--) {
            int c = hi;
            while (binom(c, k) > r) c--;       // largest c with C(c,k) <= r
            r -= binom(c, k);
            d[k - 1] = s_desc[c];
            hi = c - 1;
        }
        out[i] = (uint16_t)eval7_desc(st, d);
    }
}

// =====================================================================================================================
// K3: exact heads-up enumeration.  One CTA per query: every completion of the board x every opponent pair among the
// unseen cards.  Also ordered pairs of disjoint opponent hands on a complete board (three players, river).
// Outputs win / tie / lose from the hero's point of view (hero > / == / < best opponent).
// =====================================================================================================================
// Fast paths (at most two board cards to come, one opponent): a warp takes one board completion, computes the board part
// and the hero's value once, and its lanes walk over the opponent pairs -- per matchup one 3-input add, the table
// gathers and the flush test, exactly the per-player work of the Monte-Carlo kernels.  The list of pairs (a < b) of
// unseen cards is built once per query in shared memory and doubles as the list of two-card completions.
__global__ void __launch_bounds__(kAuxThreads, 1) enum_kernel(const EnumParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemAddr st = smem_addr(stage_tables(p.tables, smem + 128, bar));
    uint8_t* extra = smem + 128 + p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes;
    uint32_t* s_deck = reinterpret_cast<uint32_t*>(extra);            // [52] descriptors of unseen cards, ascending id
    uint16_t* s_pairval = reinterpret_cast<uint16_t*>(extra + 256);   // [1326] rank of each opponent pair (3 players, river)
    uint16_t* s_pair = reinterpret_cast<uint16_t*>(extra + 256 + 2688);   // [1326] a | b << 8, a < b
    __shared__ unsigned long long s_acc[3];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;

    // The list of slot pairs (a < b), pair number C(b,2) + a, does not depend on the query: a deck of n cards uses its first
    // n(n-1)/2 entries.  Built once per CTA (round 1 rebuilt it for every query: one thread walked up to 46 entries alone,
    // which cost a river query -- 990 matchups, two per thread -- about as much as the matchups themselves).
    for (int i = threadIdx.x; i < 1326; i += blockDim.x) {
        int b = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)i)) * 0.5f);
        while (b * (b - 1) / 2 > i) b--;
        while ((b + 1) * b / 2 <= i) b++;
        s_pair[i] = (uint16_t)((i - b * (b - 1) / 2) | b << 8);
    }

    for (long long q = blockIdx.x; q < p.nq; q += gridDim.x) {
        int known = 0;
        for (int i = 0; i < 5; i++) known += p.board[5 * q + i] != 0xFF;
        const int nopp = (int)p.n_players[q] - 1;
        // ids are clamped to the 64-slot descriptor table: an id >= 52 is the caller's error (NPK_FLAG_VALIDATE reports
        // it) and gives a meaningless count, never an out-of-bounds access or an undefined shift
        const uint32_t h0 = p.hole[2 * q] & 63u, h1 = p.hole[2 * q + 1] & 63u;
        uint64_t knownmask = (1ull << h0) | (1ull << h1);
        const uint32_t hd[2] = {p.tables.desc[h0], p.tables.desc[h1]};
        uint32_t bd[5];
        for (int i = 0; i < known; i++) { const uint32_t c = p.board[5 * q + i] & 63u; bd[i] = p.tables.desc[c]; knownmask |= 1ull << c; }
        const uint64_t avail = ~knownmask & ((1ull << 52) - 1ull);
        const int n = __popcll(avail);
        const int npairs = n * (n - 1) / 2;
        __syncthreads();
        if (threadIdx.x < 3) s_acc[threadIdx.x] = 0;
        for (int c = threadIdx.x; c < 52; c += blockDim.x)
            if (avail >> c & 1ull) s_deck[__popcll(avail & ((1ull << c) - 1ull))] = p.tables.desc[c];
        __syncthreads();

        unsigned long long win = 0, tie = 0, lose = 0;
        const int missing = 5 - known;
        if (nopp == 1 && missing <= 2) {
            const int ncomp = missing == 0 ? 1 : (missing == 1 ? n : npairs);
            const int wpc = ncomp >= nwarps ? 1 : nwarps / ncomp;        // warps sharing one completion
            const int groups = nwarps / wpc;
            uint32_t ksum = 0, kcnt = 0x5555u, klo = 0, khi = 0;           // known board: sum, suit counters, suit-major masks
            for (int i = 0; i < known; i++) {
                uint32_t l, h;
                card_bits(bd[i], l, h);
                ksum += bd[i]; kcnt += suit_inc(bd[i]); klo |= l; khi |= h;
            }
            uint32_t hlo, hhi, l, h;
            card_bits(hd[0], hlo, hhi);
            card_bits(hd[1], l, h);
            hlo |= l; hhi |= h;
            if (warp < groups * wpc) {
                for (int ic = warp / wpc; ic < ncomp; ic += groups) {
                    int c0 = -1, c1 = -1;
                    if (missing == 1) c0 = ic;
                    else if (missing == 2) { const uint32_t pr = s_pair[ic]; c0 = pr & 255; c1 = pr >> 8; }
                    const uint32_t e0 = c0 >= 0 ? s_deck[c0] : 0u, e1 = c1 >= 0 ? s_deck[c1] : 0u;
                    uint32_t bsum = ksum + e0 + e1, bcnt = kcnt;
                    if (c0 >= 0) bcnt += suit_inc(e0);
                    if (c1 >= 0) bcnt += suit_inc(e1);
                    const BoardFlush bf = board_flush(bcnt);
                    uint32_t bfield = prmt(klo, khi, bf.sel);
                    if (c0 >= 0) bfield |= flush_bit(e0, bf.fsx);
                    if (c1 >= 0) bfield |= flush_bit(e1, bf.fsx);
                    const uint32_t hv = eval_player(st, bsum + hd[0] + hd[1], bfield | prmt(hlo, hhi, bf.sel), bf.thr);
                    for (int ip = (warp % wpc) * 32 + lane; ip < npairs; ip += 32 * wpc) {
                        const uint32_t pr = s_pair[ip];
                        const int a = pr & 255, b = pr >> 8;
                        if (a == c0 || a == c1 || b == c0 || b == c1) continue;
                        const uint32_t d0 = s_deck[a], d1 = s_deck[b];
                        const uint32_t ov = eval_player(st, bsum + d0 + d1, bfield | flush_bit(d0, bf.fsx) | flush_bit(d1, bf.fsx), bf.thr);
                        win += hv > ov; tie += hv == ov; lose += hv < ov;
                    }
                }
            }
        } else if (nopp == 1) {
            // three or more board cards to come: generic walk over (completion, pair) by colexicographic unranking
            long long ncomp = 1;
            for (int i = 0; i < missing; i++) ncomp = ncomp * (n - i) / (i + 1);
            const long long total = ncomp * npairs;
            for (long long w = threadIdx.x; w < total; w += blockDim.x) {
                const long long ic = w / npairs;
                const uint32_t pr = s_pair[(int)(w - ic * npairs)];
                const int a = pr & 255, b = pr >> 8;
                int comp[5];
                {
                    unsigned long long r = (unsigned long long)ic;
                    int hi = n - 1;
                    for (int k = missing; k >= 1; k--) {
                        int c = hi;
                        while (binom(c, k) > r) c--;
                        r -= binom(c, k);
                        comp[k - 1] = c;
                        hi = c - 1;
                    }
                }
                bool clash = false;
                for (int k = 0; k < missing; k++) clash |= (comp[k] == a) | (comp[k] == b);
                if (clash) continue;
                uint32_t h7[7], o7[7];
                h7[0] = hd[0]; h7[1] = hd[1]; o7[0] = s_deck[a]; o7[1] = s_deck[b];
                for (int k = 0; k < known; k++) { h7[2 + k] = bd[k]; o7[2 + k] = bd[k]; }
                for (int k = 0; k < missing; k++) { h7[2 + known + k] = s_deck[comp[k]]; o7[2 + known + k] = h7[2 + known + k]; }
                const uint32_t hv = eval7_desc(st, h7), ov = eval7_desc(st, o7);
                win += hv > ov; tie += hv == ov; lose += hv < ov;
            }
        } else if (nopp == 2 && known == 5) {
            uint32_t h7[7] = {hd[0], hd[1], bd[0], bd[1], bd[2], bd[3], bd[4]};
            const uint32_t hv = eval7_desc(st, h7);
            for (int ip = threadIdx.x; ip < npairs; ip += blockDim.x) {
                const uint32_t pr = s_pair[ip];
                uint32_t o7[7] = {s_deck[pr & 255], s_deck[pr >> 8], bd[0], bd[1], bd[2], bd[3], bd[4]};
                s_pairval[ip] = (uint16_t)eval7_desc(st, o7);
            }
            __syncthreads();
            // ordered pairs of disjoint opponent hands: warp-strided first hand, lane-strided second hand
            for (int i1 = warp; i1 < npairs; i1 += nwarps) {
                const uint32_t p1 = s_pair[i1];
                const int a1 = p1 & 255, b1 = p1 >> 8;
                const uint32_t v1 = s_pairval[i1];
                for (int i2 = lane; i2 < npairs; i2 += 32) {
                    const uint32_t p2 = s_pair[i2];
                    const int a2 = p2 & 255, b2 = p2 >> 8;
                    if (a1 == a2 || a1 == b2 || b1 == a2 || b1 == b2) continue;
                    const uint32_t best = max(v1, (uint32_t)s_pairval[i2]);
                    win += hv > best; tie += hv == best; lose += hv < best;
                }
            }
        }
        // block reduction: warp shuffles then one shared atomic per warp
        for (int o = 16; o > 0; o >>= 1) {
            win += __shfl_down_sync(0xffffffffu, win, o);
            tie += __shfl_down_sync(0xffffffffu, tie, o);
            lose += __shfl_down_sync(0xffffffffu, lose, o);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&s_acc[0], win); atomicAdd(&s_acc[1], tie); atomicAdd(&s_acc[2], lose);
        }
        __syncthreads();
        if (threadIdx.x == 0) { p.win[q] = s_acc[0]; p.tie[q] = s_acc[1]; p.lose[q] = s_acc[2]; }
    }
}

// =====================================================================================================================
// K4: batched get_winner (hand_evaluator.py:9-17): first index among the best hands + its hand type
// =====================================================================================================================
__global__ void __launch_bounds__(kAuxThreads, 1) showdown_kernel(const DeviceTables tables, const uint8_t* __restrict__ holes,
                                                                  const uint8_t* __restrict__ n_players,
                                                                  const uint8_t* __restrict__ board, long long n, int maxp,
                                                                  int32_t* __restrict__ winner, uint8_t* __restrict__ wtype,
                                                                  uint16_t* __restrict__ ranks)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemAddr st = smem_addr(stage_tables(tables, smem + 128, bar));
    uint32_t* s_desc = reinterpret_cast<uint32_t*>(smem + 128 + tables.value_bytes + tables.rowoff_bytes + tables.flush_bytes);
    if (threadIdx.x < 64) s_desc[threadIdx.x] = threadIdx.x < 52 ? tables.desc[threadIdx.x] : 0u;
    __syncthreads();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint32_t d[7];
#pragma unroll
        for (int k = 0; k < 5; k++) d[2 + k] = s_desc[board[5 * i + k] & 63u];
        int best = -1;
        uint32_t bv = 0;
        const int np = n_players[i];
        for (int pl = 0; pl < np; pl++) {
            d[0] = s_desc[holes[(i * maxp + pl) * 2] & 63u];
            d[1] = s_desc[holes[(i * maxp + pl) * 2 + 1] & 63u];
            const uint32_t v = eval7_desc(st, d);
            if (ranks) ranks[i * maxp + pl] = (uint16_t)v;
            if (best < 0 || v > bv) { best = pl; bv = v; }
        }
        winner[i] = best;
        uint32_t ty = 0;
#pragma unroll
        for (int k = 1; k < 9; k++) ty += bv >= tables.type_start[k];
        wtype[i] = (uint8_t)ty;
    }
}

// Philox words for known-answer tests: out[4*i..] = philox(c[4*i..], key)
__global__ void philox_debug_kernel(const uint32_t* __restrict__ ctr, uint32_t k0, uint32_t k1, int n, uint32_t* __restrict__ out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        uint32_t o[4];
        philox4x32_10(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], k0, k1, o);
        out[4 * i] = o[0]; out[4 * i + 1] = o[1]; out[4 * i + 2] = o[2]; out[4 * i + 3] = o[3];
    }
}

// Integer-issue microbenchmark (roofline denominator): 8 independent dependency chains per thread, 16x unrolled.
//   variant 0: LOP3 only (alu pipe)   variant 1: IMAD only (fma pipe)   variant 2: one IMAD + one LOP3 per chain step
// Instructions per thread per outer iteration: 128 (variants 0, 1) or 256 (variant 2), plus ~3 of loop overhead that
// is NOT counted -- so the reported rate slightly understates the true issue rate.
template <int V>
__global__ void __launch_bounds__(256) int_peak_kernel(uint32_t* out, int iters, uint32_t b, uint32_t c)
{
    uint32_t a[8];
#pragma unroll
    for (int j = 0; j < 8; j++) a[j] = threadIdx.x * 8u + j + blockIdx.x;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
#pragma unroll
            for (int j = 0; j < 8; j++) {
                if (V == 1 || V == 2) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(a[j]) : "r"(b), "r"(c));
                if (V == 0 || V == 2) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[j]) : "r"(b), "r"(c));
            }
        }
    }
    uint32_t x = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) x ^= a[j];
    out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

cudaError_t launch_int_peak(int variant, uint32_t* out, int iters, int grid, cudaStream_t s)
{
    switch (variant) {
        case 0: int_peak_kernel<0><<<grid, 256, 0, s>>>(out, iters, 0x9E3779B9u, 0x7F4A7C15u); break;
        case 1: int_peak_kernel<1><<<grid, 256, 0, s>>>(out, iters, 0x9E3779B9u, 0x7F4A7C15u); break;
        case 2: int_peak_kernel<2><<<grid, 256, 0, s>>>(out, iters, 0x9E3779B9u, 0x7F4A7C15u); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------------------------
// Shared memory decides the CTA shape: tables + one private deck per warp.  As many warps as fit (at most 16) run on
// each SM; the deck of N = 45..50 cards costs 128 B per card per warp.
static int uniform_warps(const DeviceTables& t, int nb)
{
    const size_t fixed = 128 + (size_t)t.value_bytes + t.rowoff_bytes + t.flush_bytes + kDescBytes;
    const size_t per_warp = (size_t)(64 + (45 + nb) * 32) * 4;
    int w = (int)((kMaxDynamicSmem - fixed) / per_warp);
    if (w > kEquityMaxThreads / 32) w = kEquityMaxThreads / 32;
    return w < 1 ? 1 : w;
}

constexpr int kMaxDevicesForAttr = 64;

template <int NOPP, int NB>
static cudaError_t launch_uniform_t(const EquityParams& p, long long items, int sm_count, cudaStream_t s)
{
    auto k = p.reference_dealer ? equity_refdeal_kernel<NOPP, NB> : equity_uniform_kernel<NOPP, NB>;
    const int warps = uniform_warps(p.tables, NB);
    const size_t smem = 128 + (size_t)p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes + kDescBytes +
                        (size_t)warps * (64 + (45 + NB) * 32) * 4;
    // the opt-in is per kernel and per device: ask the driver once, not on every launch of a 20 us call
    static std::atomic<size_t> opted[kMaxDevicesForAttr];          // zero-initialised; several host threads may launch
    int dev = 0;
    cudaGetDevice(&dev);
    cudaError_t e = cudaSuccess;
    if (dev < 0 || dev >= kMaxDevicesForAttr || opted[dev] != smem + 2 * (size_t)p.reference_dealer + 1) {
        e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < kMaxDevicesForAttr) opted[dev] = smem + 2 * (size_t)p.reference_dealer + 1;
    }
    long long grid = (items + warps - 1) / warps;
    if (grid < 1) grid = 1;
    if (grid > sm_count) grid = sm_count;
    k<<<(int)grid, warps * 32, smem, s>>>(p);
    return cudaGetLastError();
}

template <int NB>
static cudaError_t launch_uniform_nb(int nopp, const EquityParams& p, long long items, int sm_count, cudaStream_t s)
{
    switch (nopp) {
        case 0: return launch_uniform_t<0, NB>(p, items, sm_count, s);
        case 1: return launch_uniform_t<1, NB>(p, items, sm_count, s);
        case 2: return launch_uniform_t<2, NB>(p, items, sm_count, s);
        case 3: return launch_uniform_t<3, NB>(p, items, sm_count, s);
        case 4: return launch_uniform_t<4, NB>(p, items, sm_count, s);
        case 5: return launch_uniform_t<5, NB>(p, items, sm_count, s);
        case 6: return launch_uniform_t<6, NB>(p, items, sm_count, s);
        case 7: return launch_uniform_t<7, NB>(p, items, sm_count, s);
        case 8: return launch_uniform_t<8, NB>(p, items, sm_count, s);
        case 9: return launch_uniform_t<9, NB>(p, items, sm_count, s);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_equity_uniform(int nopp, int nb, const EquityParams& p, long long items, int sm_count, cudaStream_t s)
{
    switch (nb) {
        case 0: return launch_uniform_nb<0>(nopp, p, items, sm_count, s);
        case 1: return launch_uniform_nb<1>(nopp, p, items, sm_count, s);
        case 2: return launch_uniform_nb<2>(nopp, p, items, sm_count, s);
        case 3: return launch_uniform_nb<3>(nopp, p, items, sm_count, s);
        case 4: return launch_uniform_nb<4>(nopp, p, items, sm_count, s);
        case 5: return launch_uniform_nb<5>(nopp, p, items, sm_count, s);
        default: return cudaErrorInvalidValue;
    }
}

size_t aux_smem(const DeviceTables& t) { return 128 + t.value_bytes + t.rowoff_bytes + t.flush_bytes + 256 + 2 * 2688 + 64; }

cudaError_t launch_equity_ranges(int deal_mode, const EquityParams& p, int grid, cudaStream_t s)
{
    size_t smem = aux_smem(p.tables);
    auto k = !p.plan ? (deal_mode == 1 ? equity_ranges_kernel<1, 0> : equity_ranges_kernel<0, 0>)
                     : (deal_mode == 1 ? equity_ranges_kernel<1, 1> : equity_ranges_kernel<0, 1>);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<grid, kRefThreads, smem, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_rank7(const DeviceTables& t, const uint8_t* cards, long long n, uint16_t* out, int grid, cudaStream_t s)
{
    size_t smem = 128 + t.value_bytes + t.rowoff_bytes + t.flush_bytes + kDescBytes + 64 * 32 * 8;   // + the per-lane card table
    cudaError_t e = cudaFuncSetAttribute(rank7_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    rank7_kernel<<<grid, kRank7Threads, smem, s>>>(t, cards, n, out);
    return cudaGetLastError();
}

cudaError_t launch_rank7_colex(const DeviceTables& t, long long first, long long count, uint16_t* out, int grid, cudaStream_t s)
{
    size_t smem = aux_smem(t);
    cudaError_t e = cudaFuncSetAttribute(rank7_colex_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    rank7_colex_kernel<<<grid, kAuxThreads, smem, s>>>(t, first, count, out);
    return cudaGetLastError();
}

cudaError_t launch_enum(const EnumParams& p, int grid, cudaStream_t s)
{
    size_t smem = aux_smem(p.tables);
    cudaError_t e = cudaFuncSetAttribute(enum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    enum_kernel<<<grid, kAuxThreads, smem, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_showdown(const DeviceTables& t, const uint8_t* holes, const uint8_t* n_players, const uint8_t* board,
                            long long n, int maxp, int32_t* winner, uint8_t* wtype, uint16_t* ranks, int grid, cudaStream_t s)
{
    size_t smem = aux_smem(t);
    cudaError_t e = cudaFuncSetAttribute(showdown_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    showdown_kernel<<<grid, kAuxThreads, smem, s>>>(t, holes, n_players, board, n, maxp, winner, wtype, ranks);
    return cudaGetLastError();
}

cudaError_t launch_philox_debug(const uint32_t* ctr, uint32_t k0, uint32_t k1, int n, uint32_t* out, cudaStream_t s)
{
    philox_debug_kernel<<<(n + 127) / 128, 128, 0, s>>>(ctr, k0, k1, n, out);
    return cudaGetLastError();
}

}  // namespace npk
