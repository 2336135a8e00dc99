// npk_ranges.cu -- K1''-fast: dealing with opponent / hero ranges without the reference's attempt loop over the whole deck.
//
// Reference (tools/montecarlo_python.py:136-148, :165-181): on the ordered list R of the n unseen cards draw i1 in [0,n),
// i2 in [0,n-1) and retry while i1 == i2 or the starting-hand class of (R[i1], R[i2]) -- both read BEFORE anything is popped
// (:173-174) -- is outside the range; a hero keeps exactly those two cards (:146-148), an opponent receives R.pop(i1) and then
// R.pop(i2) from the SHORTENED list (:178-179).  The generic kernel (equity_ranges_kernel in npk_kernels.cu) plays that loop
// literally: a top-30 % range rejects 70 % of the attempts, every lane of a warp loops a different number of times (lane
// efficiency 8.8 / 32, profiles/r02_ncu_ranges_before.txt) and every attempt costs two rank-selects on the 52-bit mask.
//
// The accepted (i1, i2) are uniform over  A = { i1 != i2, i2 <= n-2, class(R[i1], R[i2]) allowed }.  In card terms (card ids
// are order-isomorphic to list positions): ordered pairs (sa, sb) of distinct unseen cards with an allowed class and
// sb != max(R).  The class of a pair does not depend on the order, so per work item a warp lists the unordered allowed pairs
// of the query's INITIAL deck once (at most C(52,2) = 1,326 entries of 16 bits); a draw picks a uniform list entry and a
// uniform orientation, and is redone only when one of the two cards has been dealt earlier in this trial or sb is the last
// card of R -- a few per cent to 40 % instead of 70 %, and a redo costs one list read and two mask tests.  Every element of A
// is hit by exactly one (entry, orientation) that passes, so the accepted pair has the reference's distribution; the cards
// dealt from it follow the reference's pops: c1 = sa, c2 = sb if sb < sa, else the successor of sb in R (pop(i1) shifted the
// list).  UNIFORM mode (two distinct uniform cards, redrawn until the class is allowed): the same without the max(R) rule and
// without the successor.  Board cards: index j in [0, n-1) (REFERENCE, :188) or [0, n) of the ordered remaining list.
// `passes` (the reference's attempt counter) is not produced here: callers who ask for it get the generic kernel.
//
// Random numbers: Philox4x32-10, counter (trial, query, 0xA0000000 + block) in REFERENCE mode / 0xE0000000 in UNIFORM mode, one
// word per draw attempt (entry = hi32(w * len), orientation = bit 31 of the low product word) and per board card.
#include "npk_mc.cuh"

namespace npk {

constexpr int kPairs = 1326;                  // C(52,2): pair number of cards a < b is b*(b-1)/2 + a
constexpr int kPairWords = (kPairs + 31) / 32;

__device__ __forceinline__ bool class_bit(const uint32_t (&mask)[6], int c1, int c2)
{
    const int r1 = c1 >> 2, r2 = c2 >> 2, hi = max(r1, r2), lo = min(r1, r2);
    const int k = ((c1 ^ c2) & 3) == 0 ? hi * 13 + lo : lo * 13 + hi;
    return (mask[k >> 5] >> (k & 31)) & 1u;
}

// the warp's list of allowed pairs among the cards of `avail`: entries a | b << 8 (a < b), ascending pair number
__device__ __forceinline__ uint32_t build_list(const uint16_t* s_pair, const uint32_t* s_allowed, uint64_t avail, uint16_t* list,
                                               int lane)
{
    uint32_t n = 0;
    for (int w = 0; w < kPairWords; w++) {
        const int idx = 32 * w + lane;
        bool keep = false;
        uint32_t pr = 0;
        if (idx < kPairs && (s_allowed[w] >> lane & 1u)) {
            pr = s_pair[idx];
            keep = (avail >> (pr & 255u) & 1ull) && (avail >> (pr >> 8) & 1ull);
        }
        const uint32_t votes = __ballot_sync(0xffffffffu, keep);
        if (keep) list[n + __popc(votes & ((1u << lane) - 1u))] = (uint16_t)pr;
        n += __popc(votes);
    }
    __syncwarp();
    return n;
}

// PLAN = 1: a round of an adaptive call (npk_equity_ranges_batch_adaptive), whose items are planned on the device.
template <int MODE, int PLAN>
__global__ void __launch_bounds__(kRefThreads, 1) equity_ranges_fast_kernel(const EquityParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemTables stab = stage_tables(p.tables, smem + 128, bar);
    const SmemAddr st = smem_addr(stab);
    uint8_t* extra = smem + 128 + p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes + kDescBytes;
    uint16_t* s_pair = reinterpret_cast<uint16_t*>(extra);                         // [1326] a | b << 8
    uint32_t* s_allow_opp = reinterpret_cast<uint32_t*>(extra + 2688);            // [42] pair number -> class in the range
    uint32_t* s_allow_hero = s_allow_opp + 48;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint16_t* opp_list = reinterpret_cast<uint16_t*>(extra + 2688 + 384) + warp * (2 * 1344);
    uint16_t* hero_list = opp_list + 1344;

    // per CTA, once: the pair table and which pairs each range allows (independent of the query)
    for (int b = 1 + (int)threadIdx.x; b < 52; b += blockDim.x)
        for (int a = 0; a < b; a++) s_pair[b * (b - 1) / 2 + a] = (uint16_t)(a | b << 8);
    __syncthreads();
    for (int w = threadIdx.x; w < kPairWords; w += blockDim.x) {
        uint32_t mo = 0, mh = 0;
        for (int i = 0; i < 32 && 32 * w + i < kPairs; i++) {
            const uint32_t pr = s_pair[32 * w + i];
            if (class_bit(p.opp_mask, pr & 255u, pr >> 8)) mo |= 1u << i;
            if (p.hero_range && class_bit(p.hero_mask, pr & 255u, pr >> 8)) mh |= 1u << i;
        }
        s_allow_opp[w] = mo;
        s_allow_hero[w] = mh;
    }
    __syncthreads();

    const long long n_items = range_items<PLAN>(p);
    for (long long item = next_item(p.work_counter, lane); item < n_items; item = next_item(p.work_counter, lane)) {
        long long q, t_begin, t_end;
        range_item<PLAN>(p, item, q, t_begin, t_end);
        int known = 0;
        for (int i = 0; i < 5; i++) known += p.board[5 * q + i] != 0xFF;
        const int nknown = (int)p.n_known;                    // opponents whose cards are known (montecarlo_python.py:132-163)
        const int nopp = max(0, (int)p.n_players[q] - 1 - nknown);

        uint64_t taken = 0;
        uint32_t board_sum = 0, board_lo = 0, board_hi = 0, board_cnt = 0x5555u;
        for (int i = 0; i < known; i++) {
            const uint32_t c = p.board[5 * q + i] & 63u;
            const uint32_t d = stab.desc[c];
            uint32_t l, h;
            card_bits(d, l, h);
            board_sum += d; board_lo |= l; board_hi |= h; board_cnt += suit_inc(d);
            taken |= 1ull << c;
        }
        if (p.ghost)
            for (int i = 0; i < 2; i++) { const uint8_t c = p.ghost[2 * q + i]; if (c < 52) taken |= 1ull << c; }
        uint32_t h0 = 0, h1 = 0;
        if (!p.hero_range) { h0 = p.hole[2 * q] & 63u; h1 = p.hole[2 * q + 1] & 63u; taken |= (1ull << h0) | (1ull << h1); }
        for (int f = 0; f < 2 * nknown; f++) taken |= 1ull << (p.known_opp[2 * q * nknown + f] & 63u);
        const uint64_t avail0 = ~taken & ((1ull << 52) - 1ull);
        const int n0 = __popcll(avail0);

        __syncwarp();
        const uint32_t n_opp_list = nopp > 0 ? build_list(s_pair, s_allow_opp, avail0, opp_list, lane) : 0u;
        const uint32_t n_hero_list = p.hero_range ? build_list(s_pair, s_allow_hero, avail0, hero_list, lane) : 0u;
        if ((nopp > 0 && n_opp_list == 0) || (p.hero_range && n_hero_list == 0)) {
            if (lane == 0) atomicExch(p.abort_flag, 1u);           // no hand of the range is left in this query's deck
            continue;
        }

        uint32_t wins = 0, ties = 0;
        unsigned long long wt_pack = 0;
        for (long long tb = t_begin; tb < t_end; tb += 32) {
            if (*reinterpret_cast<volatile uint32_t*>(p.abort_flag)) break;
            const long long t_local = tb + lane;
            bool active = t_local < t_end;
            const unsigned long long trial = (unsigned long long)(p.trial_offset + t_local);
            WordStream rs;
            rs.c0 = (uint32_t)trial; rs.c1 = (uint32_t)(trial >> 32); rs.c2 = (uint32_t)q + p.query_offset;
            rs.k0 = p.seed_lo; rs.k1 = p.seed_hi; rs.blk = MODE == 1 ? 0xA0000000u : 0xE0000000u; rs.have = 0;

            uint64_t avail = avail0;
            int n = n0;
            uint32_t best = 0;
            uint32_t oc1[9], oc2[9];
            // one hand from a pair list (see the header): returns false when the attempt limit is hit
            auto draw = [&](const uint16_t* list, uint32_t len, bool is_hero, uint32_t& c1, uint32_t& c2) {
                for (uint32_t tries = 0; tries < kMaxRangeAttempts; tries++) {
                    const uint64_t prod = (uint64_t)rs.next() * len;
                    NPK_CHECK(st.check, (uint32_t)(prod >> 32) < len && len <= 1344u, 9);
                    const uint32_t pr = list[(uint32_t)(prod >> 32)];
                    uint32_t sa = pr & 255u, sb = pr >> 8;
                    NPK_CHECK(st.check, sa < 52u && sb < 52u && sa != sb, 9);
                    if ((uint32_t)prod >> 31) { const uint32_t t = sa; sa = sb; sb = t; }
                    if (!((avail >> sa) & (avail >> sb) & 1ull)) continue;             // one of them was dealt earlier in this trial
                    if (MODE == 1 && sb == 63u - (uint32_t)__clzll((long long)avail)) continue;   // i2 never reaches the last element
                    c1 = sa;
                    c2 = sb;
                    if (MODE == 1 && !is_hero && sb > sa)                              // pop(i1) shifted the list: successor of sb
                        c2 = sb + (uint32_t)__ffsll((long long)(avail >> (sb + 1u)));
                    avail &= ~((1ull << c1) | (1ull << c2));
                    n -= 2;
                    return true;
                }
                atomicExch(p.abort_flag, 1u);
                return false;
            };
            if (active && p.hero_range) active = draw(hero_list, n_hero_list, true, h0, h1);
            // the opponents, unrolled over the nine seats so that their cards stay in registers
#pragma unroll
            for (int o = 0; o < 9; o++) {
                if (o < nopp && active) {
                    uint32_t c1 = 0, c2 = 0;
                    active = draw(opp_list, n_opp_list, false, c1, c2);
                    oc1[o] = stab.desc[c1]; oc2[o] = stab.desc[c2];
                }
            }
            const uint32_t hd0 = stab.desc[h0], hd1 = stab.desc[h1];
            uint32_t bsum = board_sum, bcnt = board_cnt;
            uint32_t bd[5] = {0, 0, 0, 0, 0};
#pragma unroll
            for (int k = 0; k < 5; k++) {
                if (k >= known && active) {
                    const uint32_t j = __umulhi(rs.next(), (uint32_t)(MODE == 1 ? n - 1 : n));
                    const int c = select_bit(avail, (int)j);
                    avail &= ~(1ull << c);
                    n--;
                    const uint32_t d = stab.desc[c];
                    bd[k] = d;
                    bsum += d; bcnt += suit_inc(d);
                }
            }
            const BoardFlush bf = board_flush(bcnt);
            uint32_t bfield = prmt(board_lo, board_hi, bf.sel);
#pragma unroll
            for (int k = 0; k < 5; k++)
                if (k >= known && active) bfield |= flush_bit(bd[k], bf.fsx);
            const uint32_t hv = eval_player(st, bsum + hd0 + hd1, bfield | flush_bit(hd0, bf.fsx) | flush_bit(hd1, bf.fsx), bf.thr);
#pragma unroll
            for (int o = 0; o < 9; o++)
                if (o < nopp && active)
                    best = max(best, eval_player(st, bsum + oc1[o] + oc2[o],
                                                 bfield | flush_bit(oc1[o], bf.fsx) | flush_bit(oc2[o], bf.fsx), bf.thr));
            for (int f = 0; f < nknown && active; f++) {
                const uint32_t k1 = stab.desc[p.known_opp[2 * (q * nknown + f)] & 63u];
                const uint32_t k2 = stab.desc[p.known_opp[2 * (q * nknown + f) + 1] & 63u];
                best = max(best, eval_player(st, bsum + k1 + k2, bfield | flush_bit(k1, bf.fsx) | flush_bit(k2, bf.fsx), bf.thr));
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
        if (p.win_types) {
#pragma unroll
            for (int i = 0; i < 9; i++) {
                uint32_t c = __reduce_add_sync(0xffffffffu, (uint32_t)(wt_pack >> (7 * i)) & 127u);
                if (lane == 0 && c) atomicAdd(&p.win_types[9 * q + i], (unsigned long long)c);
            }
        }
    }
}

cudaError_t launch_equity_ranges_fast(int deal_mode, const EquityParams& p, int grid, cudaStream_t s)
{
    const size_t smem = 128 + (size_t)p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes + kDescBytes + 2688 + 384 +
                        (size_t)(kRefThreads / 32) * 2 * 1344 * 2;
    auto k = p.plan ? (deal_mode == 1 ? equity_ranges_fast_kernel<1, 1> : equity_ranges_fast_kernel<0, 1>)
                    : (deal_mode == 1 ? equity_ranges_fast_kernel<1, 0> : equity_ranges_fast_kernel<0, 0>);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<grid, kRefThreads, smem, s>>>(p);
    return cudaGetLastError();
}

}  // namespace npk
