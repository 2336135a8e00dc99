// npk_showdown_equity.cu -- K5: exact showdown equity of known hands.
//
// Every hand of a spot is known, so the only unknown is the rest of the board: every m-subset (m = 5 - known board cards) of
// the unseen cards U' is enumerated once and scored for every player (win / tie / split-pot share, include/npk.h).  U' = the
// 52 cards minus hands, board and dead cards, in ascending id order; the reference's dealer never deals the last card of its
// id-ordered list (montecarlo_python.py:185-189), so in REFERENCE mode the highest unseen id is simply left out of U'.
//
// Completions are numbered in colexicographic order over the slots of U' (c0 < c1 < ... < c(m-1), rank = sum C(c_i, i+1)).
// Those sharing the top m-2 cards form one contiguous block whose pairs (c0, c1) are the prefix [0, C(c2, 2)) of the pair list
// numbered C(b, 2) + a (the list of enum_kernel): a warp fixes the top cards, sums their descriptors, suit counters and rank
// masks once, and its lanes walk the pairs of the block -- no unranking and no clash test per completion.
//
// Work split: the completions of all spots of a batch form one global sequence (an exclusive prefix of the per-spot counts in the
// workspace); a work item is a fixed-size range of that sequence, so one heads-up preflop spot spreads over every SM while a
// single item carries several small spots.  Three kernels, all on the caller's stream and without a host round trip:
//   se_prepare_kernel   per spot: completions, zeroed outputs
//   se_plan_kernel      one CTA: prefix of the completions, item size, work counter reset
//   showdown_equity_kernel  persistent, one CTA per SM: tables staged once per CTA, warps pull items from the work counter
#include <algorithm>
#include "npk_mc.cuh"

namespace npk {

constexpr int kSeThreads = 512;
constexpr int kSeWarps = kSeThreads / 32;
constexpr int kSePlanThreads = 1024;
// completions per work item: a lane scores at most one item's worth per spot, so its win and tie counts stay below 2^16 and
// share below 2^32 (32,768 * 2,520)
constexpr uint32_t kSeMaxItem = 32768, kSeMinItem = 512;
// workspace: [0,8) work counter | [8,12) completions per item | [64, 64 + 8 (N+1)) exclusive prefix of the completions
constexpr int kSeWsCounter = 0, kSeWsItem = 8, kSeWsPrefix = 64;
// dynamic shared memory behind the tables: descriptors [64] | pair list [1326] u16 | C(c, k) [6][64] u32 | warp decks [16][64]
constexpr uint32_t kSePairOff = kDescBytes, kSeBinomOff = kSePairOff + 2688, kSeDeckOff = kSeBinomOff + 6 * 64 * 4,
                   kSeExtraBytes = kSeDeckOff + kSeWarps * 64 * 4;

long long showdown_equity_workspace_bytes(long long n) { return kSeWsPrefix + 8 * ((n > 0 ? n : 0) + 1); }

struct SpotShape {
    uint64_t avail;    // unseen cards U, one bit per id
    int n;             // |U'|
    int missing;       // board cards to come
    int players;       // 0 when n_players is outside 1..maxp
};

// Ids are clamped to the 64-slot descriptor table and the dead mask to 52 bits: any bytes give a memory-safe spot.
__device__ __forceinline__ SpotShape spot_shape(const ShowdownEquityParams& p, long long s)
{
    SpotShape sh;
    const int np = p.n_players[s];
    sh.players = np >= 1 && np <= p.maxp ? np : 0;
    uint64_t known = p.dead ? p.dead[s] : 0ull;
    for (int i = 0; i < 2 * sh.players; i++) known |= 1ull << (p.holes[2 * p.maxp * s + i] & 63u);
    int nb = 0;
    for (int i = 0; i < 5; i++) {
        const uint32_t c = p.board[5 * s + i];
        if (c != 0xFFu) { known |= 1ull << (c & 63u); nb++; }
    }
    sh.avail = ~known & ((1ull << 52) - 1ull);
    sh.missing = 5 - nb;
    sh.n = __popcll(sh.avail) - (p.reference && sh.missing > 0 ? 1 : 0);
    return sh;
}

__device__ __forceinline__ unsigned long long se_binom(int n, int k)
{
    if (k < 0 || n < k) return 0;
    unsigned long long r = 1;
    for (int i = 1; i <= k; i++) r = r * (unsigned long long)(n - k + i) / (unsigned long long)i;
    return r;
}

__global__ void __launch_bounds__(256) se_prepare_kernel(const ShowdownEquityParams p)
{
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < p.n; s += (long long)gridDim.x * blockDim.x) {
        const SpotShape sh = spot_shape(p, s);
        p.completions[s] = sh.players && sh.n >= sh.missing ? se_binom(sh.n, sh.missing) : 0ull;
        for (int q = 0; q < p.maxp; q++) {
            p.win[s * p.maxp + q] = 0; p.tie[s * p.maxp + q] = 0; p.share[s * p.maxp + q] = 0;
        }
    }
}

// One CTA: exclusive prefix of the completions (four spots per thread and pass), then the item size -- about four items per
// warp of the grid, within [kSeMinItem, kSeMaxItem] -- and the work counter for the enumeration kernel.
__global__ void __launch_bounds__(kSePlanThreads) se_plan_kernel(const ShowdownEquityParams p)
{
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    unsigned long long* prefix = reinterpret_cast<unsigned long long*>(p.workspace + kSeWsPrefix);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (long long base = 0; base < p.n; base += 4 * kSePlanThreads) {
        unsigned long long v[4], sum = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const long long i = base + 4 * threadIdx.x + k;
            v[k] = i < p.n ? p.completions[i] : 0ull;
            sum += v[k];
        }
        unsigned long long incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        unsigned long long excl = s_carry + (warp ? s_warp[warp - 1] : 0ull) + incl - sum;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const long long i = base + 4 * threadIdx.x + k;
            if (i < p.n) prefix[i] = excl;
            excl += v[k];
        }
        __syncthreads();
        if (threadIdx.x == 0) s_carry += s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const unsigned long long total = s_carry;
        prefix[p.n] = total;
        unsigned long long item = total / (4ull * (unsigned long long)p.sm_count * kSeWarps);
        item = (item + 31) / 32 * 32;
        item = item < kSeMinItem ? kSeMinItem : (item > kSeMaxItem ? kSeMaxItem : item);
        *reinterpret_cast<uint32_t*>(p.workspace + kSeWsItem) = (uint32_t)item;
        *reinterpret_cast<unsigned long long*>(p.workspace + kSeWsCounter) = 0ull;
    }
}

// One completion scored for P players: `bsum` / `bfield` / `bf` describe the complete board.  wt packs win (bits 0..15) and
// tie (bits 16..31) counts; sh collects the split-pot shares of ties only (a win's 2520 is added at the reduction).
template <int P>
__device__ __forceinline__ void se_score(const SmemAddr& st, uint32_t bsum, uint32_t bfield, const BoardFlush& bf,
                                         const uint32_t (&hs)[P], const uint32_t (&hl)[P], const uint32_t (&hh)[P],
                                         uint32_t (&wt)[P], uint32_t (&sh)[P])
{
    uint32_t v[P], best = 0, k = 0;
#pragma unroll
    for (int q = 0; q < P; q++) {
        v[q] = eval_player(st, bsum + hs[q], bfield | prmt(hl[q], hh[q], bf.sel), bf.thr);
        best = max(best, v[q]);
    }
#pragma unroll
    for (int q = 0; q < P; q++) {
        const uint32_t eq = v[q] == best;
        wt[q] += eq;
        k += eq;
    }
    if (k > 1) {
        const uint32_t part = 2520u / k;
#pragma unroll
        for (int q = 0; q < P; q++)
            if (v[q] == best) { wt[q] += 0xFFFFu; sh[q] += part; }
    }
}

struct SeSmem {
    const uint32_t* desc;      // [64], ids 52..63 -> 0
    const uint16_t* pair;      // [1326] a | b << 8, number C(b,2) + a
    const uint32_t* binom;     // [k * 64 + c] = C(c, k), k = 0..5
    uint32_t* deck;            // this warp's [52] descriptors of U, ascending id
};

// Completions r0..r1-1 (colex ranks) of spot s, P players, on one warp; adds the counts into the outputs.
template <int P>
__device__ __forceinline__ void se_segment(const ShowdownEquityParams& p, const SmemAddr& st, const SeSmem& sm, const SpotShape& sh,
                                        long long s, uint32_t r0, uint32_t r1, int lane)
{
    const uint32_t* deck = sm.deck;
    uint32_t hs[P], hl[P], hh[P], wt[P], shr[P];
#pragma unroll
    for (int q = 0; q < P; q++) {
        const uint32_t d0 = sm.desc[p.holes[2 * (p.maxp * s + q)] & 63u], d1 = sm.desc[p.holes[2 * (p.maxp * s + q) + 1] & 63u];
        uint32_t l, h;
        hs[q] = d0 + d1;
        card_bits(d0, hl[q], hh[q]);
        card_bits(d1, l, h);
        hl[q] |= l; hh[q] |= h;
        wt[q] = 0; shr[q] = 0;
    }
    uint32_t ksum = 0, kcnt = 0x5555u, klo = 0, khi = 0;     // known board; counters biased by 5 (>= 8 <=> >= 3 cards)
    for (int i = 0; i < 5; i++) {
        const uint32_t c = p.board[5 * s + i];
        if (c == 0xFFu) continue;
        const uint32_t d = sm.desc[c & 63u];
        uint32_t l, h;
        card_bits(d, l, h);
        ksum += d; kcnt += suit_inc(d); klo |= l; khi |= h;
    }
    const int n = sh.n, missing = sh.missing;

    if (missing >= 2) {
        const int t = missing - 2;                             // top cards c2.. held fixed by the warp
        int top[3] = {0, 0, 0};
        uint32_t r = r0;
#pragma unroll
        for (int i = 2; i >= 0; i--) {
            if (i < t) {
                int c = n - 1;
                while (sm.binom[(i + 3) * 64 + c] > r) c--;
                top[i] = c;
                r -= sm.binom[(i + 3) * 64 + c];
            }
        }
        uint32_t pos = r0, first = r;                          // first pair of the current block
        while (pos < r1) {
            const uint32_t lim = sm.binom[2 * 64 + (t > 0 ? top[0] : n)];
            const uint32_t len = min(lim - first, r1 - pos);
            uint32_t tsum = ksum, tcnt = kcnt, tlo = klo, thi = khi;
#pragma unroll
            for (int i = 0; i < 3; i++) {
                if (i < t) {
                    NPK_CHECK(p.tables.check, top[i] >= 0 && top[i] < n, 10);
                    const uint32_t d = deck[top[i]];
                    uint32_t l, h;
                    card_bits(d, l, h);
                    tsum += d; tcnt += suit_inc(d); tlo |= l; thi |= h;
                }
            }
            for (uint32_t ip = first + lane; ip < first + len; ip += 32) {
                NPK_CHECK(p.tables.check, ip < 1326u, 10);
                const uint32_t pr = sm.pair[ip];
                const uint32_t a = pr & 255u, b = pr >> 8;
                NPK_CHECK(p.tables.check, a < b && (int)b < n, 10);
                const uint32_t d0 = deck[a], d1 = deck[b];
                const BoardFlush bf = board_flush(tcnt + suit_inc(d0) + suit_inc(d1));
                const uint32_t bfield = prmt(tlo, thi, bf.sel) | flush_bit(d0, bf.fsx) | flush_bit(d1, bf.fsx);
                se_score<P>(st, tsum + d0 + d1, bfield, bf, hs, hl, hh, wt, shr);
            }
            pos += len;
            first = 0;
            if (pos < r1) {                                    // next top in colex order
                bool moved = false;
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    if (j < t && !moved) {
                        const int ub = j + 1 < t ? top[j + 1 < 3 ? j + 1 : 2] : n;
                        if (top[j] + 1 < ub) { top[j]++; moved = true; }
                        else top[j] = j + 2;
                    }
                }
            }
        }
    } else {
        for (uint32_t r = r0 + lane; r < r1; r += 32) {
            uint32_t bsum = ksum, bcnt = kcnt, blo = klo, bhi = khi;
            if (missing == 1) {
                NPK_CHECK(p.tables.check, (int)r < n, 10);
                const uint32_t d = deck[r];
                uint32_t l, h;
                card_bits(d, l, h);
                bsum += d; bcnt += suit_inc(d); blo |= l; bhi |= h;
            }
            const BoardFlush bf = board_flush(bcnt);
            se_score<P>(st, bsum, prmt(blo, bhi, bf.sel), bf, hs, hl, hh, wt, shr);
        }
    }

    uint32_t mw = 0, mt = 0, ms = 0;
#pragma unroll
    for (int q = 0; q < P; q++) {
        const uint32_t w = __reduce_add_sync(0xffffffffu, wt[q] & 0xFFFFu);
        const uint32_t ti = __reduce_add_sync(0xffffffffu, wt[q] >> 16);
        const uint32_t x = __reduce_add_sync(0xffffffffu, shr[q]);
        if (lane == q) { mw = w; mt = ti; ms = x; }
    }
    if (lane < P) {
        const long long o = s * p.maxp + lane;
        if (mw) atomicAdd(&p.win[o], (unsigned long long)mw);
        if (mt) atomicAdd(&p.tie[o], (unsigned long long)mt);
        if (mw || ms) atomicAdd(&p.share[o], 2520ull * mw + ms);
    }
}

__global__ void __launch_bounds__(kSeThreads, 1) showdown_equity_kernel(const ShowdownEquityParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const SmemAddr st = smem_addr(stage_tables(p.tables, smem + 128, bar));
    uint8_t* extra = smem + 128 + p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes;
    uint32_t* s_desc = reinterpret_cast<uint32_t*>(extra);
    uint16_t* s_pair = reinterpret_cast<uint16_t*>(extra + kSePairOff);
    uint32_t* s_binom = reinterpret_cast<uint32_t*>(extra + kSeBinomOff);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 64) s_desc[threadIdx.x] = threadIdx.x < 52 ? p.tables.desc[threadIdx.x] : 0u;
    for (int i = threadIdx.x; i < 1326; i += blockDim.x) {
        int b = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)i)) * 0.5f);
        while (b * (b - 1) / 2 > i) b--;
        while ((b + 1) * b / 2 <= i) b++;
        s_pair[i] = (uint16_t)((i - b * (b - 1) / 2) | b << 8);
    }
    for (int i = threadIdx.x; i < 6 * 64; i += blockDim.x) s_binom[i] = (uint32_t)se_binom(i & 63, i >> 6);
    __syncthreads();
    SeSmem sm;
    sm.desc = s_desc; sm.pair = s_pair; sm.binom = s_binom;
    sm.deck = reinterpret_cast<uint32_t*>(extra + kSeDeckOff) + 64 * warp;

    const unsigned long long* prefix = reinterpret_cast<const unsigned long long*>(p.workspace + kSeWsPrefix);
    unsigned long long* counter = reinterpret_cast<unsigned long long*>(p.workspace + kSeWsCounter);
    const unsigned long long total = prefix[p.n];
    const unsigned long long item_size = *reinterpret_cast<const uint32_t*>(p.workspace + kSeWsItem);
    const long long n_items = (long long)((total + item_size - 1) / item_size);
    for (long long item = next_item(counter, lane); item < n_items; item = next_item(counter, lane)) {
        unsigned long long g0 = (unsigned long long)item * item_size;
        const unsigned long long g1 = min(total, g0 + item_size);
        // the spot holding completion g0: the last s with prefix[s] <= g0, by a 32-way search
        long long s = 0, hi = p.n;
        while (hi - s > 1) {
            const long long step = (hi - s + 31) / 32, idx = s + (long long)(lane + 1) * step;
            const unsigned int le = __ballot_sync(0xffffffffu, idx < hi && prefix[idx] <= g0);
            s += (long long)__popc(le) * step;
            hi = min(hi, s + step);
        }
        for (; g0 < g1; s++) {
            const unsigned long long a = prefix[s], b = prefix[s + 1];
            if (b <= g0) continue;                             // a spot without completions
            const unsigned long long e = min(g1, b);
            const SpotShape sh = spot_shape(p, s);
            __syncwarp();
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int c = lane + 32 * h;
                if (c < 52 && (sh.avail >> c & 1ull)) sm.deck[__popcll(sh.avail & ((1ull << c) - 1ull))] = s_desc[c];
            }
            __syncwarp();
            const uint32_t r0 = (uint32_t)(g0 - a), r1 = (uint32_t)(e - a);
            switch (sh.players) {
                case 1: se_segment<1>(p, st, sm, sh, s, r0, r1, lane); break;
                case 2: se_segment<2>(p, st, sm, sh, s, r0, r1, lane); break;
                case 3: se_segment<3>(p, st, sm, sh, s, r0, r1, lane); break;
                case 4: se_segment<4>(p, st, sm, sh, s, r0, r1, lane); break;
                case 5: se_segment<5>(p, st, sm, sh, s, r0, r1, lane); break;
                case 6: se_segment<6>(p, st, sm, sh, s, r0, r1, lane); break;
                case 7: se_segment<7>(p, st, sm, sh, s, r0, r1, lane); break;
                case 8: se_segment<8>(p, st, sm, sh, s, r0, r1, lane); break;
                case 9: se_segment<9>(p, st, sm, sh, s, r0, r1, lane); break;
                case 10: se_segment<10>(p, st, sm, sh, s, r0, r1, lane); break;
                default: break;
            }
            g0 = e;
        }
    }
}

cudaError_t launch_showdown_equity(const ShowdownEquityParams& p, cudaStream_t s)
{
    const int prep_grid = (int)std::min<long long>((p.n + 255) / 256, 8ll * p.sm_count);
    se_prepare_kernel<<<prep_grid, 256, 0, s>>>(p);
    se_plan_kernel<<<1, kSePlanThreads, 0, s>>>(p);
    const size_t smem = 128 + (size_t)p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes + kSeExtraBytes;
    cudaError_t e = cudaFuncSetAttribute(showdown_equity_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    showdown_equity_kernel<<<p.sm_count, kSeThreads, smem, s>>>(p);
    return cudaGetLastError();
}

}  // namespace npk
