// npk_device.cuh -- device-side building blocks shared by the sm_100a kernels in npk_kernels.cu.
//
// Data layout (all of it produced on the host by npk_tables.cpp / npk_capi.cu and resident in HBM after npk_init):
//   g_value   u16[n_value]   rank ids, row-displaced:  value[row_offset[mk >> 10] + (mk & 1023)]
//   g_rowoff  u16[8192]      one offset per row of the mixed key mk (23 bits)
//   g_flush   u16[8192]      rank id by 13-bit rank mask of the flush suit
//   g_desc    u32[52]        per-card descriptor  d = (mixkey[rank] << 9) | (16*suit + 12 - rank)
// Summing the descriptors of 7 cards with ordinary 32-bit wrap-around adds gives  total = (mk << 9) | psum  where
// mk = sum of mixed rank keys mod 2^23 identifies the rank histogram and psum < 512 never carries into mk.
// The three tables (about 129 KB) are copied once per CTA into shared memory with the bulk-copy engine (TMA 1-D).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace npk {

constexpr int kDevDescShift = 9;   // descriptor: bits 9..31 mixed rank key, bits 4..5 suit, bits 0..3 = 12 - rank
constexpr int kRowBits = 10;       // column bits of the mixed key   (== npk_tables.h kDescShift / kRowShift,
constexpr uint32_t kColMask = (1u << kRowBits) - 1u;   //              checked by a static_assert in npk_capi.cu)

struct DeviceTables {
    const uint16_t* value;
    const uint16_t* rowoff;
    const uint16_t* flush;
    const uint32_t* desc;          // [52]
    uint32_t value_bytes;          // padded to 16
    uint32_t rowoff_bytes;
    uint32_t flush_bytes;
    uint16_t type_start[10];
    uint32_t* check;               // one device word: highest code of a failed NPK_CHECK (checked builds), else untouched
};

struct SmemTables {
    const uint16_t* value;
    const uint16_t* rowoff;
    const uint16_t* flush;
    const uint32_t* desc;          // [52] (+ padding to kDescBytes)
    uint32_t value_bytes, rowoff_bytes, flush_bytes;
    uint32_t* check;
};

// ---- checked build (-DNPK_CHECKED, tools/checked_build.sh) ------------------------------------------------------------------
// compute-sanitizer is not available on the GPU pool this was developed on, so the library carries its own bounds checks:
// every shared-memory gather of the evaluator, every deck slot of the dealers and every decoded Lehmer slot is checked
// against its bounds, and the shuffled deck is compared with the canonical one after every work item (a racing or missing
// restore shows up there).  A failed check records its code in DeviceTables::check (npk_checked_status reads it).
// Codes: 1 rowoff gather, 2 value gather, 3 flush gather, 4 Fisher-Yates slot, 5 Lehmer slot, 6 duplicate Lehmer slot,
//        7 deck not restored, 8 descriptor index, 9 pair list of the range sampler (entry index, card ids),
//        10 unseen-card slot or pair index of the showdown-equity enumeration,
//        11 query slot of a device-planned range round, or the query id read from its qindex.
#ifdef NPK_CHECKED
#define NPK_CHECK(ptr, cond, code) do { if (!(cond)) atomicMax((ptr), (unsigned)(code)); } while (0)
#else
#define NPK_CHECK(ptr, cond, code) do { } while (0)
#endif

constexpr uint32_t kDescBytes = 256;   // the 52 card descriptors follow the flush table in the device blob, padded

// What a valid equity query is, on the host and on the device: card ids < 52, no card twice, the board's empty slots (0xFF)
// only at its end, and 1..10 players.  `hole` may be null (a hero drawn from a range).  Returns the number of known board
// cards, or -1; `mask` (if given) receives the cards seen, one bit per id.
__host__ __device__ __forceinline__ int validate_query(const uint8_t* hole, const uint8_t* board, int players,
                                                       unsigned long long* mask = nullptr)
{
    unsigned long long m = 0;
    int known = 0;
    bool bad = players < 1 || players > 10, ended = false;
    for (int i = 0; hole && i < 2; i++) {
        const int c = hole[i];
        if (c >= 52) bad = true; else { bad |= (m >> c & 1ull) != 0; m |= 1ull << c; }
    }
    for (int i = 0; i < 5; i++) {
        const int c = board[i];
        if (c == 0xFF) { ended = true; continue; }
        if (ended || c >= 52) { bad = true; continue; }
        bad |= (m >> c & 1ull) != 0;
        m |= 1ull << c;
        known++;
    }
    if (mask) *mask = m;
    return bad ? -1 : known;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier + 1-D bulk copy (cp.async.bulk -> UBLKCP) -------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}

// Stage the three lookup tables into shared memory.  Called by every thread of the CTA; returns shared pointers.
// `base` must be 16-byte aligned; uses value_bytes + rowoff_bytes + flush_bytes + kDescBytes bytes; `bar` is one 8-byte slot.
__device__ __forceinline__ SmemTables stage_tables(const DeviceTables& t, uint8_t* base, uint64_t* bar)
{
    uint8_t* s_value = base;
    uint8_t* s_rowoff = s_value + t.value_bytes;
    uint8_t* s_flush = s_rowoff + t.rowoff_bytes;
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, t.value_bytes + t.rowoff_bytes + t.flush_bytes + kDescBytes);
        const uint32_t kChunk = 32768;
        for (uint32_t o = 0; o < t.value_bytes; o += kChunk)
            bulk_g2s(s_value + o, (const uint8_t*)t.value + o, min(kChunk, t.value_bytes - o), bar);
        bulk_g2s(s_rowoff, t.rowoff, t.rowoff_bytes, bar);
        bulk_g2s(s_flush, t.flush, t.flush_bytes, bar);
        bulk_g2s(s_flush + t.flush_bytes, t.desc, kDescBytes, bar);
    }
    mbar_wait(bar, 0);
    SmemTables s;
    s.value = (const uint16_t*)s_value;
    s.rowoff = (const uint16_t*)s_rowoff;
    s.flush = (const uint16_t*)s_flush;
    s.desc = (const uint32_t*)(s_flush + t.flush_bytes);
    s.value_bytes = t.value_bytes; s.rowoff_bytes = t.rowoff_bytes; s.flush_bytes = t.flush_bytes; s.check = t.check;
    return s;
}

// ---- Philox4x32-10 (Salmon et al., SC'11): counter (c0,c1,c2,c3), key (k0,k1) -> 4 x 32 random bits -----------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4])
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
        k0 += W0;
        k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

// ---- evaluator -----------------------------------------------------------------------------------------------------
// PTX shr / shl clamp shift amounts above 31 to 32 (result 0), unlike the C++ operators whose behaviour is undefined.
__device__ __forceinline__ uint32_t shr_clamp(uint32_t v, uint32_t n)
{
    uint32_t r;
    asm("shr.u32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
    return r;
}

// 16-bit gather from shared memory by 32-bit shared address, zero-extended into a full register (keeps ptxas from
// switching to packed 16x2 arithmetic and the PRMT traffic that comes with it)
__device__ __forceinline__ uint32_t lds_u16(uint32_t saddr)
{
    uint32_t v;
    asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}

struct SmemAddr {          // 32-bit shared-window addresses of the staged tables
    uint32_t value, rowoff, flush;
#ifdef NPK_CHECKED
    uint32_t value_bytes, rowoff_bytes, flush_bytes;
    uint32_t* check;
#endif
};

__device__ __forceinline__ SmemAddr smem_addr(const SmemTables& s)
{
    SmemAddr a;
    a.value = smem_u32(s.value); a.rowoff = smem_u32(s.rowoff); a.flush = smem_u32(s.flush);
#ifdef NPK_CHECKED
    a.value_bytes = s.value_bytes; a.rowoff_bytes = s.rowoff_bytes; a.flush_bytes = s.flush_bytes; a.check = s.check;
#endif
    return a;
}

// rank id of a hand WITHOUT a flush from the wrapped sum of its 7 card descriptors.
// The two constant right shifts are written as multiply-high so they issue on the (otherwise idle) fma pipe.
__device__ __forceinline__ uint32_t lookup_nonflush(const SmemAddr& a, uint32_t total)
{
    const uint32_t row2 = __umulhi(total, 1u << (32 - (kDevDescShift + kRowBits - 1))) & (0xFFFFu << 1);   // 2*row
    NPK_CHECK(a.check, row2 + 2u <= a.rowoff_bytes, 1);
    const uint32_t off = lds_u16(a.rowoff + row2);
    const uint32_t col2 = __umulhi(total, 1u << (32 - (kDevDescShift - 1))) & (kColMask << 1);              // 2*col
    NPK_CHECK(a.check, col2 + (off << 1) + 2u <= a.value_bytes, 2);
    return lds_u16(a.value + col2 + (off << 1));
}

// contribution of a card to the 13-bit rank mask of suit fs (fsx = fs << 4): 1 << rank if the suit matches, else 0
__device__ __forceinline__ uint32_t flush_bit(uint32_t d, uint32_t fsx) { return shr_clamp(0x1000u, (d ^ fsx) & 63u); }

// 64-bit suit-major one-hot of a card descriptor: bit 16*suit + rank
__device__ __forceinline__ void card_bits(uint32_t d, uint32_t& lo, uint32_t& hi)
{
    const uint64_t b = 1ull << ((d & 0x30u) + 12u - (d & 15u));
    lo = (uint32_t)b;
    hi = (uint32_t)(b >> 32);
}

// nibble-per-suit counter increment of a card descriptor: 1 << 4*suit
__device__ __forceinline__ uint32_t suit_inc(uint32_t d) { return 1u << ((d >> 2) & 12u); }

// PRMT selector that extracts the 16-bit field of suit fs from a (lo, hi) suit-major pair and zeroes the upper half
// (selector nibble 8|k replicates the sign bit of byte k, which is always 0 here: ranks use bits 0..12 of a field)
__device__ __forceinline__ uint32_t field_selector(uint32_t fs) { return 0x9910u + fs * 0x2222u; }

// Plain 7-card evaluation from card descriptors (rank7 / showdown / enumeration kernels; the Monte-Carlo loops carry the
// board part across players instead).  Per card: one add into the key sum and one into the nibble-per-suit counters;
// the flush suit's rank mask is only assembled for the few hands that hold five cards of a suit.
__device__ __forceinline__ uint32_t eval7_desc(const SmemAddr& a, const uint32_t d[7])
{
    uint32_t total = 0, cnt = 0x3333u;
#pragma unroll
    for (int i = 0; i < 7; i++) {
        total += d[i];
        cnt += suit_inc(d[i]);
    }
    uint32_t v = lookup_nonflush(a, total);
    const uint32_t f = cnt & 0x8888u;                 // nibble >= 8  <=>  that suit holds >= 5 cards
    if (f) {
        const uint32_t fsx = (((31u - __clz(f)) >> 2) & 3u) << 4;
        uint32_t field = 0;
#pragma unroll
        for (int i = 0; i < 7; i++) field |= shr_clamp(0x1000u, (d[i] ^ fsx) & 63u);
        NPK_CHECK(a.check, 2u * field + 2u <= a.flush_bytes, 3);
        v = lds_u16(a.flush + 2u * field);            // a flush excludes full house / quads in 7 cards
    }
    return v;
}

}  // namespace npk
