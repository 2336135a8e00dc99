// npk_mixed.cu -- ONE persistent kernel for batches that mix player counts and board sizes (BASELINE config 5: the
// get_equity call of 65,536 self-play tables per step, gym_env/env.py:261-263).
//
// The queries have been sorted by shape on the device (classify kernels in npk_capi.cu): group g = opponents * 6 + known
// board cards holds counts[g] queries, listed in qindex from offsets[g].  Work items of all groups form one sequence --
// group after group -- and the
// warps of a persistent grid (one CTA per SM) pull from it through one global counter.  Per item a warp looks up its
// group and calls that shape's specialised item function (the same code the per-shape kernels inline), so
//   * the rank tables are staged once per CTA per call instead of once per shape,
//   * there is one tail per call instead of one per shape, and no SM partitioning to guess,
//   * the host needs no shape counts: no device->host read, the call is asynchronous and graph-capturable,
//   * neighbouring items belong to the same shape, so the warps of an SM run the same code most of the time.
// Round 1 launched one kernel per shape present (eleven per self-play step, side by side on SM shares sized on the host
// from a synchronous read of the counts): 1.15 ms of Monte-Carlo kernels per step for 65,536 tables.
#include "npk_mc.cuh"

namespace npk {

// Out-of-line so that the persistent kernel stays one dispatch loop plus 60 separately compiled bodies.  The kernel's
// parameter block reaches a body through a pointer (local memory); copying it into locals of the body lets the compiler keep
// the fields the trial loop reads (seed, offsets, counter pointers) in registers -- read through the pointer they were
// reloaded in every iteration (5 LDL + 2 LD per trial in the first version, profiles/r02_ncu_mixed_v1.txt), because the
// shared-memory asm statements of the dealer are memory clobbers.
template <int NOPP, int NB, int REF>
__device__ __noinline__ void shape_item(const EquityParams* p, const WarpCtx* cx, long long q, long long t_begin, long long t_end)
{
    const EquityParams lp = *p;
    const WarpCtx lcx = *cx;
    if (REF) refdeal_item<NOPP, NB>(lp, lcx, q, t_begin, t_end);
    else uniform_item<NOPP, NB>(lp, lcx, q, t_begin, t_end);
}

template <int NOPP, int REF>
__device__ __forceinline__ void dispatch_known(int known, const EquityParams* p, const WarpCtx* cx, long long q, long long b,
                                               long long e)
{
    switch (known) {
        case 0: shape_item<NOPP, 5, REF>(p, cx, q, b, e); break;
        case 1: shape_item<NOPP, 4, REF>(p, cx, q, b, e); break;
        case 2: shape_item<NOPP, 3, REF>(p, cx, q, b, e); break;
        case 3: shape_item<NOPP, 2, REF>(p, cx, q, b, e); break;
        case 4: shape_item<NOPP, 1, REF>(p, cx, q, b, e); break;
        default: shape_item<NOPP, 0, REF>(p, cx, q, b, e); break;
    }
}

// PLAN = 1: the rounds of an adaptive call, whose work items are planned on the device (p.plan = {chunk, chunks}).
template <int REF, int PLAN>
__global__ void __launch_bounds__(kMixedThreads, 1) equity_mixed_kernel(const EquityParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ long long s_first[kShapeGroups + 1];          // first item of every group in the concatenated sequence
    const WarpCtx cx = warp_context(p, smem, 64 + 50 * 32);  // decks sized for the largest shape (preflop: 50 unseen cards)
    const int lane = cx.lane;
    const uint32_t* counts = p.group;                        // [64] queries per group, [64..128) first qindex slot per group
    const uint32_t plan_chunk = PLAN ? p.plan[0] : 0u, plan_chunks = PLAN ? p.plan[1] : 0u;
    const long long per_query = PLAN ? (long long)plan_chunks : (long long)p.chunks;
    if (threadIdx.x == 0) {
        long long acc = 0;
        for (int g = 0; g < kShapeGroups; g++) { s_first[g] = acc; acc += (long long)counts[g] * per_query; }
        s_first[kShapeGroups] = acc;
    }
    __syncthreads();
    const long long n_items = s_first[kShapeGroups];
    for (long long item = next_item(p.work_counter, lane); item < n_items; item = next_item(p.work_counter, lane)) {
        // group of this item = number of groups that end at or before it (two groups per lane)
        uint32_t before = 0;
        if (lane < kShapeGroups) before += item >= s_first[lane + 1];
        if (lane + 32 < kShapeGroups) before += item >= s_first[lane + 33];
        const int g = (int)__reduce_add_sync(0xffffffffu, before);
        long long qslot, t_begin, t_end;
        if (PLAN) {
            const long long rel = item - s_first[g];
            qslot = rel / plan_chunks;
            t_begin = (rel - qslot * plan_chunks) * plan_chunk;
            t_end = min(p.trials, t_begin + (long long)plan_chunk);
        } else {
            item_range(p, item - s_first[g], qslot, t_begin, t_end);
        }
        const long long q = p.qindex[counts[64 + g] + qslot];
        const int known = g % 6;
        switch (g / 6) {
            case 0: dispatch_known<0, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 1: dispatch_known<1, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 2: dispatch_known<2, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 3: dispatch_known<3, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 4: dispatch_known<4, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 5: dispatch_known<5, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 6: dispatch_known<6, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 7: dispatch_known<7, REF>(known, &p, &cx, q, t_begin, t_end); break;
            case 8: dispatch_known<8, REF>(known, &p, &cx, q, t_begin, t_end); break;
            default: dispatch_known<9, REF>(known, &p, &cx, q, t_begin, t_end); break;
        }
    }
}

// =====================================================================================================================
// Resident one-query server (npk_resident_start; protocol in npk_kernels.h).  Same per-shape bodies as the mixed kernel, the
// tables staged ONCE for the lifetime of the kernel; per request: poll (PCIe) -> gen (L2) -> items by static striding ->
// one ticket per CTA -> 16-byte result store to the host.  What get_equity (tools/montecarlo_python.py:401-406) costs
// per call is then the work itself plus two PCIe crossings, not a kernel launch.
// =====================================================================================================================
__device__ __forceinline__ uint4 ld_volatile_v4(const void* p)
{
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_v4(void* p, uint4 v)
{
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <int REF>
__device__ __forceinline__ void dispatch_players(int players, int known, const EquityParams* p, const WarpCtx* cx, long long b,
                                                 long long e)
{
    switch (players - 1) {
        case 0: dispatch_known<0, REF>(known, p, cx, 0, b, e); break;
        case 1: dispatch_known<1, REF>(known, p, cx, 0, b, e); break;
        case 2: dispatch_known<2, REF>(known, p, cx, 0, b, e); break;
        case 3: dispatch_known<3, REF>(known, p, cx, 0, b, e); break;
        case 4: dispatch_known<4, REF>(known, p, cx, 0, b, e); break;
        case 5: dispatch_known<5, REF>(known, p, cx, 0, b, e); break;
        case 6: dispatch_known<6, REF>(known, p, cx, 0, b, e); break;
        case 7: dispatch_known<7, REF>(known, p, cx, 0, b, e); break;
        case 8: dispatch_known<8, REF>(known, p, cx, 0, b, e); break;
        default: dispatch_known<9, REF>(known, p, cx, 0, b, e); break;
    }
}

// One request on the warps of this grid: a = {-, trials, packed_lo, packed_hi}, b = {-, seed_lo, seed_hi, sequence number}.
// The CTA's counts go to s_cnt (shared), then ONE packed atomic per CTA on *acc; the CTA that completes the count publishes.
__device__ __forceinline__ void serve_request(EquityParams& p, const WarpCtx& cx, const uint4 a, const uint4 b,
                                              unsigned long long* s_cnt, unsigned long long* acc, ResidentMailbox* mb)
{
    const int warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const unsigned int total_warps = gridDim.x * warps;
    const unsigned int trials = a.y, hi = a.w;
    unsigned int chunk = trials / (8u * total_warps);
    chunk = (chunk + 63u) / 64u * 64u;
    chunk = chunk < 64u ? 64u : (chunk > 2048u ? 2048u : chunk);
    const unsigned int chunks = (trials + chunk - 1u) / chunk;
    const int players = (int)(hi >> 24 & 15u);
    const unsigned long long packed = (unsigned long long)a.z | (unsigned long long)(hi & 0xFFFFFFu) << 32;
    int known = 0;
#pragma unroll
    for (int i = 0; i < 5; i++) known += (packed >> (16 + 8 * i) & 0xFFull) != 0xFFull;
    p.hole = nullptr; p.inline_query = packed;
    p.trials = trials; p.trial_offset = 0; p.query_offset = 0;
    p.seed_lo = b.y; p.seed_hi = b.z;
    p.chunk = chunk; p.chunks = chunks;
    p.wins = &s_cnt[0]; p.ties = &s_cnt[1];              // generic pointers to shared memory: one RED.shared per warp and item
    // items spread over the CTAs first: a 10,000-trial call (157 items of 64 trials) puts one or two warps on every SM
    for (unsigned int item = warp * gridDim.x + blockIdx.x; item < chunks; item += total_warps) {
        const long long t_begin = (long long)item * chunk;
        const long long t_end = min((long long)trials, t_begin + (long long)chunk);
        if (hi >> 31) dispatch_players<1>(players, known, &p, &cx, t_begin, t_end);
        else dispatch_players<0>(players, known, &p, &cx, t_begin, t_end);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long mine = s_cnt[0] | s_cnt[1] << 28 | 1ull << 56;
        const unsigned long long old = atomicAdd(acc, mine);
        if ((old >> 56) == gridDim.x - 1u) {             // this CTA completes the count: old + mine are the totals
            const unsigned long long tot = old + mine;
            asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(&mb->done), "r"((unsigned int)(tot & 0xFFFFFFFu)),
                         "r"((unsigned int)(tot >> 28 & 0xFFFFFFFu)), "r"(b.w), "r"(0u)
                         : "memory");
        }
    }
}

__global__ void __launch_bounds__(kMixedThreads, 1)
equity_resident_kernel(const DeviceTables tables, ResidentState* st, ResidentMailbox* mb, const unsigned long long launch_id,
                       const unsigned int last_seq, const long long idle_cycles)
{
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint4 s_a, s_b;                               // the current command
    __shared__ unsigned long long s_cnt[2];                  // this CTA's wins, ties of the current request
    EquityParams p{};
    p.tables = tables;
    const WarpCtx cx = warp_context(p, smem, 64 + 50 * 32);
    unsigned int cmd = 0;                                    // commands seen so far (the state block is zeroed before the launch)
    unsigned int seq_seen = last_seq;
    long long t_last = clock64();
    for (;;) {
        if (threadIdx.x == 0) {
            uint4 a, b;
            if (blockIdx.x == 0) {
                // the poller: wait for a request with a new sequence number in both records, a stop request, or the idle limit
                bool leave = false;
                for (;;) {
                    a = ld_volatile_v4(&mb->a);
                    b = ld_volatile_v4(&mb->b);
                    if (a.x == b.x && a.x != seq_seen) break;
                    if (b.w == (unsigned int)launch_id || clock64() - t_last > idle_cycles) { leave = true; break; }
                }
                seq_seen = leave ? seq_seen : a.x;
                a.x = cmd + 1; b.w = leave ? 0u : b.x; b.x = cmd + 1;
                st_volatile_v4(&st->a, a);
                st_volatile_v4(&st->b, b);
            } else {
                do {
                    a = ld_volatile_v4(&st->a);
                    b = ld_volatile_v4(&st->b);
                } while (a.x != cmd + 1 || b.x != cmd + 1);
            }
            s_a = a; s_b = b;
            s_cnt[0] = 0; s_cnt[1] = 0;
        }
        __syncthreads();
        cmd++;
        const uint4 a = s_a, b = s_b;
        if (b.w == 0u) break;                                // leave
        serve_request(p, cx, a, b, s_cnt, &st->acc[cmd & 1], mb);
        if (threadIdx.x == 0) {
            if (blockIdx.x == 0) {
                // the accumulator of the NEXT command (idle since command cmd - 1) is cleared here, off the path of the request
                // just served and before the next one can be published (this thread is the one that publishes it)
                st->acc[(cmd + 1) & 1] = 0;
                __threadfence();
            }
            t_last = clock64();
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        __threadfence_system();
        *reinterpret_cast<volatile unsigned long long*>(&mb->exited) = launch_id;
    }
}

// The same request served by a kernel launched for it (the default one-query path, npk_equity_one without resident mode):
// the request travels in the kernel parameters, a few small CTAs (four warps each while the call has few items) stage the tables,
// and the hand-over is the packed atomic + 16-byte store of the resident server instead of per-warp counters, a ticket and a
// read-back.  `parity` alternates between calls; the other accumulator is cleared for the next call.
__global__ void __launch_bounds__(kMixedThreads, 1)
equity_oneshot_kernel(const DeviceTables tables, ResidentState* st, ResidentMailbox* mb, const uint4 a, const uint4 b,
                      const unsigned int parity)
{
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ unsigned long long s_cnt[2];
    EquityParams p{};
    p.tables = tables;
    if (threadIdx.x == 0) {
        s_cnt[0] = 0; s_cnt[1] = 0;
        if (blockIdx.x == 0) st->acc[parity ^ 1u] = 0;
    }
    const WarpCtx cx = warp_context(p, smem, 64 + 50 * 32);       // (synchronises the CTA while it stages the tables)
    serve_request(p, cx, a, b, s_cnt, &st->acc[parity], mb);
}

cudaError_t launch_equity_resident(const DeviceTables& t, ResidentState* st, ResidentMailbox* mb, unsigned long long launch_id,
                                   unsigned int last_seq, long long idle_cycles, int ctas, cudaStream_t s)
{
    const size_t fixed = 128 + (size_t)t.value_bytes + t.rowoff_bytes + t.flush_bytes + kDescBytes;
    const size_t smem = fixed + (size_t)(kMixedThreads / 32) * (64 + 50 * 32) * 4;
    cudaError_t e = cudaFuncSetAttribute(equity_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    equity_resident_kernel<<<ctas, kMixedThreads, smem, s>>>(t, st, mb, launch_id, last_seq, idle_cycles);
    return cudaGetLastError();
}

cudaError_t launch_equity_oneshot(const DeviceTables& t, ResidentState* st, ResidentMailbox* mb, uint4 a, uint4 b,
                                  unsigned int parity, int sm_count, cudaStream_t s)
{
    const long long items = ((long long)a.y + 63) / 64;
    const int warps = items <= 4ll * sm_count ? 4 : kMixedThreads / 32;
    long long grid = (items + warps - 1) / warps;
    if (grid < 1) grid = 1;
    if (grid > sm_count) grid = sm_count;
    if (grid > 255) grid = 255;                              // the CTA count of the packed accumulator has 8 bits
    const size_t fixed = 128 + (size_t)t.value_bytes + t.rowoff_bytes + t.flush_bytes + kDescBytes;
    const size_t smem_max = fixed + (size_t)(kMixedThreads / 32) * (64 + 50 * 32) * 4;
    const size_t smem = fixed + (size_t)warps * (64 + 50 * 32) * 4;
    static bool opted[64];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !opted[dev]) {
        cudaError_t e = cudaFuncSetAttribute(equity_oneshot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) opted[dev] = true;
    }
    equity_oneshot_kernel<<<(int)grid, warps * 32, smem, s>>>(t, st, mb, a, b, parity);
    return cudaGetLastError();
}

cudaError_t launch_equity_mixed(const EquityParams& p, int sm_count, cudaStream_t s)
{
    auto k = p.plan ? (p.reference_dealer ? equity_mixed_kernel<1, 1> : equity_mixed_kernel<0, 1>)
                    : (p.reference_dealer ? equity_mixed_kernel<1, 0> : equity_mixed_kernel<0, 0>);
    const size_t fixed = 128 + (size_t)p.tables.value_bytes + p.tables.rowoff_bytes + p.tables.flush_bytes + kDescBytes;
    const size_t smem = fixed + (size_t)(kMixedThreads / 32) * (64 + 50 * 32) * 4;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<sm_count, kMixedThreads, smem, s>>>(p);
    return cudaGetLastError();
}

}  // namespace npk
