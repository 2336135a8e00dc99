// npk_enum_plan.cuh -- the work split shared by the batched exact enumerations (npk_showdown_equity.cu, npk_exact_equity.cu).
//
// The enumerated units of all spots of a batch form one global sequence: an exclusive prefix of the per-spot counts sits in a
// caller-owned workspace, a work item is a fixed-size range of that sequence, and the persistent enumeration kernel pulls items
// from the work counter.  One large spot therefore spreads over every SM while one item can carry many small spots.
#pragma once
#include <stdint.h>

namespace npk {

constexpr int kPlanThreads = 1024;
// workspace: [0,8) work counter | [8,12) units per item | [64, 64 + 8 (N+1)) exclusive prefix of the units
constexpr int kPlanWsCounter = 0, kPlanWsItem = 8, kPlanWsPrefix = 64;

__host__ __device__ inline long long plan_workspace_bytes(long long n) { return kPlanWsPrefix + 8 * ((n > 0 ? n : 0) + 1); }

__device__ __forceinline__ unsigned long long plan_binom(int n, int k)
{
    if (k < 0 || n < k) return 0;
    unsigned long long r = 1;
    for (int i = 1; i <= k; i++) r = r * (unsigned long long)(n - k + i) / (unsigned long long)i;
    return r;
}

// One CTA of kPlanThreads: exclusive prefix of counts[0, n) (four spots per thread and pass), then the item size -- the total
// over `parts`, rounded up to a multiple of `align`, within [lo, hi] -- and the work counter reset.
__device__ __forceinline__ void plan_items(const unsigned long long* counts, long long n, uint8_t* ws, unsigned long long parts,
                                           unsigned long long align, unsigned long long lo, unsigned long long hi)
{
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    unsigned long long* prefix = reinterpret_cast<unsigned long long*>(ws + kPlanWsPrefix);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (long long base = 0; base < n; base += 4 * kPlanThreads) {
        unsigned long long v[4], sum = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const long long i = base + 4 * threadIdx.x + k;
            v[k] = i < n ? counts[i] : 0ull;
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
            if (i < n) prefix[i] = excl;
            excl += v[k];
        }
        __syncthreads();
        if (threadIdx.x == 0) s_carry += s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const unsigned long long total = s_carry;
        prefix[n] = total;
        unsigned long long item = total / parts;
        item = (item + align - 1) / align * align;
        item = item < lo ? lo : (item > hi ? hi : item);
        *reinterpret_cast<uint32_t*>(ws + kPlanWsItem) = (uint32_t)item;
        *reinterpret_cast<unsigned long long*>(ws + kPlanWsCounter) = 0ull;
    }
}

}  // namespace npk
