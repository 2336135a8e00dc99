// npk_capi.cu -- the C ABI declared in include/npk.h: table upload, query classification, kernel launches.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/npk.h"
#include "../../include/npk_holdem.h"
#include "npk_holdem_launch.h"
#include "npk_kernels.h"
#include "npk_tables.h"

static_assert(npk::kDevDescShift == npk::kDescShift && npk::kRowBits == npk::kRowShift,
              "device and host table geometry differ");

namespace {

thread_local std::string g_err;
std::mutex g_mu;

struct DeviceState {
    bool ready = false;
    int sm_count = 0;
    int clock_khz = 0;
    npk::DeviceTables t{};
    void* blob = nullptr;
};

npk::Tables g_tables;
bool g_tables_ready = false;
constexpr int kMaxDevices = 64;
DeviceState g_dev[kMaxDevices];

// One resident server per device and process: a second one could not get the SMs the first one holds and its requests would
// starve.  Owner = address of the owning thread's staging block, 0 = none.
std::atomic<uintptr_t> g_resident_owner[kMaxDevices];

// One batch in flight through the host entry points: its own pinned staging, device buffers, workspace, stream and "done"
// event, so that the copies and the host-side work of batch i+1 overlap the kernel of batch i (npk_equity_host_submit / _wait).
struct HostSlot {
    int64_t cap_q = 0;
    uint8_t* h_in = nullptr;      // pinned: hole[2Q] board[5Q] players[Q]
    uint64_t* h_out = nullptr;    // pinned: wins[Q] ties[Q] types[9Q] passes[Q]
    uint8_t* d_in = nullptr;
    uint64_t* d_out = nullptr;
    void* d_ws = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    int64_t ticket = -1;          // -1: free
    int64_t Q = 0;
    uint32_t want = 0;            // bit 0: win types, bit 1: passes
    void free_buffers()
    {
        cudaFreeHost(h_in); cudaFreeHost(h_out); cudaFree(d_in); cudaFree(d_out); cudaFree(d_ws);
        h_in = nullptr; h_out = nullptr; d_in = nullptr; d_out = nullptr; d_ws = nullptr; cap_q = 0;
    }
};
constexpr int kHostSlots = NPK_HOST_SLOTS;

// host-staging state of the host entry points: one per CALLING THREAD (its own streams, pinned buffers and one-query scratch),
// so they are re-entrant -- two host threads never share a stream, a counter or a result block
struct HostStage {
    int device = -1;
    HostSlot slot[kHostSlots];
    int64_t next_ticket = 0;
    cudaStream_t stream = nullptr;       // the one-query path
    // one-query blocking calls (Q == 1): counters in device memory, results in mapped host memory
    npk::SingleCall* single = nullptr;
    npk::SingleResult* single_host = nullptr;
    unsigned long long single_seq = 0;
    // resident mode of the one-query path (npk_resident_start): a persistent kernel serves this thread's calls from a mailbox
    bool res_enabled = false, res_running = false;
    int res_ctas = 0;
    long long res_idle_cycles = 0;
    npk::ResidentMailbox* res_mb = nullptr;       // mapped host memory
    npk::ResidentMailbox* res_mb_dev = nullptr;   // the same block as the device sees it
    npk::ResidentState* res_state = nullptr;      // device memory
    unsigned long long res_launch_id = 0;
    unsigned int res_seq = 0;
    unsigned int oneshot_parity = 0;              // accumulator the next launched one-query call uses
    bool res_dirty = false;                       // a server has used the state block since the last launched call
    void stop_resident();
    void release_resident_slot();
    void release()
    {
        if (device < 0) return;
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess) { device = -1; return; }     // runtime already torn down
        cudaSetDevice(device);
        stop_resident();
        release_resident_slot();
        cudaFree(res_state); cudaFreeHost(res_mb);
        for (HostSlot& s : slot) {
            if (s.stream) cudaStreamSynchronize(s.stream);
            s.free_buffers();
            if (s.done) cudaEventDestroy(s.done);
            if (s.stream) cudaStreamDestroy(s.stream);
        }
        cudaFree(single); cudaFreeHost(single_host);
        if (stream) cudaStreamDestroy(stream);
        if (cur >= 0) cudaSetDevice(cur);
        *this = HostStage{};
    }
    ~HostStage() { release(); }
};
thread_local HostStage t_stage;

// Ask this thread's resident server to leave and wait until it has (it polls the mailbox every couple of microseconds).
void HostStage::stop_resident()
{
    if (!res_running || !res_mb) { res_running = false; return; }
    volatile npk::ResidentMailbox* mb = res_mb;
    mb->b.stop = (unsigned int)res_launch_id;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    for (long spins = 0; spins < 20000000 && mb->exited != res_launch_id; spins++) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    cudaStreamSynchronize(stream);            // the kernel itself has ended (bounded by its idle limit in any case)
    res_running = false;
}

// give the device's resident slot back if this thread holds it (the thread stops serving its calls through a server)
void HostStage::release_resident_slot()
{
    if (device >= 0 && device < kMaxDevices) {
        uintptr_t mine = reinterpret_cast<uintptr_t>(this);
        g_resident_owner[device].compare_exchange_strong(mine, 0);
    }
}

int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}

int cuda_fail(cudaError_t e, const char* what)
{
    return fail(NPK_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

// Copy one u32 of device memory to `out` once the work enqueued on `s` before it has finished.
int read_word(const void* src, cudaStream_t s, uint32_t* out, const char* what)
{
    cudaError_t e = cudaMemcpyAsync(out, src, 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, what);
}

// The causes of an invalid query of the batched calls, as their NPK_ERR_INVALID_CARDS messages list them.
constexpr const char* kQueryCauses = "card id >= 52, duplicate cards, gap in the board, or players outside 1..10";
constexpr const char* kRangeQueryCauses = "card id >= 52, duplicate cards, gap in the board, ghost card on the board or in a "
                                          "hand, more known opponents than opponents, or players outside 1..10";

std::string invalid_queries(uint32_t n, const char* causes, const char* tail = "")
{
    return std::to_string(n) + " invalid quer" + (n == 1 ? "y" : "ies") + " (" + causes + ")" + tail;
}

int ensure_host_tables()
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_tables_ready) return NPK_OK;
    const char* err = npk::build_tables(g_tables);
    if (err && err[0]) return fail(NPK_ERR_TABLES, std::string("table construction failed: ") + err);
    g_tables_ready = true;
    return NPK_OK;
}

int current_state(DeviceState** out)
{
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
    if (dev < 0 || dev >= kMaxDevices || !g_dev[dev].ready)
        return fail(NPK_ERR_NOT_INITIALIZED, "npk_init(device) has not been called for the current CUDA device");
    *out = &g_dev[dev];
    return NPK_OK;
}

// ---- query classification (mixed player counts / board sizes) --------------------------------------------------------
// workspace layout (bytes): [0,512) 64 work counters u64 | [512,768) 64 group counts u32 | [768,1024) 64 group offsets u32
//                           (exclusive prefix of the counts; a kernel reads its group as {count = group[0], offset =
//                           group[64]}) | [1024,1028) invalid-query count | [1028,1092) abort flag + diagnostics
//                           | [1092,1096) queries of shapes outside the caller's shape mask | [1096,1100) blocks done
//                           | [1280,1536) 64 fill cursors u32 | [2048, 2048+4Q) qindex
constexpr int kWsCounters = 0, kWsCounts = 512, kWsOffsets = 768, kWsInvalid = 1024, kWsAbort = 1028, kWsSkipped = 1092,
              kWsBlocksDone = 1096, kWsCursors = 1280, kWsIndex = 2048;
constexpr int kGroups = npk::kShapeGroups;   // group = nopp * 6 + known, nopp 0..9, known 0..5

__device__ __forceinline__ int classify_query(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players,
                                              long long q)
{
    const int np = n_players[q];
    const int known = npk::validate_query(hole + 2 * q, board + 5 * q, np);
    return known < 0 ? -1 : (np - 1) * 6 + known;
}

// Count the queries of every shape -- per block in shared memory, then one global atomic per shape and block (65,536
// self-play queries fall into a dozen shapes: per-query global atomics on a dozen addresses took 35 us) -- and let the last
// block to finish drop the shapes outside `shape_mask` and write the exclusive prefix of the counts behind them.
// `active` [Q] or null: queries with active[q] == 0 (retired by an adaptive call) are left out altogether.
__global__ void __launch_bounds__(256) classify_count_kernel(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players,
                                                             long long Q, uint8_t* ws, unsigned long long shape_mask,
                                                             const uint8_t* active)
{
    __shared__ uint32_t s_cnt[65];                         // [64] = invalid
    __shared__ bool last;
    uint32_t* counts = reinterpret_cast<uint32_t*>(ws + kWsCounts);
    if (threadIdx.x < 65) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < Q; q += (long long)gridDim.x * blockDim.x) {
        if (active && !active[q]) continue;
        const int g = classify_query(hole, board, n_players, q);
        atomicAdd(&s_cnt[g < 0 ? 64 : g], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 64 && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], s_cnt[threadIdx.x]);
    if (threadIdx.x == 64 && s_cnt[64]) atomicAdd(reinterpret_cast<uint32_t*>(ws + kWsInvalid), s_cnt[64]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(reinterpret_cast<uint32_t*>(ws + kWsBlocksDone), 1u) == gridDim.x - 1;
    __syncthreads();
    if (last && threadIdx.x == 0) {
        __threadfence();
        uint32_t* offsets = reinterpret_cast<uint32_t*>(ws + kWsOffsets);
        uint32_t acc = 0, skipped = 0;
        for (int g = 0; g < 64; g++) {
            uint32_t c = *reinterpret_cast<volatile uint32_t*>(&counts[g]);
            if (!(shape_mask >> g & 1ull)) { skipped += c; c = 0; counts[g] = 0; }
            offsets[g] = acc;
            acc += c;
        }
        *reinterpret_cast<uint32_t*>(ws + kWsSkipped) = skipped;
    }
}

// Sort the query numbers by shape: a block counts its own queries per shape, reserves one range per shape in qindex with a
// single global atomic, and its threads take slots inside the range from shared-memory cursors.
__global__ void __launch_bounds__(256) classify_fill_kernel(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players,
                                                            long long Q, uint8_t* ws, const uint8_t* active)
{
    __shared__ uint32_t s_cnt[64], s_base[64];
    uint32_t* cursors = reinterpret_cast<uint32_t*>(ws + kWsCursors);
    const uint32_t* counts = reinterpret_cast<const uint32_t*>(ws + kWsCounts);
    const uint32_t* offsets = reinterpret_cast<const uint32_t*>(ws + kWsOffsets);
    int32_t* qindex = reinterpret_cast<int32_t*>(ws + kWsIndex);
    // every block handles ONE contiguous span of queries, each thread at most kPerThread of them (held in registers
    // between the counting and the placing pass)
    constexpr int kPerThread = 8;
    const long long per_block = (Q + gridDim.x - 1) / gridDim.x;
    const long long q0 = (long long)blockIdx.x * per_block, q1 = min(Q, q0 + per_block);
    for (long long base = q0; base < q1; base += (long long)blockDim.x * kPerThread) {
        if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
        __syncthreads();
        int g[kPerThread];
        uint32_t slot[kPerThread];
#pragma unroll
        for (int k = 0; k < kPerThread; k++) {
            const long long q = base + (long long)k * blockDim.x + threadIdx.x;
            g[k] = -1;
            if (q < q1 && (!active || active[q])) {
                g[k] = classify_query(hole, board, n_players, q);
                if (g[k] >= 0 && counts[g[k]] == 0) g[k] = -1;          // a shape outside the caller's mask
                if (g[k] >= 0) slot[k] = atomicAdd(&s_cnt[g[k]], 1u);
            }
        }
        __syncthreads();
        if (threadIdx.x < 64 && s_cnt[threadIdx.x])
            s_base[threadIdx.x] = offsets[threadIdx.x] + atomicAdd(&cursors[threadIdx.x], s_cnt[threadIdx.x]);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kPerThread; k++)
            if (g[k] >= 0) qindex[s_base[g[k]] + slot[k]] = (int32_t)(base + (long long)k * blockDim.x + threadIdx.x);
        __syncthreads();
    }
}

// ---- adaptive calls (npk_equity_batch_adaptive, npk_equity_ranges_batch_adaptive) ----------------------------------------
// Workspace: the header and qindex of npk_equity_workspace_bytes(Q) (reused by every round), then at adaptive_base(Q) a
// 64-byte block of u32 words -- queries still active (a running sum), blocks done, invalid queries, the qindex cursor of the
// range call, the next round's {chunk, chunks, queries} -- and active [Q] bytes.  The running sum, the cursor and the block
// count are reset by the block that consumes them.
constexpr int kAdActive = 0, kAdBlocksDone = 1, kAdInvalid = 2, kAdCursor = 3, kAdPlan = 4, kAdHeaderBytes = 64;
int64_t adaptive_base(int64_t Q) { return (npk_equity_workspace_bytes(Q) + 255) & ~int64_t(255); }

// The stopping rule after checkpoint t: x = wins + ties, p = (x + 1) / (t + 2), var = p (1 - p) / t, stop if var <= bound
// (= stderr * stderr).  IEEE double, rounded to nearest at every step and never contracted into an FMA, so that a host restatement
// in double arithmetic takes the same decision at the boundary.
__device__ __forceinline__ bool adaptive_stop(unsigned long long x, long long t, double bound)
{
    const double p = __ddiv_rn(__dadd_rn(__ull2double_rn(x), 1.0), __ll2double_rn(t + 2));
    const double var = __ddiv_rn(__dmul_rn(p, __dsub_rn(1.0, p)), __ll2double_rn(t));
    return var <= bound;
}

// Block sums of the queries still active (and of invalid ones) go to the workspace; the last block to finish plans the next
// round's work items from the total (items a multiple of `lanes_worth` trials, as the round's kernel iterates), publishes the
// total next to the plan and resets the sum and the cursor for the next round.
__device__ void adaptive_count(uint32_t n_active, uint32_t n_invalid, uint32_t* hdr, long long next_trials, int sm_count,
                               int lanes_worth)
{
    __shared__ uint32_t s_n[2];
    if (threadIdx.x == 0) { s_n[0] = 0; s_n[1] = 0; }
    __syncthreads();
    if (n_active) atomicAdd(&s_n[0], n_active);
    if (n_invalid) atomicAdd(&s_n[1], n_invalid);
    __syncthreads();
    if (threadIdx.x != 0) return;
    if (s_n[0]) atomicAdd(&hdr[kAdActive], s_n[0]);
    if (s_n[1]) atomicAdd(&hdr[kAdInvalid], s_n[1]);
    __threadfence();
    if (atomicAdd(&hdr[kAdBlocksDone], 1u) != gridDim.x - 1) return;
    __threadfence();
    const uint32_t total = *reinterpret_cast<volatile uint32_t*>(&hdr[kAdActive]);
    uint32_t chunk, chunks;
    npk::item_plan(total, next_trials, sm_count, lanes_worth, chunk, chunks);
    hdr[kAdPlan] = chunk; hdr[kAdPlan + 1] = chunks; hdr[kAdPlan + 2] = total;
    hdr[kAdActive] = 0; hdr[kAdBlocksDone] = 0; hdr[kAdCursor] = 0;
}

// Append the queries of the warp with `keep` to `list` at the cursor, one atomic per warp (the order does not matter: the
// counters are integer atomics).  Every lane of the warp calls it.
__device__ __forceinline__ void append_queries(uint32_t* cursor, int32_t* list, bool keep, long long q)
{
    const uint32_t votes = __ballot_sync(0xffffffffu, keep);
    if (!votes) return;
    const int lane = threadIdx.x & 31, leader = __ffs(votes) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(cursor, (uint32_t)__popc(votes));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (keep) list[base + __popc(votes & ((1u << lane) - 1u))] = (int32_t)q;
}

// The query test of npk_equity_batch_adaptive: 1 = run it, 0 = a valid query outside the caller's shapes, -1 = invalid.
// (The range call's is RangeTest.)
struct ShapeTest {
    const uint8_t *hole, *board, *n_players;
    unsigned long long shape_mask;
    __device__ int operator()(long long q) const
    {
        const int g = classify_query(hole, board, n_players, q);
        return g < 0 ? -1 : (int)(shape_mask >> g & 1ull);
    }
};

// Zero the outputs (the stopping rule reads the counters, so the call owns them), mark the queries `test` accepts active,
// list them in `qindex` when it is given, and plan the first round.  Grid: one thread per query (append_queries wants whole
// warps).
template <class Test>
__global__ void __launch_bounds__(256) adaptive_init_kernel(Test test, long long Q, unsigned long long* wins,
                                                            unsigned long long* ties, unsigned long long* win_types,
                                                            unsigned long long* passes, unsigned long long* trials,
                                                            uint8_t* active, uint32_t* hdr, int32_t* qindex,
                                                            long long first_trials, int sm_count, int lanes_worth)
{
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int v = 0;
    if (q < Q) {
        wins[q] = 0; ties[q] = 0; trials[q] = 0;
        if (win_types)
            for (int i = 0; i < 9; i++) win_types[9 * q + i] = 0;
        if (passes) passes[q] = 0;
        v = test(q);
        active[q] = v > 0 ? 1 : 0;
    }
    if (qindex) append_queries(hdr + kAdCursor, qindex, v > 0, q);
    adaptive_count(v > 0 ? 1u : 0u, v < 0 ? 1u : 0u, hdr, first_trials, sm_count, lanes_worth);
}

// After the round that ends at checkpoint t: retire every active query the rule stops (all of them in the final round),
// recording trials = t, and plan the next round of `next_trials` trials for the queries left.  Grid: one thread per query.
// `qindex` or null: the list of the queries left, which the range kernels read (the all-shapes kernel's rounds classify).
__global__ void __launch_bounds__(256) adaptive_retire_kernel(long long Q, const unsigned long long* wins,
                                                              const unsigned long long* ties, unsigned long long* trials,
                                                              uint8_t* active, uint32_t* hdr, long long t, double max_stderr,
                                                              int final_round, long long next_trials, int sm_count,
                                                              int32_t* qindex, int lanes_worth)
{
    const double bound = __dmul_rn(max_stderr, max_stderr);
    uint32_t n = 0;
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // one query per thread: a grid-stride loop kept
    if (q < Q && active[q]) {                                               // enough values live across the division's slow
        if (final_round || adaptive_stop(wins[q] + ties[q], t, bound)) {    // path to spill
            active[q] = 0;
            trials[q] = (unsigned long long)t;
        } else {
            n = 1;
        }
    }
    if (qindex) append_queries(hdr + kAdCursor, qindex, n != 0, q);
    adaptive_count(n, 0, hdr, next_trials, sm_count, lanes_worth);
}

// T_0 = min_trials, T_{k+1} = min(2 T_k, max_trials), up to max_trials.
std::vector<long long> adaptive_checkpoints(long long min_trials, long long max_trials)
{
    std::vector<long long> t{min_trials};
    while (t.back() < max_trials) t.push_back(t.back() > max_trials / 2 ? max_trials : 2 * t.back());
    return t;
}

// The arguments of the stopping rule, checked before anything else: these errors need no device.
int check_rule(int64_t min_trials, int64_t max_trials, double max_stderr)
{
    if (!std::isfinite(max_stderr) || max_stderr <= 0.0)
        return fail(NPK_ERR_INVALID_ARGUMENT, "stderr must be a finite number > 0");
    if (min_trials < 1) return fail(NPK_ERR_INVALID_ARGUMENT, "min_trials must be >= 1");
    if (min_trials > max_trials) return fail(NPK_ERR_INVALID_ARGUMENT, "min_trials must not exceed max_trials");
    return NPK_OK;
}

// The checkpoint sequence of an adaptive call, back to back on `s`; `p` holds the call's outputs and launch fields.  Start with
// adaptive_init_kernel (with `validate`, an invalid query is an error before any trial: one read-back, the message
// invalid_queries(n, causes, tail)), then one round per checkpoint: `round(active)` enqueues the trials [T_{k-1}, T_k)
// (p.trial_offset, p.trials) of the queries still active, and the rule retires queries and plans the next round, appending
// the queries left to `qindex` when it is given.  Items are planned in multiples of `lanes_worth` trials.
template <class Test, class Round>
int run_adaptive(const DeviceState& ds, npk::EquityParams& p, const Test& test, int64_t Q, int64_t min_trials,
                 int64_t max_trials, double max_stderr, uint64_t* trials, uint8_t* ws, int32_t* qindex, int lanes_worth,
                 bool validate, const char* what, const char* causes, const char* tail, cudaStream_t s, const Round& round)
{
    uint32_t* hdr = reinterpret_cast<uint32_t*>(ws + adaptive_base(Q));
    uint8_t* active = ws + adaptive_base(Q) + kAdHeaderBytes;
    auto* n_trials = reinterpret_cast<unsigned long long*>(trials);
    const std::vector<long long> cp = adaptive_checkpoints(min_trials, max_trials);
    const unsigned int grid = (unsigned int)((Q + 255) / 256);

    cudaError_t e = cudaMemsetAsync(hdr, 0, kAdHeaderBytes, s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(workspace)");
    adaptive_init_kernel<<<grid, 256, 0, s>>>(test, Q, p.wins, p.ties, p.win_types, p.passes, n_trials, active, hdr, qindex,
                                              cp[0], ds.sm_count, lanes_worth);
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "adaptive_init_kernel launch");
    int rc;
    if (validate) {
        uint32_t bad = 0;
        if ((rc = read_word(hdr + kAdInvalid, s, &bad, what))) return rc;
        if (bad) return fail(NPK_ERR_INVALID_CARDS, invalid_queries(bad, causes, tail));
    }
    p.plan = hdr + kAdPlan;
    long long done = 0;
    for (size_t k = 0; k < cp.size(); k++) {
        p.trials = cp[k] - done;
        p.trial_offset = done;
        if ((rc = round(active))) return rc;
        const bool final_round = k + 1 == cp.size();
        adaptive_retire_kernel<<<grid, 256, 0, s>>>(Q, p.wins, p.ties, n_trials, active, hdr, cp[k], max_stderr,
                                                    final_round ? 1 : 0, final_round ? 0 : cp[k + 1] - cp[k], ds.sm_count,
                                                    qindex, lanes_worth);
        if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "adaptive_retire_kernel launch");
        done = cp[k];
    }
    return NPK_OK;
}

// Work items of a launch (npk::item_plan).  Returns the number of items per query.
long long plan_items(npk::EquityParams& p, long long queries, long long trials, int sm_count, int lanes_worth = 64)
{
    npk::item_plan(queries, trials, sm_count, lanes_worth, p.chunk, p.chunks);
    return p.chunks;
}

int grid_for(const DeviceState& ds, long long items, int warps_per_cta)
{
    long long ctas = (items + warps_per_cta - 1) / warps_per_cta;
    if (ctas < 1) ctas = 1;
    if (ctas > ds.sm_count) ctas = ds.sm_count;
    return (int)ctas;
}

int check_deal_mode(int deal_mode)
{
    if (deal_mode == NPK_DEAL_UNIFORM || deal_mode == NPK_DEAL_REFERENCE) return NPK_OK;
    return fail(NPK_ERR_INVALID_ARGUMENT, "deal_mode must be NPK_DEAL_UNIFORM or NPK_DEAL_REFERENCE");
}

// First checks of the batched Monte-Carlo entry points: the current device and the sizes.  Returns NPK_OK, an error code,
// or kEmptyBatch when there is nothing to compute (Q or trials is 0; the pointers are not looked at then).
constexpr int kEmptyBatch = 1;
int batch_start(DeviceState** ds, int64_t Q, int64_t trials, int64_t trial_offset)
{
    int rc = current_state(ds);
    if (rc) return rc;
    if (Q < 0 || trials < 0 || trial_offset < 0) return fail(NPK_ERR_INVALID_ARGUMENT, "negative size");
    if (Q == 0 || trials == 0) return kEmptyBatch;
    if (Q > 0x7fffffffLL) return fail(NPK_ERR_INVALID_ARGUMENT, "at most 2^31-1 queries per call");
    return NPK_OK;
}

// Zero the workspace header (work counters, shape counts, invalid / abort words) before a batch's kernels.
int clear_workspace(uint8_t* ws, cudaStream_t s)
{
    const cudaError_t e = cudaMemsetAsync(ws, 0, kWsIndex, s);
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "cudaMemsetAsync(workspace)");
}

// The fields of a Monte-Carlo launch that every entry point fills alike, and the plan of its work items: returns the items
// per query.  Only the reference's dealer and the range kernels count `passes`; the uniform dealer never reads it.
long long fill_params(npk::EquityParams& p, const DeviceState& ds, const uint8_t* hole, const uint8_t* board,
                      const uint8_t* n_players, int64_t Q, int64_t trials, int64_t trial_offset, int64_t query_offset,
                      uint64_t seed, int deal_mode, uint64_t* wins, uint64_t* ties, uint64_t* win_types, uint64_t* passes,
                      uint32_t* abort_flag, int lanes_worth = 64)
{
    p = npk::EquityParams{};
    p.tables = ds.t;
    p.hole = hole; p.board = board; p.n_players = n_players;
    p.nq = Q; p.trials = trials; p.trial_offset = trial_offset; p.query_offset = (uint32_t)query_offset;
    p.seed_lo = (uint32_t)seed; p.seed_hi = (uint32_t)(seed >> 32);
    p.reference_dealer = deal_mode == NPK_DEAL_REFERENCE ? 1u : 0u;
    p.wins = reinterpret_cast<unsigned long long*>(wins);
    p.ties = reinterpret_cast<unsigned long long*>(ties);
    p.win_types = reinterpret_cast<unsigned long long*>(win_types);
    p.passes = reinterpret_cast<unsigned long long*>(passes);
    p.abort_flag = abort_flag;
    return plan_items(p, Q, trials, ds.sm_count, lanes_worth);
}

}  // namespace

extern "C" {

const char* npk_last_error(void) { return g_err.c_str(); }

int npk_init_host_tables(void) { return ensure_host_tables(); }

int npk_init(int device)
{
    int rc = ensure_host_tables();
    if (rc) return rc;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(NPK_ERR_CUDA, std::string("no CUDA device available (there is no CPU fallback): ") +
                                      (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device < 0 || device >= count || device >= kMaxDevices) return fail(NPK_ERR_INVALID_ARGUMENT, "bad device index");
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    std::lock_guard<std::mutex> lk(g_mu);
    DeviceState& ds = g_dev[device];
    if (ds.ready) return NPK_OK;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
    if (prop.major < 10)
        return fail(NPK_ERR_CUDA, "libnpk is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
                                      std::to_string(prop.minor));
    ds.sm_count = prop.multiProcessorCount;
    if (cudaDeviceGetAttribute(&ds.clock_khz, cudaDevAttrClockRate, device) != cudaSuccess || ds.clock_khz <= 0) ds.clock_khz = 2000000;

    const size_t vb = (g_tables.value.size() * 2 + 15) & ~size_t(15);
    const size_t rb = g_tables.row_offset.size() * 2, fb = g_tables.flush.size() * 2, db = 52 * 4;
    std::vector<uint8_t> blob(vb + rb + fb + 256, 0);
    std::memcpy(blob.data(), g_tables.value.data(), g_tables.value.size() * 2);
    std::memcpy(blob.data() + vb, g_tables.row_offset.data(), rb);
    std::memcpy(blob.data() + vb + rb, g_tables.flush.data(), fb);
    uint32_t desc[52];
    for (int c = 0; c < 52; c++) desc[c] = npk::card_desc(c);
    std::memcpy(blob.data() + vb + rb + fb, desc, db);
    e = cudaMalloc(&ds.blob, blob.size());
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(tables)");
    e = cudaMemcpy(ds.blob, blob.data(), blob.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(tables)");
    uint8_t* b = static_cast<uint8_t*>(ds.blob);
    ds.t.value = reinterpret_cast<const uint16_t*>(b);
    ds.t.rowoff = reinterpret_cast<const uint16_t*>(b + vb);
    ds.t.flush = reinterpret_cast<const uint16_t*>(b + vb + rb);
    ds.t.desc = reinterpret_cast<const uint32_t*>(b + vb + rb + fb);
    ds.t.value_bytes = (uint32_t)vb;
    ds.t.rowoff_bytes = (uint32_t)rb;
    ds.t.flush_bytes = (uint32_t)fb;
    for (int i = 0; i < 10; i++) ds.t.type_start[i] = g_tables.type_start[i];
    e = cudaMalloc(&ds.t.check, 4);
    if (e == cudaSuccess) e = cudaMemset(ds.t.check, 0, 4);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(check word)");
    ds.ready = true;
    return NPK_OK;
}

int npk_set_device(int device)
{
    if (device < 0 || device >= kMaxDevices || !g_dev[device].ready)
        return fail(NPK_ERR_NOT_INITIALIZED, "npk_init(device) has not been called for this device");
    cudaError_t e = cudaSetDevice(device);
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "cudaSetDevice");
}

int npk_shutdown(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    for (int d = 0; d < kMaxDevices; d++) {
        if (!g_dev[d].ready) continue;
        cudaSetDevice(d);
        cudaFree(g_dev[d].blob);
        cudaFree(g_dev[d].t.check);
        g_dev[d] = DeviceState{};
    }
    t_stage.release();            // the calling thread's staging; other threads release theirs when they exit
    return NPK_OK;
}

int npk_checked_status(int* checked_build, uint32_t* first_failure)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
#ifdef NPK_CHECKED
    if (checked_build) *checked_build = 1;
#else
    if (checked_build) *checked_build = 0;
#endif
    uint32_t v = 0;
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(&v, ds->t.check, 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return cuda_fail(e, "npk_checked_status");
    if (first_failure) *first_failure = v;
    return NPK_OK;
}

int npk_sm_count(void)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    return rc ? rc : ds->sm_count;
}

int npk_get_tables(uint16_t* value, int64_t* n_value, uint16_t* rowoff, uint16_t* flush, uint32_t* desc,
                   uint16_t* type_start, uint64_t* class_keys)
{
    int rc = ensure_host_tables();
    if (rc) return rc;
    if (n_value) *n_value = (int64_t)g_tables.value.size();
    if (value) std::memcpy(value, g_tables.value.data(), g_tables.value.size() * 2);
    if (rowoff) std::memcpy(rowoff, g_tables.row_offset.data(), g_tables.row_offset.size() * 2);
    if (flush) std::memcpy(flush, g_tables.flush.data(), g_tables.flush.size() * 2);
    if (desc) for (int c = 0; c < 52; c++) desc[c] = npk::card_desc(c);
    if (type_start) for (int i = 0; i < 10; i++) type_start[i] = g_tables.type_start[i];
    if (class_keys) std::memcpy(class_keys, g_tables.class_key.data(), g_tables.class_key.size() * 8);
    return NPK_OK;
}

int npk_host_rank7(const uint8_t* cards, int64_t n, uint16_t* ranks)
{
    int rc = ensure_host_tables();
    if (rc) return rc;
    for (int64_t i = 0; i < n; i++) {
        for (int k = 0; k < 7; k++)
            if (cards[7 * i + k] >= 52) return fail(NPK_ERR_INVALID_CARDS, "card id >= 52");
        ranks[i] = npk::host_rank7(g_tables, cards + 7 * i);
    }
    return NPK_OK;
}

int64_t npk_equity_workspace_bytes(int64_t Q) { return kWsIndex + 4 * (Q > 0 ? Q : 0) + 64; }

namespace {
// Mixed batch: classify on the device (two small kernels), then ONE persistent kernel for all shapes (npk_mixed.cu).
// Nothing is read back: asynchronous on `s`.
// `active` [Q] or null: an adaptive call's round, which runs only the queries still active.
int enqueue_mixed(DeviceState* ds, npk::EquityParams& p, const uint8_t* hole, const uint8_t* board, const uint8_t* n_players,
                  int64_t Q, uint64_t shape_mask, uint8_t* ws, cudaStream_t s, const uint8_t* active = nullptr)
{
    const int cg = (int)std::min<long long>((Q + 255) / 256, 4 * ds->sm_count);
    classify_count_kernel<<<cg, 256, 0, s>>>(hole, board, n_players, Q, ws, shape_mask, active);
    classify_fill_kernel<<<cg, 256, 0, s>>>(hole, board, n_players, Q, ws, active);
    p.group = reinterpret_cast<const uint32_t*>(ws + kWsCounts);
    p.qindex = reinterpret_cast<const int32_t*>(ws + kWsIndex);
    p.nq = 0;
    p.work_counter = reinterpret_cast<unsigned long long*>(ws + kWsCounters);
    cudaError_t e = npk::launch_equity_mixed(p, ds->sm_count, s);
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "equity_mixed_kernel launch");
}
}  // namespace

int npk_equity_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                     int uniform_players, int uniform_known, uint64_t seed, int64_t trial_offset, int64_t query_offset,
                     int deal_mode, uint32_t flags, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes,
                     void* workspace, void* stream)
{
    DeviceState* ds;
    int rc = batch_start(&ds, Q, trials, trial_offset);
    if (rc) return rc == kEmptyBatch ? NPK_OK : rc;
    if (!hole || !board || !n_players || !wins_strict || !ties || !workspace)
        return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if ((rc = check_deal_mode(deal_mode))) return rc;
    const bool uniform_shape = uniform_players >= 0 && uniform_known >= 0;
    if (uniform_shape && (uniform_players < 1 || uniform_players > 10 || uniform_known > 5))
        return fail(NPK_ERR_INVALID_CARDS, "players must be 1..10 and known board cards 0..5");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    if ((rc = clear_workspace(ws, s))) return rc;

    npk::EquityParams p;
    const long long chunks = fill_params(p, *ds, hole, board, n_players, Q, trials, trial_offset, query_offset, seed, deal_mode,
                                         wins_strict, ties, win_types, passes,
                                         reinterpret_cast<uint32_t*>(ws + kWsAbort));   // + 15 diagnostic words, all inside the header
    const bool validate = (flags & NPK_FLAG_VALIDATE) != 0;
    cudaError_t e;

    if (uniform_shape && !validate) {
        p.work_counter = reinterpret_cast<unsigned long long*>(ws + kWsCounters);
        e = npk::launch_equity_uniform(uniform_players - 1, 5 - uniform_known, p, Q * chunks, ds->sm_count, s);
        return e == cudaSuccess ? NPK_OK : cuda_fail(e, "equity_uniform_kernel launch");
    }
    if (uniform_shape) {
        // validated: classify first (one small device->host read), then the shape's own kernel
        const int cg = (int)std::min<long long>((Q + 255) / 256, 4 * ds->sm_count);
        classify_count_kernel<<<cg, 256, 0, s>>>(hole, board, n_players, Q, ws, ~0ull, nullptr);
        uint32_t host[64 + 64 + 1];
        e = cudaMemcpyAsync(host, ws + kWsCounts, 4 * 129, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return cuda_fail(e, "query classification");
        if (host[128]) return fail(NPK_ERR_INVALID_CARDS, invalid_queries(host[128], kQueryCauses));
        if (host[(uniform_players - 1) * 6 + uniform_known] != (uint32_t)Q)
            return fail(NPK_ERR_INVALID_ARGUMENT, "queries do not all have the declared uniform shape");
        p.work_counter = reinterpret_cast<unsigned long long*>(ws + kWsCounters) + 1;
        e = npk::launch_equity_uniform(uniform_players - 1, 5 - uniform_known, p, Q * chunks, ds->sm_count, s);
        return e == cudaSuccess ? NPK_OK : cuda_fail(e, "equity_uniform_kernel launch");
    }
    rc = enqueue_mixed(ds, p, hole, board, n_players, Q, ~0ull, ws, s);
    if (rc || !validate) return rc;
    uint32_t bad = 0;
    if ((rc = read_word(ws + kWsInvalid, s, &bad, "mixed batch"))) return rc;
    if (bad) return fail(NPK_ERR_INVALID_CARDS, invalid_queries(bad, kQueryCauses, "; their counters are untouched, the other "
                                                                                   "queries have been computed"));
    return NPK_OK;
}

int npk_equity_batch_async(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                           uint64_t shape_mask, uint64_t seed, int64_t trial_offset, int64_t query_offset, int deal_mode,
                           uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes, void* workspace,
                           void* stream)
{
    DeviceState* ds;
    int rc = batch_start(&ds, Q, trials, trial_offset);
    if (rc) return rc == kEmptyBatch ? NPK_OK : rc;
    if (!hole || !board || !n_players || !wins_strict || !ties || !workspace)
        return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if ((rc = check_deal_mode(deal_mode))) return rc;
    shape_mask &= (1ull << kGroups) - 1ull;
    if (!shape_mask) return fail(NPK_ERR_INVALID_ARGUMENT, "empty shape mask");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    if ((rc = clear_workspace(ws, s))) return rc;
    npk::EquityParams p;
    fill_params(p, *ds, hole, board, n_players, Q, trials, trial_offset, query_offset, seed, deal_mode, wins_strict, ties,
                win_types, passes, reinterpret_cast<uint32_t*>(ws + kWsAbort));
    return enqueue_mixed(ds, p, hole, board, n_players, Q, shape_mask, ws, s);
}

int npk_equity_batch_status(const void* workspace, void* stream, uint32_t* invalid, uint32_t* skipped)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (!workspace) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    const uint8_t* ws = static_cast<const uint8_t*>(workspace);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint32_t v[2] = {0, 0};
    if ((rc = read_word(ws + kWsInvalid, s, &v[0], "npk_equity_batch_status")) ||
        (rc = read_word(ws + kWsSkipped, s, &v[1], "npk_equity_batch_status")))
        return rc;
    if (invalid) *invalid = v[0];
    if (skipped) *skipped = v[1];
    return NPK_OK;
}

int64_t npk_equity_adaptive_workspace_bytes(int64_t Q) { return adaptive_base(Q) + kAdHeaderBytes + (Q > 0 ? Q : 0); }

int npk_equity_batch_adaptive(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q,
                              int64_t min_trials, int64_t max_trials, double max_stderr, uint64_t shape_mask, uint64_t seed,
                              int64_t query_offset, int deal_mode, uint32_t flags, uint64_t* wins_strict, uint64_t* ties,
                              uint64_t* win_types, uint64_t* passes, uint64_t* trials, void* workspace, void* stream)
{
    int rc = check_rule(min_trials, max_trials, max_stderr);
    if (rc) return rc;
    DeviceState* ds;
    if ((rc = batch_start(&ds, Q, max_trials, 0))) return rc == kEmptyBatch ? NPK_OK : rc;
    if (!hole || !board || !n_players || !wins_strict || !ties || !trials || !workspace)
        return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if ((rc = check_deal_mode(deal_mode))) return rc;
    shape_mask &= (1ull << kGroups) - 1ull;
    if (!shape_mask) return fail(NPK_ERR_INVALID_ARGUMENT, "empty shape mask");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    npk::EquityParams p;
    fill_params(p, *ds, hole, board, n_players, Q, min_trials, 0, query_offset, seed, deal_mode, wins_strict, ties, win_types,
                passes, reinterpret_cast<uint32_t*>(ws + kWsAbort));
    // a round classifies the queries still active and runs the all-shapes kernel on them
    return run_adaptive(*ds, p, ShapeTest{hole, board, n_players, shape_mask}, Q, min_trials, max_trials, max_stderr, trials,
                        ws, nullptr, 64, (flags & NPK_FLAG_VALIDATE) != 0, "adaptive batch", kQueryCauses,
                        "; nothing has been computed", s, [&](const uint8_t* active) {
                            const int rc = clear_workspace(ws, s);
                            return rc ? rc : enqueue_mixed(ds, p, hole, board, n_players, Q, ~0ull, ws, s, active);
                        });
}

namespace {
// The query of a one-query call as the one-query kernels read it (ResidentMailbox::ReqA, serve_request in npk_mixed.cu):
// x = hole[0] | hole[1] << 8 | board[0] << 16 | board[1] << 24, y = board[2..4] | players << 24 | reference dealer << 31.
uint2 pack_query(const uint8_t* hole, const uint8_t* board, int players, int deal_mode)
{
    return make_uint2((unsigned int)hole[0] | (unsigned int)hole[1] << 8 | (unsigned int)board[0] << 16 |
                          (unsigned int)board[1] << 24,
                      (unsigned int)board[2] | (unsigned int)board[3] << 8 | (unsigned int)board[4] << 16 |
                          (unsigned int)players << 24 | (deal_mode == NPK_DEAL_REFERENCE ? 1u << 31 : 0u));
}

// Wait for a launched one-query kernel: spin on the sequence word it writes to mapped host memory last, and after a few
// hundred ms ask the driver.
int await_result(const volatile unsigned long long* seq_word, unsigned long long seq, cudaStream_t s)
{
    for (long spins = 0; spins < 4000000 && *seq_word != seq; spins++) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    if (*seq_word != seq) {
        const cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return cuda_fail(e, "equity kernel");
        if (*seq_word != seq) return fail(NPK_ERR_CUDA, "the one-query kernel finished without publishing its result");
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    return NPK_OK;
}

// (Re)start this thread's resident server on its stream.  `completed` = sequence number of the last request whose result has
// been received: a request posted after it is picked up by the new server at its first poll.
int resident_buffers(HostStage& st)
{
    cudaError_t e;
    if (st.res_mb) return NPK_OK;
    if ((e = cudaHostAlloc(&st.res_mb, sizeof(npk::ResidentMailbox), cudaHostAllocMapped)) != cudaSuccess) return cuda_fail(e, "cudaHostAlloc");
    std::memset(st.res_mb, 0, sizeof(npk::ResidentMailbox));
    if ((e = cudaHostGetDevicePointer(&st.res_mb_dev, st.res_mb, 0)) != cudaSuccess) return cuda_fail(e, "cudaHostGetDevicePointer");
    if ((e = cudaMalloc(&st.res_state, sizeof(npk::ResidentState))) != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    if ((e = cudaMemset(st.res_state, 0, sizeof(npk::ResidentState))) != cudaSuccess) return cuda_fail(e, "cudaMemset");
    return NPK_OK;
}

int resident_launch(DeviceState* ds, HostStage& st)
{
    cudaError_t e;
    int rc = resident_buffers(st);
    if (rc) return rc;
    st.res_dirty = true;
    if ((e = cudaMemsetAsync(st.res_state, 0, sizeof(npk::ResidentState), st.stream)) != cudaSuccess) return cuda_fail(e, "memset");
    const unsigned int completed = (unsigned int)const_cast<volatile npk::ResidentMailbox*>(st.res_mb)->done.seq;
    ++st.res_launch_id;
    e = npk::launch_equity_resident(ds->t, st.res_state, st.res_mb_dev, st.res_launch_id, completed, st.res_idle_cycles,
                                    st.res_ctas, st.stream);
    if (e != cudaSuccess) return cuda_fail(e, "resident kernel launch");
    st.res_running = true;
    return NPK_OK;
}

// One query through the resident server: post the request in the mailbox, spin on the result.  No CUDA call on this path
// unless the server has left in the meantime (idle limit) and is started again.
int resident_query(DeviceState* ds, HostStage& st, uint2 query, int64_t trials, uint64_t seed, uint64_t* wins_strict,
                   uint64_t* ties)
{
    if (!st.res_mb) { int rc = resident_launch(ds, st); if (rc) return rc; }
    volatile npk::ResidentMailbox* mb = st.res_mb;
    unsigned int seq = ++st.res_seq;
    if (seq == 0) seq = ++st.res_seq;
    // the halves that carry the sequence number go last (x86 keeps the order of stores): a record the device reads is
    // either complete or still shows the old number
    volatile unsigned long long* ra = reinterpret_cast<volatile unsigned long long*>(&st.res_mb->a);
    volatile unsigned long long* rb = reinterpret_cast<volatile unsigned long long*>(&st.res_mb->b);
    ra[1] = (unsigned long long)query.x | (unsigned long long)query.y << 32;
    rb[1] = (unsigned long long)(uint32_t)(seed >> 32);                                   // seed_hi, stop = 0
    std::atomic_thread_fence(std::memory_order_release);
    rb[0] = (unsigned long long)seq | (unsigned long long)(uint32_t)seed << 32;
    ra[0] = (unsigned long long)seq | (unsigned long long)(uint32_t)trials << 32;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    if (!st.res_running) { int rc = resident_launch(ds, st); if (rc) return rc; }
    int relaunches = 0;
    for (long spins = 0;; spins++) {
        if ((unsigned int)mb->done.seq == seq) break;
        if (mb->exited == st.res_launch_id) {                 // the server has left (idle limit): was this request served?
            std::atomic_thread_fence(std::memory_order_acquire);
            if ((unsigned int)mb->done.seq == seq) break;
            st.res_running = false;
            if (++relaunches > 3) return fail(NPK_ERR_CUDA, "the resident server keeps leaving without serving the request");
            cudaError_t e = cudaStreamSynchronize(st.stream);
            if (e != cudaSuccess) return cuda_fail(e, "resident kernel");
            int rc = resident_launch(ds, st);
            if (rc) return rc;
        }
        if ((spins & 0xFFFFF) == 0xFFFFF) {                   // every ~million spins: is the kernel still healthy?
            const cudaError_t q = cudaStreamQuery(st.stream);
            if (q != cudaSuccess && q != cudaErrorNotReady) { st.res_running = false; return cuda_fail(q, "resident kernel"); }
        }
        if (spins > 400000000L) return fail(NPK_ERR_CUDA, "the resident server did not answer");
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    wins_strict[0] = mb->done.wins; ties[0] = mb->done.ties;
    return NPK_OK;
}

// One query from the host.  Three ways, all without H2D / D2H copies, memsets or cudaStreamSynchronize on the fast path, all
// publishing the counters together with the call's sequence number in mapped host memory, where the host spins on that number:
//   * resident mode on: post the query in the mailbox of this thread's persistent server (resident_query above);
//   * wins and ties only (what get_equity needs): ONE launch of equity_oneshot_kernel, query in the kernel parameters, one packed
//     atomic per CTA, one 16-byte store (csrc/npk_mixed.cu);
//   * win types / passes wanted, or 2^28 trials and more: one launch of the shape's own kernel; the counters stay in device
//     memory between calls, the last warp of the grid hands them over and zeroes them (finish_single_call, csrc/npk_mc.cuh).
int single_query(DeviceState* ds, HostStage& st, const uint8_t* hole, const uint8_t* board, int players, int64_t trials,
                 uint64_t seed, int deal_mode, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes)
{
    cudaError_t e;
    int rc = check_deal_mode(deal_mode);
    if (rc) return rc;
    if (trials < 0) return fail(NPK_ERR_INVALID_ARGUMENT, "negative size");
    const int known = npk::validate_query(hole, board, players);
    if (known < 0) return fail(NPK_ERR_INVALID_CARDS, "query 0: card id >= 52, duplicate cards, gap in the board, or players outside 1..10");
    wins_strict[0] = 0; ties[0] = 0;
    if (win_types) std::memset(win_types, 0, 72);
    if (passes) passes[0] = 0;
    if (trials == 0) return NPK_OK;
    const uint2 query = pack_query(hole, board, players, deal_mode);
    const bool counts_only = !win_types && !passes && trials < npk::kResidentMaxTrials;   // the packed hand-over's limit
    if (st.res_enabled && counts_only) return resident_query(ds, st, query, trials, seed, wins_strict, ties);
    st.stop_resident();                            // the launches below use the stream the server would be holding
    if (counts_only) {
        // the common call: a kernel launched for this request, handing over like the resident server (npk_mixed.cu)
        if ((rc = resident_buffers(st))) return rc;
        if (st.res_dirty) {
            if ((e = cudaMemsetAsync(st.res_state, 0, sizeof(npk::ResidentState), st.stream)) != cudaSuccess) return cuda_fail(e, "memset");
            st.oneshot_parity = 0;
            st.res_dirty = false;
        }
        unsigned int seq = ++st.res_seq;
        if (seq == 0) seq = ++st.res_seq;
        e = npk::launch_equity_oneshot(ds->t, st.res_state, st.res_mb_dev, make_uint4(0u, (unsigned int)trials, query.x, query.y),
                                       make_uint4(0u, (unsigned int)seed, (unsigned int)(seed >> 32), seq), st.oneshot_parity,
                                       ds->sm_count, st.stream);
        if (e != cudaSuccess) return cuda_fail(e, "equity kernel launch");
        st.oneshot_parity ^= 1u;
        volatile npk::ResidentMailbox* mb = st.res_mb;
        if ((rc = await_result(&mb->done.seq, seq, st.stream))) return rc;
        wins_strict[0] = mb->done.wins; ties[0] = mb->done.ties;
        return NPK_OK;
    }
    if (!st.single) {
        if ((e = cudaHostAlloc(&st.single_host, sizeof(npk::SingleResult), cudaHostAllocMapped)) != cudaSuccess) return cuda_fail(e, "cudaHostAlloc");
        std::memset(st.single_host, 0, sizeof(npk::SingleResult));
        npk::SingleResult* dptr = nullptr;
        if ((e = cudaHostGetDevicePointer(&dptr, st.single_host, 0)) != cudaSuccess) return cuda_fail(e, "cudaHostGetDevicePointer");
        if ((e = cudaMalloc(&st.single, sizeof(npk::SingleCall))) != cudaSuccess) return cuda_fail(e, "cudaMalloc");
        npk::SingleCall init{};
        init.host = dptr;
        if ((e = cudaMemcpy(st.single, &init, sizeof init, cudaMemcpyHostToDevice)) != cudaSuccess) return cuda_fail(e, "cudaMemcpy");
        st.single_seq = 0;
    }
    npk::EquityParams p;
    const long long chunks = fill_params(p, *ds, nullptr, nullptr, nullptr, 1, trials, 0, 0, seed, deal_mode,
                                         reinterpret_cast<uint64_t*>(&st.single->wins),
                                         reinterpret_cast<uint64_t*>(&st.single->ties),
                                         win_types ? reinterpret_cast<uint64_t*>(st.single->win_types) : nullptr,
                                         passes ? reinterpret_cast<uint64_t*>(&st.single->passes) : nullptr,
                                         st.single->abort_flag);
    p.inline_query = (uint64_t)query.x | (uint64_t)(query.y & 0xFFFFFFu) << 32;
    p.single = st.single;
    p.single_seq = ++st.single_seq;
    p.work_counter = &st.single->work_counter;
    e = npk::launch_equity_uniform(players - 1, 5 - known, p, chunks, ds->sm_count, st.stream);
    if (e != cudaSuccess) return cuda_fail(e, "equity kernel launch");
    const volatile npk::SingleResult* r = st.single_host;
    if ((rc = await_result(&r->seq, p.single_seq, st.stream))) return rc;
    wins_strict[0] = r->wins; ties[0] = r->ties;
    if (win_types) for (int i = 0; i < 9; i++) win_types[i] = r->win_types[i];
    if (passes) passes[0] = r->passes;
    return NPK_OK;
}
}  // namespace

namespace {
// this thread's staging on the current device (created on first use, rebuilt when the thread switches devices)
int thread_stage(HostStage** out)
{
    int dev = 0;
    cudaGetDevice(&dev);
    HostStage& st = t_stage;                       // no lock, no shared stream
    if (st.device != dev) st.release();
    if (st.device < 0) {
        cudaError_t e = cudaStreamCreateWithFlags(&st.stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) return cuda_fail(e, "stream");
        st.device = dev;
    }
    *out = &st;
    return NPK_OK;
}

// Validate a batch on the host, stage it in the next slot and enqueue H2D copy + counter reset + kernels + D2H copy on that
// slot's stream.  Nothing waits for the device here.
int host_submit(DeviceState* ds, HostStage& st, const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q,
                int64_t trials, uint64_t seed, int deal_mode, uint32_t want, int64_t* ticket)
{
    (void)ds;
    if (st.res_running) st.stop_resident();          // a batch needs the SMs the resident server is holding
    int free_slot = -1;
    for (int i = 0; i < kHostSlots && free_slot < 0; i++)
        if (st.slot[i].ticket < 0) free_slot = i;
    HostSlot& sl = st.slot[free_slot < 0 ? 0 : free_slot];
    if (free_slot < 0)
        return fail(NPK_ERR_INVALID_ARGUMENT, "npk_equity_host_submit: NPK_HOST_SLOTS batches are already in flight on this "
                                              "thread; wait for one of them first");
    // a uniform shape lets the call run without the classification pass; validate on the host instead
    int up = n_players[0], uk = 0;
    for (int i = 0; i < 5; i++) uk += board[i] != 0xFF;
    bool uniform = true;
    for (int64_t q = 0; q < Q; q++) {
        const int known = npk::validate_query(hole + 2 * q, board + 5 * q, n_players[q]);
        if (known < 0) return fail(NPK_ERR_INVALID_CARDS, "query " + std::to_string(q) +
                                   ": card id >= 52, duplicate cards, gap in the board, or players outside 1..10");
        if (n_players[q] != up || known != uk) uniform = false;
    }
    cudaError_t e;
    if (!sl.stream) {
        if ((e = cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking)) != cudaSuccess) return cuda_fail(e, "stream");
        if ((e = cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "event");
    }
    if (sl.cap_q < Q) {
        sl.free_buffers();
        const int64_t cap = Q < 1024 ? 1024 : Q;
        if ((e = cudaMallocHost(&sl.h_in, 8 * cap)) != cudaSuccess) return cuda_fail(e, "cudaMallocHost");
        if ((e = cudaMallocHost(&sl.h_out, 8 * 12 * cap)) != cudaSuccess) return cuda_fail(e, "cudaMallocHost");
        if ((e = cudaMalloc(&sl.d_in, 8 * cap)) != cudaSuccess) return cuda_fail(e, "cudaMalloc");
        if ((e = cudaMalloc(&sl.d_out, 8 * 12 * cap)) != cudaSuccess) return cuda_fail(e, "cudaMalloc");
        if ((e = cudaMalloc(&sl.d_ws, npk_equity_workspace_bytes(cap))) != cudaSuccess) return cuda_fail(e, "cudaMalloc");
        sl.cap_q = cap;
    }
    std::memcpy(sl.h_in, hole, 2 * Q);
    std::memcpy(sl.h_in + 2 * Q, board, 5 * Q);
    std::memcpy(sl.h_in + 7 * Q, n_players, Q);
    const bool types = want & 1u, pass = want & 2u;
    const size_t n_out = (size_t)Q * (pass ? 12 : (types ? 11 : 2));
    if ((e = cudaMemcpyAsync(sl.d_in, sl.h_in, 8 * Q, cudaMemcpyHostToDevice, sl.stream)) != cudaSuccess) return cuda_fail(e, "H2D");
    if ((e = cudaMemsetAsync(sl.d_out, 0, 8 * n_out, sl.stream)) != cudaSuccess) return cuda_fail(e, "memset");
    uint64_t* d_wins = sl.d_out;
    uint64_t* d_ties = sl.d_out + Q;
    uint64_t* d_types = sl.d_out + 2 * Q;
    uint64_t* d_pass = sl.d_out + 11 * Q;
    int rc = npk_equity_batch(sl.d_in, sl.d_in + 2 * Q, sl.d_in + 7 * Q, Q, trials, uniform ? up : -1, uniform ? uk : -1, seed,
                              0, 0, deal_mode, 0, d_wins, d_ties, types ? d_types : nullptr, pass ? d_pass : nullptr,
                              sl.d_ws, sl.stream);
    if (rc) return rc;
    if ((e = cudaMemcpyAsync(sl.h_out, sl.d_out, 8 * n_out, cudaMemcpyDeviceToHost, sl.stream)) != cudaSuccess) return cuda_fail(e, "D2H");
    if ((e = cudaEventRecord(sl.done, sl.stream)) != cudaSuccess) return cuda_fail(e, "event record");
    sl.Q = Q;
    sl.want = want;
    sl.ticket = (st.next_ticket++) * kHostSlots + free_slot;      // ticket % NPK_HOST_SLOTS = its slot
    *ticket = sl.ticket;
    return NPK_OK;
}

int host_wait(HostStage& st, int64_t ticket, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes)
{
    if (ticket < 0) return fail(NPK_ERR_INVALID_ARGUMENT, "npk_equity_host_wait: bad ticket");
    HostSlot& sl = st.slot[ticket % kHostSlots];
    if (sl.ticket != ticket)
        return fail(NPK_ERR_INVALID_ARGUMENT, "npk_equity_host_wait: no such batch in flight on this thread (tickets belong to "
                                              "the submitting thread and can be waited for once)");
    cudaError_t e = cudaEventSynchronize(sl.done);
    sl.ticket = -1;
    if (e != cudaSuccess) return cuda_fail(e, "equity kernels");
    const int64_t Q = sl.Q;
    if (wins_strict) std::memcpy(wins_strict, sl.h_out, 8 * Q);
    if (ties) std::memcpy(ties, sl.h_out + Q, 8 * Q);
    if (win_types && (sl.want & 1u)) std::memcpy(win_types, sl.h_out + 2 * Q, 8 * 9 * Q);
    if (passes && (sl.want & 2u)) std::memcpy(passes, sl.h_out + 11 * Q, 8 * Q);
    return NPK_OK;
}
}  // namespace

int npk_equity_host(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                    uint64_t seed, int deal_mode, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types,
                    uint64_t* passes)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (Q <= 0) return Q == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative Q");
    if (!hole || !board || !n_players || !wins_strict || !ties) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    HostStage* st;
    if ((rc = thread_stage(&st))) return rc;
    if (Q == 1)
        return single_query(ds, *st, hole, board, n_players[0], trials, seed, deal_mode, wins_strict, ties, win_types, passes);
    int64_t ticket = -1;
    rc = host_submit(ds, *st, hole, board, n_players, Q, trials, seed, deal_mode, (win_types ? 1u : 0u) | (passes ? 2u : 0u),
                     &ticket);
    if (rc) return rc;
    return host_wait(*st, ticket, wins_strict, ties, win_types, passes);
}

int64_t npk_equity_host_submit(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                               uint64_t seed, int deal_mode, uint32_t want)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (Q <= 0) return fail(NPK_ERR_INVALID_ARGUMENT, "npk_equity_host_submit: Q must be positive");
    if (!hole || !board || !n_players) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (trials < 0) return fail(NPK_ERR_INVALID_ARGUMENT, "negative size");
    HostStage* st;
    if ((rc = thread_stage(&st))) return rc;
    int64_t ticket = -1;
    rc = host_submit(ds, *st, hole, board, n_players, Q, trials, seed, deal_mode, want, &ticket);
    return rc ? rc : ticket;
}

int npk_equity_host_wait(int64_t ticket, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    HostStage* st;
    if ((rc = thread_stage(&st))) return rc;
    return host_wait(*st, ticket, wins_strict, ties, win_types, passes);
}

/* One query from the host with as few arguments as a foreign-function call can have (the Python drop-in's get_equity):
 * packed = hole[0] | hole[1] << 8 | board[0..4] << 16.. (bytes, 0xFF = no card); out[12] = wins, ties, win types[9], passes. */
int npk_equity_one(uint64_t packed, int players, int64_t trials, uint64_t seed, int deal_mode, uint32_t want, uint64_t* out)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (!out) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    uint8_t q[7];
    for (int i = 0; i < 7; i++) q[i] = (uint8_t)(packed >> (8 * i));
    HostStage* stp;
    if ((rc = thread_stage(&stp))) return rc;
    return single_query(ds, *stp, q, q + 2, players, trials, seed, deal_mode, out, out + 1, (want & 1u) ? out + 2 : nullptr,
                        (want & 2u) ? out + 11 : nullptr);
}

int npk_resident_start(int ctas, int idle_us)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    HostStage* st;
    if ((rc = thread_stage(&st))) return rc;
    if (ctas <= 0 || ctas > ds->sm_count) ctas = ds->sm_count;
    if (ctas > 255) ctas = 255;                              // the CTA count of the packed accumulator has 8 bits
    if (idle_us <= 0) idle_us = 200;
    if (idle_us > 100000) idle_us = 100000;                  // the kernel must never hold the device for long on its own
    if (st->device >= 0 && st->device < kMaxDevices) {
        uintptr_t none = 0;
        const uintptr_t mine = reinterpret_cast<uintptr_t>(st);
        if (!g_resident_owner[st->device].compare_exchange_strong(none, mine) && none != mine)
            return fail(NPK_ERR_INVALID_ARGUMENT, "another thread of this process already runs the resident server on this device "
                                                  "(one per device: a second one could not get the SMs the first one holds)");
    }
    st->stop_resident();
    st->res_ctas = ctas;
    st->res_idle_cycles = (long long)idle_us * ds->clock_khz / 1000;
    st->res_enabled = true;
    return resident_launch(ds, *st);
}

int npk_resident_stop(void)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    HostStage* st;
    if ((rc = thread_stage(&st))) return rc;
    st->res_enabled = false;
    st->stop_resident();
    st->release_resident_slot();
    return NPK_OK;
}

// ---- trial-sharded jobs: count reduction over NVLink peer memory inside the kernel -----------------------------------------
namespace {
struct PeerGroup {
    int device = -1, rank = 0, world = 1;
    int64_t stride = 0;                       // u64 words per (parity, rank) slot
    uint8_t* buf = nullptr;                   // this rank's PeerBuf: flags [2][kMaxPeers] u64, then slots [2][world][stride] u64
    void* peer_buf[npk::kMaxPeers] = {};      // every rank's buffer in this process's address space (own: buf)
    npk::PeerCall* call = nullptr;            // device copy of the pointers + local counters' bookkeeping
    unsigned long long* acc = nullptr;        // local counters [stride]
    uint32_t* abort_flag = nullptr;
    unsigned long long epoch = 0;
    bool connected = false;
};
constexpr size_t kPeerFlagBytes = 2 * npk::kMaxPeers * sizeof(unsigned long long);
}  // namespace

extern "C" {

int npk_peer_create(int rank, int world, int64_t max_words, void** group, uint8_t* handle /*[64] host*/)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (!group || !handle || world < 1 || world > npk::kMaxPeers || rank < 0 || rank >= world || max_words < 2)
        return fail(NPK_ERR_INVALID_ARGUMENT, "npk_peer_create: 1..16 ranks, rank inside, max_words >= 2");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    PeerGroup* g = new PeerGroup;
    cudaGetDevice(&g->device);
    g->rank = rank; g->world = world; g->stride = max_words;
    const size_t bytes = kPeerFlagBytes + (size_t)2 * world * max_words * 8;
    cudaError_t e = cudaMalloc(&g->buf, bytes);
    if (e == cudaSuccess) e = cudaMemset(g->buf, 0, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&g->acc, (size_t)max_words * 8);
    if (e == cudaSuccess) e = cudaMemset(g->acc, 0, (size_t)max_words * 8);
    if (e == cudaSuccess) e = cudaMalloc(&g->call, sizeof(npk::PeerCall));
    if (e == cudaSuccess) e = cudaMalloc(&g->abort_flag, 64);
    if (e == cudaSuccess) e = cudaMemset(g->abort_flag, 0, 64);
    cudaIpcMemHandle_t h;
    std::memset(&h, 0, sizeof h);
    if (e == cudaSuccess && world > 1) e = cudaIpcGetMemHandle(&h, g->buf);
    if (e != cudaSuccess) {
        cudaFree(g->buf); cudaFree(g->acc); cudaFree(g->call); cudaFree(g->abort_flag);
        delete g;
        return cuda_fail(e, "npk_peer_create");
    }
    std::memcpy(handle, &h, 64);
    *group = g;
    return NPK_OK;
}

int npk_peer_connect(void* group, const uint8_t* handles /*[world,64] host, rank order*/)
{
    PeerGroup* g = static_cast<PeerGroup*>(group);
    if (!g || !handles) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (g->connected) return NPK_OK;
    cudaError_t e = cudaSetDevice(g->device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    npk::PeerCall pc{};
    for (int r = 0; r < g->world; r++) {
        if (r == g->rank) g->peer_buf[r] = g->buf;
        else {
            cudaIpcMemHandle_t h;
            std::memcpy(&h, handles + 64 * r, 64);
            e = cudaIpcOpenMemHandle(&g->peer_buf[r], h, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) return cuda_fail(e, "cudaIpcOpenMemHandle (are the ranks' GPUs NVLink / P2P peers on one node?)");
        }
        pc.flags[r] = reinterpret_cast<unsigned long long*>(g->peer_buf[r]);
        pc.slots[r] = reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(g->peer_buf[r]) + kPeerFlagBytes);
    }
    pc.acc = g->acc; pc.world = (uint32_t)g->world; pc.rank = (uint32_t)g->rank; pc.stride = (uint32_t)g->stride;
    e = cudaMemcpy(g->call, &pc, sizeof pc, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(PeerCall)");
    g->connected = true;
    return NPK_OK;
}

int npk_peer_destroy(void* group)
{
    PeerGroup* g = static_cast<PeerGroup*>(group);
    if (!g) return NPK_OK;
    cudaSetDevice(g->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < g->world; r++)
        if (r != g->rank && g->peer_buf[r]) cudaIpcCloseMemHandle(g->peer_buf[r]);
    cudaFree(g->buf); cudaFree(g->acc); cudaFree(g->call); cudaFree(g->abort_flag);
    delete g;
    return NPK_OK;
}

int npk_peer_error(void* group, int* error /*host*/)
{
    PeerGroup* g = static_cast<PeerGroup*>(group);
    if (!g || !error) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    unsigned int v = 0;
    cudaError_t e = cudaMemcpy(&v, &g->call->error, 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return cuda_fail(e, "npk_peer_error");
    *error = (int)v;
    return NPK_OK;
}

int npk_equity_batch_sharded(void* group, const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q,
                             int64_t trials_total, int players, int known, uint64_t seed, int64_t query_offset,
                             int deal_mode, uint64_t* totals, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    PeerGroup* g = static_cast<PeerGroup*>(group);
    if (!g || !g->connected) return fail(NPK_ERR_INVALID_ARGUMENT, "peer group not connected");
    if (!hole || !board || !n_players || !totals) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (Q <= 0 || 2 * Q > g->stride) return fail(NPK_ERR_INVALID_ARGUMENT, "Q must be 1..max_words/2 of the peer group");
    if (trials_total < 0) return fail(NPK_ERR_INVALID_ARGUMENT, "negative size");
    if (players < 1 || players > 10 || known < 0 || known > 5) return fail(NPK_ERR_INVALID_CARDS, "players must be 1..10 and known board cards 0..5");
    if ((rc = check_deal_mode(deal_mode))) return rc;
    // this rank's trial range: the same split as neuron_poker_b200.dist.trial_shard
    const int64_t base = trials_total / g->world, extra = trials_total % g->world;
    const int64_t begin = g->rank * base + std::min<int64_t>(g->rank, extra);
    const int64_t count = base + (g->rank < extra ? 1 : 0);
    npk::EquityParams p;
    const long long chunks = fill_params(p, *ds, hole, board, n_players, Q, count, begin, query_offset, seed, deal_mode,
                                         reinterpret_cast<uint64_t*>(g->acc), reinterpret_cast<uint64_t*>(g->acc + Q), nullptr,
                                         nullptr, g->abort_flag);
    p.peer = g->call; p.peer_epoch = ++g->epoch; p.peer_totals = reinterpret_cast<unsigned long long*>(totals);
    p.peer_words = (uint32_t)(2 * Q);
    p.work_counter = &g->call->work_counter;
    // a rank without trials (more ranks than trials) still takes part in the exchange: one item-less CTA
    cudaError_t e = npk::launch_equity_uniform(players - 1, 5 - known, p, std::max<long long>(Q * chunks, 1), ds->sm_count,
                                               static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "equity kernel launch (sharded)");
}

}  // extern "C"

// ---- ranges ------------------------------------------------------------------------------------------------------------
namespace {
// Is query q of a range call valid?  `hole` is null when the hero is drawn from a range.
__device__ bool range_query_valid(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                                  const uint8_t* known_opp, int n_known, long long q)
{
    const int np = n_players[q];
    unsigned long long mask;
    int bad = npk::validate_query(hole ? hole + 2 * q : nullptr, board + 5 * q, np, &mask) < 0;
    if (ghost) {
        // the reference pops ghost cards from the deck first (montecarlo_python.py:206-208): a board card equal to
        // a ghost card then fails list.index (ValueError); a hero card equal to one is silently kept (:154-161)
        const int g0 = ghost[2 * q], g1 = ghost[2 * q + 1];
        if ((g0 == 0xFF) != (g1 == 0xFF)) bad = 1;
        else if (g0 != 0xFF) {
            if (g0 >= 52 || g1 >= 52 || g0 == g1) bad = 1;
            else { bad |= (int)((mask >> g0 | mask >> g1) & 1ull); mask |= (1ull << g0) | (1ull << g1); }
        }
    }
    // opponents with known cards: valid ids, no card twice anywhere, and no more of them than opponents
    if (n_known > np - 1) bad = 1;
    for (int f = 0; f < 2 * n_known; f++) {
        const int c = known_opp[2 * q * n_known + f];
        if (c >= 52) bad = 1; else { bad |= (int)(mask >> c & 1ull); mask |= 1ull << c; }
    }
    return !bad;
}

__global__ void validate_ranges_kernel(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players,
                                       const uint8_t* ghost, const uint8_t* known_opp, int n_known, long long Q, uint8_t* ws)
{
    uint32_t* invalid = reinterpret_cast<uint32_t*>(ws + kWsInvalid);
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < Q; q += (long long)gridDim.x * blockDim.x)
        if (!range_query_valid(hole, board, n_players, ghost, known_opp, n_known, q)) atomicAdd(invalid, 1u);
}

// The query test of npk_equity_ranges_batch_adaptive (adaptive_init_kernel): 1 = valid, -1 = invalid.
struct RangeTest {
    const uint8_t *hole, *board, *n_players, *ghost, *known_opp;
    int n_known;
    __device__ int operator()(long long q) const
    {
        return range_query_valid(hole, board, n_players, ghost, known_opp, n_known, q) ? 1 : -1;
    }
};

int ranges_aborted()
{
    return fail(NPK_ERR_RANGE, "a draw needed more than 65536 attempts: no remaining hand satisfies the range (the reference "
                               "would loop forever); the counters are incomplete");
}

// The arguments both range entry points share, checked before the device is touched -- null pointers (`buffers`: the
// caller's outputs and workspace are all given), known opponents, the dealing mode, empty ranges -- and the launch fields
// that carry them: ghost cards, known hands, the two class masks.  `p` comes from fill_params.
int range_params(npk::EquityParams& p, const uint8_t* hole, const uint8_t* board, const uint8_t* n_players,
                 const uint8_t* ghost, const uint8_t* known_opp, int n_known, const uint64_t* opp_allowed,
                 const uint64_t* hero_allowed, bool buffers, int deal_mode)
{
    if ((!hole && !hero_allowed) || !board || !n_players || !buffers || !opp_allowed)
        return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (n_known < 0 || n_known > 9 || (n_known > 0 && !known_opp))
        return fail(NPK_ERR_INVALID_ARGUMENT, "n_known must be 0..9 and known_opp must be given when it is not 0");
    if (n_known > 0 && hero_allowed)
        return fail(NPK_ERR_INVALID_ARGUMENT, "a hero range together with known opponent hands is not supported (the reference "
                                              "draws the hero before it removes the known hands, montecarlo_python.py:132-163)");
    int rc = check_deal_mode(deal_mode);
    if (rc) return rc;
    const uint64_t top = (1ull << (169 - 128)) - 1ull;
    if (!(opp_allowed[0] | opp_allowed[1] | (opp_allowed[2] & top)))
        return fail(NPK_ERR_RANGE, "the opponent range is empty (the reference would never finish a draw)");
    if (hero_allowed && !(hero_allowed[0] | hero_allowed[1] | (hero_allowed[2] & top)))
        return fail(NPK_ERR_RANGE, "the hero range is empty (the reference would never finish a draw)");
    p.ghost = ghost;
    p.known_opp = n_known > 0 ? known_opp : nullptr; p.n_known = (uint32_t)n_known;
    for (int i = 0; i < 3; i++) {
        const uint64_t o = i == 2 ? opp_allowed[i] & top : opp_allowed[i];
        const uint64_t h = hero_allowed ? (i == 2 ? hero_allowed[i] & top : hero_allowed[i]) : 0;
        p.opp_mask[2 * i] = (uint32_t)o; p.opp_mask[2 * i + 1] = (uint32_t)(o >> 32);
        p.hero_mask[2 * i] = (uint32_t)h; p.hero_mask[2 * i + 1] = (uint32_t)(h >> 32);
    }
    p.hero_range = hero_allowed ? 1u : 0u;
    return NPK_OK;
}

// `passes` is a by-product of the reference's attempt loop: only the generic kernel, which plays that loop literally,
// can count it; everyone else gets the pair-list sampler (csrc/npk_ranges.cu), which redraws far less often
int launch_ranges(const DeviceState* ds, const npk::EquityParams& p, int deal_mode, long long items, cudaStream_t s)
{
    const int grid = grid_for(*ds, items, npk::kRefThreads / 32);
    const cudaError_t e = p.passes ? npk::launch_equity_ranges(deal_mode, p, grid, s)
                                   : npk::launch_equity_ranges_fast(deal_mode, p, grid, s);
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "equity_ranges_kernel launch");
}
}  // namespace

int npk_equity_ranges_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                            int64_t Q, int64_t trials, const uint64_t* opp_allowed, const uint64_t* hero_allowed,
                            uint64_t seed, int64_t trial_offset, int64_t query_offset, int deal_mode, uint32_t flags,
                            uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes, void* workspace,
                            void* stream)
{
    return npk_equity_ranges_known_batch(hole, board, n_players, ghost, nullptr, 0, Q, trials, opp_allowed, hero_allowed, seed,
                                         trial_offset, query_offset, deal_mode, flags, wins_strict, ties, win_types, passes,
                                         workspace, stream);
}

int npk_equity_ranges_known_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                                  const uint8_t* known_opp, int n_known, int64_t Q, int64_t trials,
                                  const uint64_t* opp_allowed, const uint64_t* hero_allowed, uint64_t seed,
                                  int64_t trial_offset, int64_t query_offset, int deal_mode, uint32_t flags,
                                  uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes,
                                  void* workspace, void* stream)
{
    DeviceState* ds;
    int rc = batch_start(&ds, Q, trials, trial_offset);
    if (rc) return rc == kEmptyBatch ? NPK_OK : rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    npk::EquityParams p;
    const long long chunks = fill_params(p, *ds, hero_allowed ? nullptr : hole, board, n_players, Q, trials, trial_offset,
                                         query_offset, seed, deal_mode, wins_strict, ties, win_types, passes,
                                         reinterpret_cast<uint32_t*>(ws + kWsAbort), 32);
    if ((rc = range_params(p, hole, board, n_players, ghost, known_opp, n_known, opp_allowed, hero_allowed,
                           wins_strict && ties && workspace, deal_mode)))
        return rc;
    if ((rc = clear_workspace(ws, s))) return rc;
    p.work_counter = reinterpret_cast<unsigned long long*>(ws + kWsCounters);

    const bool validate = (flags & NPK_FLAG_VALIDATE) != 0;
    if (validate) {
        const int cg = (int)std::min<long long>((Q + 255) / 256, 4 * ds->sm_count);
        validate_ranges_kernel<<<cg, 256, 0, s>>>(p.hole, board, n_players, ghost, p.known_opp, n_known, Q, ws);
        uint32_t bad = 0;
        if ((rc = read_word(ws + kWsInvalid, s, &bad, "query validation"))) return rc;
        if (bad) return fail(NPK_ERR_INVALID_CARDS, invalid_queries(bad, kRangeQueryCauses));
    }
    if ((rc = launch_ranges(ds, p, deal_mode, Q * chunks, s)) || !validate) return rc;
    uint32_t aborted = 0;
    if ((rc = read_word(ws + kWsAbort, s, &aborted, "equity_ranges_kernel"))) return rc;
    return aborted ? ranges_aborted() : NPK_OK;
}

int npk_equity_ranges_batch_adaptive(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                                     const uint8_t* known_opp, int n_known, int64_t Q, int64_t min_trials, int64_t max_trials,
                                     double max_stderr, const uint64_t* opp_allowed, const uint64_t* hero_allowed,
                                     uint64_t seed, int64_t query_offset, int deal_mode, uint32_t flags,
                                     uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes,
                                     uint64_t* trials, void* workspace, void* stream)
{
    int rc = check_rule(min_trials, max_trials, max_stderr);
    if (rc) return rc;
    DeviceState* ds;
    if ((rc = batch_start(&ds, Q, max_trials, 0))) return rc == kEmptyBatch ? NPK_OK : rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    npk::EquityParams p;
    fill_params(p, *ds, hero_allowed ? nullptr : hole, board, n_players, Q, min_trials, 0, query_offset, seed, deal_mode,
                wins_strict, ties, win_types, passes, reinterpret_cast<uint32_t*>(ws + kWsAbort), 32);
    if ((rc = range_params(p, hole, board, n_players, ghost, known_opp, n_known, opp_allowed, hero_allowed,
                           wins_strict && ties && trials && workspace, deal_mode)))
        return rc;
    int32_t* qindex = reinterpret_cast<int32_t*>(ws + kWsIndex);
    p.qindex = qindex;
    p.work_counter = reinterpret_cast<unsigned long long*>(ws + kWsCounters);
    const bool validate = (flags & NPK_FLAG_VALIDATE) != 0;

    // the abort flag is cleared once: a round that hits the attempt limit stops every later round at once
    if ((rc = clear_workspace(ws, s))) return rc;
    // a round runs the range kernel on the queries listed in qindex; there is no re-classification
    rc = run_adaptive(*ds, p, RangeTest{p.hole, board, n_players, ghost, p.known_opp, n_known}, Q, min_trials, max_trials,
                      max_stderr, trials, ws, qindex, 32, validate, "query validation", kRangeQueryCauses, "", s,
                      [&](const uint8_t*) {
                          const cudaError_t e = cudaMemsetAsync(p.work_counter, 0, sizeof(unsigned long long), s);
                          if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(workspace)");
                          uint32_t chunk, chunks;        // the grid: sized for every query, the most this round can have
                          npk::item_plan(Q, p.trials, ds->sm_count, 32, chunk, chunks);
                          return launch_ranges(ds, p, deal_mode, Q * (long long)chunks, s);
                      });
    if (rc || !validate) return rc;
    uint32_t aborted = 0;
    if ((rc = read_word(ws + kWsAbort, s, &aborted, "equity_ranges_kernel"))) return rc;
    return aborted ? ranges_aborted() : NPK_OK;
}

int npk_equity_ranges_host(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                           int64_t Q, int64_t trials, const uint64_t* opp_allowed, const uint64_t* hero_allowed,
                           uint64_t seed, int deal_mode, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types,
                           uint64_t* passes)
{
    return npk_equity_ranges_known_host(hole, board, n_players, ghost, nullptr, 0, Q, trials, opp_allowed, hero_allowed, seed,
                                        deal_mode, wins_strict, ties, win_types, passes);
}

int npk_equity_ranges_known_host(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                                 const uint8_t* known_opp, int n_known, int64_t Q, int64_t trials, const uint64_t* opp_allowed,
                                 const uint64_t* hero_allowed, uint64_t seed, int deal_mode, uint64_t* wins_strict,
                                 uint64_t* ties, uint64_t* win_types, uint64_t* passes)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (Q <= 0) return Q == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative Q");
    if ((!hole && !hero_allowed) || !board || !n_players || !wins_strict || !ties)
        return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    // device staging private to this call (ranges are the rare path; the plain path keeps its pinned staging)
    uint8_t* d_in = nullptr;
    uint64_t* d_out = nullptr;
    void* d_ws = nullptr;
    cudaError_t e;
    auto cleanup = [&]() { cudaFree(d_in); cudaFree(d_out); cudaFree(d_ws); };
    if (n_known < 0 || n_known > 9 || (n_known > 0 && !known_opp))
        return fail(NPK_ERR_INVALID_ARGUMENT, "n_known must be 0..9 and known_opp must be given when it is not 0");
    const int64_t per_q = 10 + 2 * n_known;                                       // bytes of input per query
    if ((e = cudaMalloc(&d_in, per_q * Q)) != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    if ((e = cudaMalloc(&d_out, 8 * 12 * Q)) != cudaSuccess) { cleanup(); return cuda_fail(e, "cudaMalloc"); }
    if ((e = cudaMalloc(&d_ws, npk_equity_workspace_bytes(Q))) != cudaSuccess) { cleanup(); return cuda_fail(e, "cudaMalloc"); }
    std::vector<uint8_t> h_in((size_t)(per_q * Q), 0xFF);
    if (hole) std::memcpy(h_in.data(), hole, 2 * Q);
    std::memcpy(h_in.data() + 2 * Q, board, 5 * Q);
    std::memcpy(h_in.data() + 7 * Q, n_players, Q);
    if (ghost) std::memcpy(h_in.data() + 8 * Q, ghost, 2 * Q);
    if (n_known > 0) std::memcpy(h_in.data() + 10 * Q, known_opp, (size_t)(2 * n_known) * Q);
    if ((e = cudaMemcpy(d_in, h_in.data(), per_q * Q, cudaMemcpyHostToDevice)) != cudaSuccess) { cleanup(); return cuda_fail(e, "H2D"); }
    if ((e = cudaMemset(d_out, 0, 8 * 12 * Q)) != cudaSuccess) { cleanup(); return cuda_fail(e, "memset"); }
    rc = npk_equity_ranges_known_batch(hole ? d_in : nullptr, d_in + 2 * Q, d_in + 7 * Q, ghost ? d_in + 8 * Q : nullptr,
                                       n_known > 0 ? d_in + 10 * Q : nullptr, n_known, Q, trials, opp_allowed, hero_allowed, seed,
                                       0, 0, deal_mode, NPK_FLAG_VALIDATE, d_out, d_out + Q, win_types ? d_out + 2 * Q : nullptr,
                                       passes ? d_out + 11 * Q : nullptr, d_ws, nullptr);
    if (rc) { cleanup(); return rc; }
    std::vector<uint64_t> h_out(12 * (size_t)Q);
    if ((e = cudaMemcpy(h_out.data(), d_out, 8 * 12 * Q, cudaMemcpyDeviceToHost)) != cudaSuccess) { cleanup(); return cuda_fail(e, "D2H"); }
    cleanup();
    std::memcpy(wins_strict, h_out.data(), 8 * Q);
    std::memcpy(ties, h_out.data() + Q, 8 * Q);
    if (win_types) std::memcpy(win_types, h_out.data() + 2 * Q, 8 * 9 * Q);
    if (passes) std::memcpy(passes, h_out.data() + 11 * Q, 8 * Q);
    return NPK_OK;
}

// ---- validation of the evaluator entry points (NPK_FLAG_VALIDATE) -----------------------------------------------------------
// rows of `len` card ids: every id < 52 and no id twice.  enum_mode: the row is hole[2] + board[5] (0xFF padding allowed
// at the end of the board only) and the shape must be one enum_kernel implements.
// mode 2 (npk_showdown_equity_batch): the same board rule, the optional dead mask of the row takes part in the duplicate test
// (a bit >= 52 is an invalid card), and the cards left to deal from -- one fewer in REFERENCE mode -- must cover the board.
__global__ void check_rows_kernel(const uint8_t* a, int len_a, const uint8_t* b, int len_b, const uint8_t* n_players,
                                  int maxp, int enum_mode, long long n, uint32_t* bad /*[2]: cards, shape*/,
                                  const uint64_t* dead, int deal_mode)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        unsigned long long mask = 0;
        int wrong = 0, known = 0;
        bool ended = false;
        int na = len_a;
        if (maxp > 0) {                                       // showdown: only the first n_players hands count
            const int np = n_players[i];
            if (np < 1 || np > maxp) { atomicAdd(&bad[1], 1u); continue; }
            na = 2 * np;
        }
        for (int k = 0; k < na; k++) {
            const int c = a[(long long)len_a * i + k];
            if (c >= 52) wrong = 1; else { wrong |= (int)(mask >> c & 1ull); mask |= 1ull << c; }
        }
        for (int k = 0; k < len_b; k++) {
            const int c = b[(long long)len_b * i + k];
            if (enum_mode && c == 0xFF) { ended = true; continue; }
            if (ended || c >= 52) { wrong = 1; continue; }
            wrong |= (int)(mask >> c & 1ull);
            mask |= 1ull << c;
            known++;
        }
        if (dead) {
            const unsigned long long d = dead[i];
            wrong |= (d >> 52) != 0 || (d & mask) != 0;
            mask |= d;
        }
        if (wrong) atomicAdd(&bad[0], 1u);
        if (enum_mode == 2) {
            const int missing = 5 - known;
            const int left = 52 - __popcll(mask & ((1ull << 52) - 1ull)) - (deal_mode == NPK_DEAL_REFERENCE && missing > 0 ? 1 : 0);
            if (left < missing) atomicAdd(&bad[1], 1u);
        } else if (enum_mode) {
            const int np = n_players[i];
            if (!(np == 2 || (np == 3 && known == 5))) atomicAdd(&bad[1], 1u);
        }
    }
}

namespace {
int check_rows(DeviceState* ds, const uint8_t* a, int len_a, const uint8_t* b, int len_b, const uint8_t* n_players, int maxp,
               int enum_mode, int64_t n, cudaStream_t s, const char* shape_msg, const uint64_t* dead = nullptr,
               int deal_mode = NPK_DEAL_UNIFORM)
{
    uint32_t* d_bad = nullptr;
    cudaError_t e = cudaMalloc(&d_bad, 8);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_bad, 0, 8, s);
    if (e != cudaSuccess) { cudaFree(d_bad); return cuda_fail(e, "validation scratch"); }
    const int grid = (int)std::min<long long>((n + 255) / 256, 8 * ds->sm_count);
    check_rows_kernel<<<grid, 256, 0, s>>>(a, len_a, b, len_b, n_players, maxp, enum_mode, n, d_bad, dead, deal_mode);
    uint32_t bad[2] = {0, 0};
    e = cudaMemcpyAsync(bad, d_bad, 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(d_bad);
    if (e != cudaSuccess) return cuda_fail(e, "validation");
    if (bad[0]) return fail(NPK_ERR_INVALID_CARDS, std::to_string(bad[0]) + " row(s) with a card id >= 52, a duplicate card or a gap in the board");
    if (bad[1]) return fail(NPK_ERR_INVALID_ARGUMENT, std::to_string(bad[1]) + shape_msg);
    return NPK_OK;
}
}  // namespace

int npk_rank7_batch(const uint8_t* cards, int64_t N, uint16_t* ranks, uint32_t flags, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (!cards || !ranks) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (flags & NPK_FLAG_VALIDATE) {
        rc = check_rows(ds, cards, 7, nullptr, 0, nullptr, 0, 0, N, static_cast<cudaStream_t>(stream), "");
        if (rc) return rc;
    }
    cudaError_t e = npk::launch_rank7(ds->t, cards, N, ranks, grid_for(*ds, (N + 127) / 128, npk::kRank7Threads / 32),
                                      static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "rank7_kernel launch");
}

int npk_rank7_colex(int64_t first, int64_t count, uint16_t* ranks, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (first < 0 || count < 0 || first + count > 133784560LL) return fail(NPK_ERR_INVALID_ARGUMENT, "range outside C(52,7)");
    if (count == 0) return NPK_OK;
    cudaError_t e = npk::launch_rank7_colex(ds->t, first, count, ranks, grid_for(*ds, (count + 31) / 32, npk::kAuxThreads / 32),
                                            static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "rank7_colex_kernel launch");
}

int npk_enum_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, uint64_t* win,
                   uint64_t* tie, uint64_t* lose, uint32_t flags, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (Q <= 0) return Q == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative Q");
    if (!hole || !board || !n_players || !win || !tie || !lose) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (flags & NPK_FLAG_VALIDATE) {
        rc = check_rows(ds, hole, 2, board, 5, n_players, 0, 1, Q, static_cast<cudaStream_t>(stream),
                        " quer(ies) of a shape the enumeration does not implement (two players with 0..5 known board cards, "
                        "or three players on a complete board)");
        if (rc) return rc;
    }
    npk::EnumParams p{};
    p.tables = ds->t; p.hole = hole; p.board = board; p.n_players = n_players; p.nq = Q;
    p.win = reinterpret_cast<unsigned long long*>(win);
    p.tie = reinterpret_cast<unsigned long long*>(tie);
    p.lose = reinterpret_cast<unsigned long long*>(lose);
    const int grid = (int)std::min<long long>(Q, ds->sm_count);
    cudaError_t e = npk::launch_enum(p, grid, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "enum_kernel launch");
}

int npk_showdown_batch(const uint8_t* holes, const uint8_t* n_players, const uint8_t* board, int64_t N, int maxp,
                       int32_t* winner, uint8_t* wtype, uint16_t* ranks, uint32_t flags, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (maxp < 1 || maxp > 23) return fail(NPK_ERR_INVALID_ARGUMENT, "maxp must be 1..23");
    if (!holes || !n_players || !board || !winner || !wtype) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (flags & NPK_FLAG_VALIDATE) {
        rc = check_rows(ds, holes, 2 * maxp, board, 5, n_players, maxp, 0, N, static_cast<cudaStream_t>(stream),
                        " table(s) with n_players outside 1..maxp");
        if (rc) return rc;
    }
    cudaError_t e = npk::launch_showdown(ds->t, holes, n_players, board, N, maxp, winner, wtype, ranks,
                                         grid_for(*ds, (N + 127) / 128, npk::kRank7Threads / 32), static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "showdown_kernel launch");
}

int64_t npk_showdown_equity_workspace_bytes(int64_t N) { return npk::showdown_equity_workspace_bytes(N); }

int npk_showdown_equity_batch(const uint8_t* holes, const uint8_t* n_players, const uint8_t* board, const uint64_t* dead,
                              int64_t N, int maxp, int deal_mode, uint32_t flags, uint64_t* win, uint64_t* tie, uint64_t* share,
                              uint64_t* completions, void* workspace, void* stream)
{
    DeviceState* ds;
    int rc = batch_start(&ds, N, 1, 0);
    if (rc) return rc == kEmptyBatch ? NPK_OK : rc;
    if (maxp < 1 || maxp > 10) return fail(NPK_ERR_INVALID_ARGUMENT, "maxp must be 1..10");
    if ((rc = check_deal_mode(deal_mode))) return rc;
    if (!holes || !n_players || !board || !win || !tie || !share || !completions || !workspace)
        return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (flags & NPK_FLAG_VALIDATE) {
        rc = check_rows(ds, holes, 2 * maxp, board, 5, n_players, maxp, 2, N, s,
                        " spot(s) with n_players outside 1..maxp or fewer cards left than missing board cards", dead, deal_mode);
        if (rc) return rc;
    }
    npk::ShowdownEquityParams p{};
    p.tables = ds->t;
    p.holes = holes; p.n_players = n_players; p.board = board; p.dead = dead;
    p.n = N; p.maxp = maxp; p.reference = deal_mode == NPK_DEAL_REFERENCE; p.sm_count = ds->sm_count;
    p.win = reinterpret_cast<unsigned long long*>(win);
    p.tie = reinterpret_cast<unsigned long long*>(tie);
    p.share = reinterpret_cast<unsigned long long*>(share);
    p.completions = reinterpret_cast<unsigned long long*>(completions);
    p.workspace = static_cast<uint8_t*>(workspace);
    cudaError_t e = npk::launch_showdown_equity(p, s);
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "showdown_equity_kernel launch");
}

// ---- vectorised HoldemTable (include/npk_holdem.h) ------------------------------------------------------------------------
int64_t npk_holdem_table_bytes(void) { return (int64_t)sizeof(NpkHoldemTable); }

int npk_holdem_init(void* tables, int64_t N, int n_players, double initial_stacks, double small_blind, double big_blind,
                    int max_raises_per_player_round, const uint8_t* autoplay, uint64_t seed, int64_t table_offset,
                    void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (!tables) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (n_players < 2 || n_players > NPK_MAX_SEATS) return fail(NPK_ERR_INVALID_ARGUMENT, "2..10 players per table");
    if (max_raises_per_player_round < 1 || max_raises_per_player_round > 100)
        return fail(NPK_ERR_INVALID_ARGUMENT, "max_raises_per_player_round must be 1..100");
    if (!(initial_stacks > 0) || !(small_blind > 0) || !(big_blind > 0))
        return fail(NPK_ERR_INVALID_ARGUMENT, "stacks and blinds must be positive");
    npk::HoldemInit cfg{};
    cfg.n_players = n_players; cfg.max_raises = max_raises_per_player_round;
    cfg.initial_stacks = initial_stacks; cfg.small_blind = small_blind; cfg.big_blind = big_blind;
    for (int i = 0; i < n_players; i++) cfg.autoplay[i] = autoplay ? autoplay[i] : 0;
    cudaError_t e = npk::launch_holdem_init(ds->t, tables, N, cfg, seed, table_offset, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "holdem_init_kernel launch");
}

int npk_holdem_reset_done(void* tables, int64_t N, uint64_t seed, int64_t table_offset, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    cudaError_t e = npk::launch_holdem_reset_done(ds->t, tables, N, seed, table_offset, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "holdem_reset_done_kernel launch");
}

int npk_holdem_step(void* tables, int64_t N, const int8_t* actions, double* rewards, uint64_t seed, int64_t table_offset,
                    int restart_finished, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (!tables || !actions) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    cudaError_t e = npk::launch_holdem_step(ds->t, tables, N, actions, rewards, seed, table_offset, restart_finished, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "holdem_step_kernel launch");
}

int npk_holdem_attach_stage_data(void* tables, int64_t N, double* stage_data, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (!tables) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    cudaError_t e = npk::launch_holdem_attach(tables, N, stage_data, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "holdem_attach_kernel launch");
}

int64_t npk_holdem_observation_size(int n_players) { return 22 + 51 * (int64_t)n_players; }

int npk_holdem_observe(const void* tables, int64_t N, const double* equity, double* obs, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (!tables || !obs) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    cudaError_t e = npk::launch_holdem_observe(tables, N, equity, obs, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "holdem_observe_kernel launch");
}

int npk_holdem_queries(const void* tables, int64_t N, uint8_t* hole, uint8_t* board, uint8_t* n_players, uint8_t* active,
                       void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (!tables || !hole || !board || !n_players) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    cudaError_t e = npk::launch_holdem_queries(tables, N, hole, board, n_players, active, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "holdem_queries_kernel launch");
}

int npk_holdem_decide(const void* tables, int64_t N, const uint64_t* wins, const uint64_t* ties, int64_t runs,
                      const double* equity, const uint8_t* agent_kind, const double* min_call_equity,
                      const double* min_bet_equity, uint64_t seed, int64_t decision_counter, int64_t table_offset,
                      int8_t* actions, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (N <= 0) return N == 0 ? NPK_OK : fail(NPK_ERR_INVALID_ARGUMENT, "negative N");
    if (!tables || !actions || !agent_kind) return fail(NPK_ERR_INVALID_ARGUMENT, "null pointer");
    if (!equity && (!wins || !ties || runs <= 0))
        return fail(NPK_ERR_INVALID_ARGUMENT, "pass either equity or wins + ties + runs");
    npk::HoldemAgents ag{};
    for (int i = 0; i < NPK_MAX_SEATS; i++) {
        ag.kind[i] = agent_kind[i];
        ag.min_call_equity[i] = min_call_equity ? min_call_equity[i] : 0.0;
        ag.min_bet_equity[i] = min_bet_equity ? min_bet_equity[i] : 0.0;
    }
    cudaError_t e = npk::launch_holdem_decide(ds->t, tables, N, wins, ties, runs, equity, ag, seed,
                                              (unsigned long long)decision_counter, table_offset, actions,
                                              static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "holdem_decide_kernel launch");
}

int npk_int_peak(int variant, int iters, double* thread_instr_per_s, float* ms_out)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    if (variant < 0 || variant > 2 || iters < 1) return fail(NPK_ERR_INVALID_ARGUMENT, "variant 0..2, iters >= 1");
    const int grid = ds->sm_count * 8;
    uint32_t* out = nullptr;
    cudaError_t e = cudaMalloc(&out, (size_t)grid * 256 * 4);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {           // first repetition is the warm-up
        cudaEventRecord(a, 0);
        e = npk::launch_int_peak(variant, out, iters, grid, 0);
        cudaEventRecord(b, 0);
        if (e == cudaSuccess) e = cudaEventSynchronize(b);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(out);
    if (e != cudaSuccess) return cuda_fail(e, "int_peak_kernel");
    const double per_iter = variant == 2 ? 256.0 : 128.0;
    if (thread_instr_per_s) *thread_instr_per_s = per_iter * iters * (double)grid * 256.0 / (best * 1e-3);
    if (ms_out) *ms_out = best;
    return NPK_OK;
}

int npk_philox_debug(const uint32_t* ctr, uint32_t k0, uint32_t k1, int n, uint32_t* out, void* stream)
{
    DeviceState* ds;
    int rc = current_state(&ds);
    if (rc) return rc;
    cudaError_t e = npk::launch_philox_debug(ctr, k0, k1, n, out, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? NPK_OK : cuda_fail(e, "philox_debug_kernel launch");
}

}  // extern "C"
