// npk_kernels.h -- parameter blocks and host-callable launchers of the kernels in npk_kernels.cu
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "npk_device.cuh"

namespace npk {

constexpr int kEquityMaxThreads = 512; // up to 16 warps per CTA, one CTA per SM (shared memory decides, see uniform_warps)
constexpr size_t kMaxDynamicSmem = 232448;   // 227 KB opt-in limit per CTA on sm_100
constexpr int kShapeGroups = 60;       // shapes of a mixed batch: group = opponents * 6 + known board cards
constexpr int kMixedThreads = 480;     // persistent all-shapes kernel: 15 warps, decks sized for 50 unseen cards
constexpr int kRefThreads = 512;       // generic range kernel
constexpr int kAuxThreads = 512;
constexpr int kRank7Threads = 1024;    // rank7 is latency-bound at one CTA per SM: 32 warps hide twice as much

// State of the one-query fast path.  The counters live in device memory and are handed to the kernel as wins/ties/...;
// the LAST warp to finish copies them into `host` (pinned, mapped host memory), zeroes them and the work counter for the
// next call, and publishes `done`.
struct SingleResult {             // in mapped host memory
    unsigned long long wins, ties, win_types[9], passes;
    unsigned long long seq;       // number of the call these values belong to: written last, the host spins on it
};
struct SingleCall {               // in device memory
    unsigned long long wins, ties, win_types[9], passes;
    unsigned long long work_counter;
    unsigned int ticket;
    unsigned int abort_flag[16];
    SingleResult* host;
};

// Resident mode of the one-query path (opt-in, npk_resident_start): a persistent kernel keeps the tables staged on its SMs and
// serves get_equity calls out of a mailbox in mapped host memory -- no kernel launch per call.  Thread 0 of CTA 0 polls the
// mailbox over PCIe (two 16-byte reads in flight per poll) and re-publishes a new request as two 16-byte records in device
// memory, stamped with a command number; thread 0 of every other CTA spins on those records in L2.  The warps take the
// request's work items by static striding (spread over the CTAs first), add their counts into shared memory, and every CTA
// hands {wins, ties, 1} to ONE packed 64-bit atomic: the CTA whose addition completes the count knows the totals from the
// value the atomic returned and stores wins, ties and the call's sequence number to the host in one 16-byte store.
// The kernel leaves on its own once no request has arrived for `idle_cycles` (or the host raises `stop`).
struct __align__(128) ResidentMailbox {       // mapped host memory
    // host -> device: two 16-byte records, both stamped with the call's sequence number (a request is taken when both match)
    struct __align__(16) ReqA { unsigned int seq, trials, packed_lo, packed_hi; } a;   // packed_hi: board bytes 2..4, players << 24, reference dealer << 31
    struct __align__(16) ReqB { unsigned int seq, seed_lo, seed_hi, stop; } b;         // stop: launch id the host wants to leave
    unsigned long long pad0_[12];
    // device -> host
    struct __align__(16) Done { unsigned int wins, ties; unsigned long long seq; } done;
    unsigned long long exited;                // launch id of the last server that left (written after its final poll)
    unsigned long long pad1_[13];
};
struct __align__(128) ResidentState {         // device memory
    uint4 a;                                  // {command number, trials, packed_lo, packed_hi}
    uint4 b;                                  // {command number, seed_lo, seed_hi, host sequence number (0 = leave)}
    unsigned long long acc[2];                // per command parity: wins | ties << 28 | CTAs done << 56
};
constexpr long long kResidentMaxTrials = 1ll << 28;      // counters are packed 28 + 28 + 8 bits

// Trial-sharded jobs (one query spans several GPUs, SURVEY 8e): the count reduction is part of the Monte-Carlo kernel.
// Every rank owns one PeerBuf in its own HBM, mapped into every other rank's address space (CUDA IPC over NVLink):
//   flags[parity][r]          epoch of the last block rank r has pushed into slots[parity][r] of THIS buffer
//   slots[parity][r][words]   rank r's counters for the step of that parity
// The last warp of a rank's kernel pushes its counters into its slot on every rank, publishes the epoch, waits for all
// ranks' epochs in its own buffer, sums the slots into `totals` and resets the local counters for the next step: no
// memset, no pack kernel, no NCCL call on the step path.  Two parities are enough: a rank cannot start step s+2 before
// every rank has pushed step s+1, which each does only after it has finished reading step s.
constexpr int kMaxPeers = 16;
struct PeerCall {                    // in device memory, written once when the group is connected
    unsigned long long* flags[kMaxPeers];     // flags region of rank r's buffer: [2][kMaxPeers]
    unsigned long long* slots[kMaxPeers];     // slots region of rank r's buffer: [2][world][stride]
    unsigned long long* acc;                  // local counters [stride] (wins [Q], ties [Q])
    unsigned long long work_counter;
    unsigned int ticket;
    unsigned int error;                       // 1: a peer's epoch did not arrive in time
    uint32_t world, rank, stride;
};

struct EquityParams {
    DeviceTables tables;
    const uint8_t* hole;          // [Q,2] card ids
    const uint8_t* board;         // [Q,5] card ids, 0xFF = not dealt yet (known cards first)
    const uint8_t* n_players;     // [Q]
    const int32_t* qindex;        // all-shapes kernel only (npk_mixed.cu): query ids sorted by shape
    const uint32_t* group;        // all-shapes kernel only: queries per shape group[0..59], their first qindex slot
                                  // group[64..123]
    long long nq;                 // queries 0..nq-1 of the per-shape and range kernels
    long long trials;             // trials per query in this launch
    long long trial_offset;       // first trial number (sharding a query over launches / GPUs)
    uint32_t query_offset;        // added to the query number in the Philox counter (sharding queries over GPUs)
    uint32_t seed_lo, seed_hi;
    uint32_t chunk, chunks;       // trials per work item, items per query (the last one may be shorter)
    uint32_t reference_dealer;    // 0: uniform dealing (K1), 1: the Python reference's dealer (K1')
    unsigned long long* work_counter;
    unsigned long long* wins;     // [Q] hero strictly best
    unsigned long long* ties;     // [Q] hero ties for best
    unsigned long long* win_types;// [Q,9] or null: hand type of the hero whenever he wins or ties
    unsigned long long* passes;   // [Q] or null: reference-mode draw attempts (montecarlo_python.py:167)
    // ---- single blocking call (npk_equity_host with one query): no copies, no memsets ----
    uint64_t inline_query;        // hole[2] | board[5] << 16 (bytes), used when `hole` is null
    SingleCall* single;           // device scratch + mapped host result block, or null
    unsigned long long single_seq;
    // ---- trial-sharded job: reduce the counters over the ranks inside the kernel ----
    PeerCall* peer;               // or null
    unsigned long long peer_epoch;
    unsigned long long* peer_totals;   // [peer_words] reduced counters (this rank's output)
    uint32_t peer_words;
    // ---- ranges (equity_ranges_kernel only) ----
    uint32_t opp_mask[6];         // 169-bit mask of the starting-hand classes an opponent may hold
    uint32_t hero_mask[6];        // the same for the hero when hero_range != 0
    uint32_t hero_range;          // 1: the hero is drawn from hero_mask every trial (`hole` is not read)
    const uint8_t* ghost;         // [Q,2] cards removed from the deck before dealing (0xFF = none), or null
    const uint8_t* known_opp;     // [Q,n_known,2] opponents whose cards are known (the reference's several known hands in
                                  // player_card_list, montecarlo_python.py:132-163), or null
    uint32_t n_known;             // how many of the n_players - 1 opponents those are
    uint32_t* abort_flag;         // raised when one draw needs more than kMaxRangeAttempts attempts
    // ---- adaptive calls (npk_equity_batch_adaptive, npk_equity_ranges_batch_adaptive): {chunk, chunks, queries} of this
    // round, written on the device by the kernel that retired the previous round's queries; the all-shapes and range kernels
    // read them instead of chunk / chunks (and the range kernels read `queries` instead of nq, the query slots from qindex)
    // when non-null
    const uint32_t* plan;
};

// Work items of a Monte-Carlo launch: (query, chunk of trials).  Items hold up to 2,048 trials (64 per lane: the per-item
// set-up -- query load, deck initialisation, reduction -- is then a few per cent of the work) but at least eight per warp;
// small jobs are cut finer so that a single query still spreads over the whole chip (a lone get_equity call of 10,000 trials
// becomes 157 one-iteration items).  A finer-grained tail (the last eighth of every query in items an eighth of the size,
// handed out last) was measured in round 2 and lost 1.5 % on cfg3: the warps left over in the last round of items run faster,
// because the SM is throughput-bound, so the tail costs about 1 %, less than the extra item set-ups.
// The host plans a launch from its query count; an adaptive call's later rounds are planned on the device from the number of
// queries still running.  The plan changes no result: a trial's outcome depends only on (seed, query, trial number).
__host__ __device__ inline void item_plan(long long queries, long long trials, int sm_count, int lanes_worth, uint32_t& chunk,
                                          uint32_t& chunks)
{
    const long long warps = (long long)sm_count * 16;
    long long c = (queries * trials) / (8 * warps);
    c = (c + lanes_worth - 1) / lanes_worth * lanes_worth;      // a warp iteration covers 64 trials (a pair per lane)
    if (c < lanes_worth) c = lanes_worth;
    if (c > 2048) c = 2048;
    if (trials <= 0) { chunk = 1; chunks = 0; return; }
    if (trials <= c) { chunk = (uint32_t)trials; chunks = 1; return; }
    chunk = (uint32_t)c;
    chunks = (uint32_t)((trials + c - 1) / c);
}

constexpr uint32_t kMaxRangeAttempts = 1u << 16;

struct EnumParams {
    DeviceTables tables;
    const uint8_t* hole;
    const uint8_t* board;
    const uint8_t* n_players;
    long long nq;
    unsigned long long* win;
    unsigned long long* tie;
    unsigned long long* lose;
};

// exact showdown equity of known hands (npk_showdown_equity.cu)
struct ShowdownEquityParams {
    DeviceTables tables;
    const uint8_t* holes;         // [n, maxp, 2]
    const uint8_t* n_players;     // [n]
    const uint8_t* board;         // [n, 5], 0xFF padding
    const uint64_t* dead;         // [n] masks, or null
    long long n;
    int maxp;
    int reference;                // 1: NPK_DEAL_REFERENCE (the highest unseen id is never dealt)
    int sm_count;
    unsigned long long* win;      // [n, maxp]
    unsigned long long* tie;      // [n, maxp]
    unsigned long long* share;    // [n, maxp]
    unsigned long long* completions;   // [n]
    uint8_t* workspace;           // showdown_equity_workspace_bytes(n)
};

size_t aux_smem(const DeviceTables& t);
long long showdown_equity_workspace_bytes(long long n);
cudaError_t launch_showdown_equity(const ShowdownEquityParams& p, cudaStream_t s);
cudaError_t launch_equity_uniform(int nopp, int nb, const EquityParams& p, long long items, int sm_count, cudaStream_t s);
cudaError_t launch_equity_mixed(const EquityParams& p, int sm_count, cudaStream_t s);
cudaError_t launch_equity_resident(const DeviceTables& t, ResidentState* st, ResidentMailbox* mb, unsigned long long launch_id,
                                   unsigned int last_seq, long long idle_cycles, int ctas, cudaStream_t s);
cudaError_t launch_equity_oneshot(const DeviceTables& t, ResidentState* st, ResidentMailbox* mb, uint4 a, uint4 b,
                                  unsigned int parity, int sm_count, cudaStream_t s);
cudaError_t launch_equity_ranges(int deal_mode, const EquityParams& p, int grid, cudaStream_t s);
cudaError_t launch_equity_ranges_fast(int deal_mode, const EquityParams& p, int grid, cudaStream_t s);
cudaError_t launch_rank7(const DeviceTables& t, const uint8_t* cards, long long n, uint16_t* out, int grid, cudaStream_t s);
cudaError_t launch_rank7_colex(const DeviceTables& t, long long first, long long count, uint16_t* out, int grid, cudaStream_t s);
cudaError_t launch_enum(const EnumParams& p, int grid, cudaStream_t s);
cudaError_t launch_showdown(const DeviceTables& t, const uint8_t* holes, const uint8_t* n_players, const uint8_t* board,
                            long long n, int maxp, int32_t* winner, uint8_t* wtype, uint16_t* ranks, int grid, cudaStream_t s);
cudaError_t launch_int_peak(int variant, uint32_t* out, int iters, int grid, cudaStream_t s);
cudaError_t launch_philox_debug(const uint32_t* ctr, uint32_t k0, uint32_t k1, int n, uint32_t* out, cudaStream_t s);

}  // namespace npk
