/*
 * npk.h -- C ABI of libnpk.so, the B200-native replacement for neuron_poker's Monte-Carlo equity hot path.
 *
 * This is the boundary a host-language binding targets (ctypes today; pybind11 / cgo / JNI would bind the same
 * symbols).  Plain pointers and sizes only, no torch or C++ types.  Unless a function says "host", every pointer is a
 * DEVICE pointer owned by the caller (e.g. torch tensors), nothing is allocated per call, and work is enqueued on the
 * caller's CUDA stream (`stream` is a cudaStream_t passed as void*, NULL = default stream) without synchronising.
 *
 * What each entry point replaces in the reference (paths relative to the reference repository root):
 *   npk_equity_batch    MonteCarlo.run_montecarlo's trial loop   tools/montecarlo_python.py:191-252 (dealing :121-189)
 *                       and montecarlo()                          tools/montecarlo_cpp/Montecarlo.cpp:240-259,
 *                       i.e. what get_equity (montecarlo_python.py:401-406) and the pybind11 export
 *                       pymontecarlo.montecarlo (tools/montecarlo_cpp/pymontecarlo.cpp:21-23) compute, batched
 *   npk_equity_host     the same, for HOST buffers: one blocking call = one (batch of) get_equity call(s)
 *   npk_equity_ranges_* the same loop with an opponent range, a hero range and ghost cards
 *                                                                 tools/montecarlo_python.py:24-112, :136-181, :206-208
 *   npk_rank7_batch     _calc_score ordering                      tools/hand_evaluator.py:27-119
 *   npk_showdown_batch  get_winner / eval_best_hand               tools/hand_evaluator.py:9-24 (used by gym_env/env.py:576-593)
 *   npk_enum_batch      no counterpart (the reference only samples); exact enumeration used for bit-exact checks
 *   npk_enum_dealer_batch  the exact value get_equity (:401-406) converges to, under the reference's dealer
 *   npk_showdown_equity_batch  run_montecarlo with every hand in player_card_list known (:132-163, ghost cards :206-208),
 *                       computed exactly (every board completion) and for every player, split pots included
 *   npk_exact_equity_batch  run_montecarlo with one or two unknown opponents beside known hands and ghost cards, computed
 *                       exactly under either dealer: the value it converges to
 *   npk_*_equity_win_types_batch  the same two, with run_montecarlo's winTypesDict (:226-231): the wins by hand type
 *
 * Cards are bytes: id = 4*rank + suit with ranks "23456789TJQKA" and suits "CDHS" -- the order of
 * MonteCarlo.create_card_deck (tools/montecarlo_python.py:114-119).  0xFF marks "no card" in board arrays.
 * Hand strength is a rank id in [0, 5034): the index of the reference's (score, card_ranks) tuple among all distinct
 * 7-card tuples in ascending order, so ids compare exactly like the reference's tuples (ties <=> equal ids).
 *
 * All functions return 0 on success or a negative NPK_ERR_* code; npk_last_error() gives a message (thread-local).
 */
#ifndef NPK_H
#define NPK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NPK_OK 0
#define NPK_ERR_NOT_INITIALIZED (-1)
#define NPK_ERR_INVALID_ARGUMENT (-2)
#define NPK_ERR_CUDA (-3)
#define NPK_ERR_TABLES (-4)
#define NPK_ERR_INVALID_CARDS (-5)   /* card id >= 52, duplicate cards, board with holes, players outside 1..10 */
#define NPK_ERR_RANGE (-6)           /* a range that no remaining card combination can satisfy */

/* dealing semantics */
#define NPK_DEAL_UNIFORM 0   /* uniform without replacement = the C++ sibling's std::shuffle (Montecarlo.cpp:293-312)   */
#define NPK_DEAL_REFERENCE 1 /* the Python reference's dealer incl. its bias (montecarlo_python.py:165-189, SURVEY A.2) */

/* flags for npk_equity_batch */
#define NPK_FLAG_VALIDATE 1u /* check card ids / duplicates on the device and sync once to report NPK_ERR_INVALID_CARDS */

#define NPK_NUM_CLASSES 5034
#define NPK_NUM_HAND_TYPES 9

/* Build the rank tables on the host and upload them to `device`; selects that device for later calls of this thread.
 * Idempotent per device.  Fails (NPK_ERR_CUDA) when no usable GPU is present: there is no CPU fallback. */
int npk_init(int device);
/* Build the tables on the host only (no GPU needed): enough for npk_get_tables / npk_host_rank7. */
int npk_init_host_tables(void);
/* Make an initialised `device` current for this thread's later calls (cheap; call it when switching GPUs). */
int npk_set_device(int device);
int npk_shutdown(void);
const char* npk_last_error(void);
int npk_sm_count(void);

/* Copies of the host-built tables (any pointer may be NULL).  value: row-displaced rank ids (n_value entries),
 * rowoff: 8192 row offsets, flush: 8192 entries by flush-suit rank mask, desc: 52 card descriptors,
 * type_start: 10 entries (first rank id of each hand type + end), class_keys: 5034 order keys. */
int npk_get_tables(uint16_t* value, int64_t* n_value, uint16_t* rowoff, uint16_t* flush, uint32_t* desc,
                   uint16_t* type_start, uint64_t* class_keys);
/* HOST: evaluate hands through the host copy of the tables (table self-check, not a compute path). */
int npk_host_rank7(const uint8_t* cards /*[n,7] host*/, int64_t n, uint16_t* ranks /*[n] host*/);

/* Bytes of device workspace npk_equity_batch needs for Q queries. */
int64_t npk_equity_workspace_bytes(int64_t Q);

/*
 * Monte-Carlo equity for Q queries x `trials` trials each.
 *   hole       [Q,2]  hero cards
 *   board      [Q,5]  known table cards first, 0xFF padding (0..5 known cards)
 *   n_players  [Q]    players still in the hand including the hero (1..10)
 *   uniform_players / uniform_known: if >= 0, EVERY query has that many players / known board cards and that shape's own
 *                     kernel runs; if either is < 0 the queries are classified on the device and one persistent kernel
 *                     handles all shapes.  Both are fully asynchronous unless NPK_FLAG_VALIDATE is set (one small
 *                     device->host read, the stream is synchronised once).
 *   seed, trial_offset, query_offset: trial t of query q uses the Philox4x32-10 stream with counter
 *                     (t + trial_offset, q + query_offset) and key = seed: results do not depend on how trials or
 *                     queries are partitioned over calls or GPUs.
 *                     Uniformity of the dealing: indices are drawn by multiply-shift, two per 32-bit Philox word (the low
 *                     product word of the first draw feeds the second).  The first index of a word deviates from uniform by
 *                     less than 2^-26 relative, the second by less than 2^-20 (its input takes 2^32/n equally spaced values,
 *                     n <= 50).  At 10^9 trials per query the induced error of an equity is below the 3-sigma sampling
 *                     error by two orders of magnitude; callers who need more trials than that per query should split
 *                     them over seeds.  No other approximation is made: the trial count is exact, nothing is truncated.
 *   wins_strict, ties [Q] u64, ACCUMULATED into (caller zeroes them): hero strictly best / tied for best.
 *                     reference equity = (wins_strict + ties) / trials  (ties count as wins, montecarlo_python.py:223-229)
 *   win_types  [Q,9] u64 or NULL: hand type of the hero whenever he wins or ties (winnerCardTypeList, :230-231, :244-248)
 *   passes     [Q] u64 or NULL: REFERENCE mode only, opponent draw attempts (`passes`, :167)
 *   workspace  npk_equity_workspace_bytes(Q) bytes of device memory, private to this call until it completes
 */
int npk_equity_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                     int uniform_players, int uniform_known, uint64_t seed, int64_t trial_offset, int64_t query_offset,
                     int deal_mode, uint32_t flags, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes,
                     void* workspace, void* stream);

/*
 * The same for MIXED batches, guaranteed free of any host round trip (self-play loops, CUDA-graph capture).  Mixed batches
 * always run as: classification by shape on the device (two small kernels) + ONE persistent kernel that handles every shape
 * (group after group through one work counter: the tables are staged once per CTA, there is one tail per call);
 * npk_equity_batch does the same when the uniform_* hints are negative.  `shape_mask` (bit (players-1)*6 +
 * known_board_cards) restricts the call to some shapes: queries of other shapes, and invalid queries, are left untouched
 * (their counters stay as they are).  Nothing is validated or reported by this call itself;
 * npk_equity_batch_status(workspace, stream, &invalid, &skipped) -- HOST pointers, synchronises `stream` -- returns how many
 * queries of the LAST call on that workspace were invalid / outside the mask.  Results are identical to npk_equity_batch.
 */
int npk_equity_batch_async(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                           uint64_t shape_mask, uint64_t seed, int64_t trial_offset, int64_t query_offset, int deal_mode,
                           uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes, void* workspace,
                           void* stream);
int npk_equity_batch_status(const void* workspace, void* stream, uint32_t* invalid, uint32_t* skipped);

/*
 * Monte-Carlo equity to a target PRECISION: every query runs until its standard error reaches `max_stderr`, checked at fixed
 * checkpoints, or until max_trials.  The checkpoints are the same for every query of the call:
 *     T_0 = min_trials,  T_{k+1} = min(2 T_k, max_trials),  up to max_trials       (1 <= min_trials <= max_trials)
 * After checkpoint T_k a query still running stops when var <= max_stderr * max_stderr, computed in IEEE double in this order
 * (every operation rounded to nearest, no fused multiply-add, so that a restatement in double arithmetic decides alike):
 *     x = wins_strict + ties          (the reference's equity numerator: ties count as wins)
 *     p = (x + 1) / (T_k + 2)         (add-one estimate: x = 0 or x = T_k does not give zero variance)
 *     var = p * (1 - p) / T_k
 * At max_trials every query stops.  The decision reads only the query's own counters, and trial t of query q is the same
 * Philox stream as in npk_equity_batch (trial_offset 0), so the outputs of a query are EXACTLY the counters npk_equity_batch
 * computes with trials = T_stop and the same seed and query_offset: they depend neither on the other queries of the batch nor
 * on how it is split over calls or GPUs (query sharding through query_offset).
 *   max_stderr  target standard error of the equity (wins_strict + ties) / trials; finite and > 0
 *   shape_mask  as npk_equity_batch_async: queries of other shapes are left out
 *   wins_strict, ties [Q], win_types [Q,9] or NULL, passes [Q] or NULL (REFERENCE mode): the counts of trials [0, T_stop)
 *   trials      [Q] u64: T_stop of every query
 * UNLIKE npk_equity_batch the call zeroes its outputs itself (the stopping rule reads them); invalid queries and queries outside
 * shape_mask are left at 0 with trials = 0.  With NPK_FLAG_VALIDATE an invalid query is an error (NPK_ERR_INVALID_CARDS,
 * reported after one small device->host read, before any trial runs).  Without it the call is asynchronous and free of host
 * round trips (CUDA-graph capturable): it runs in rounds, one per checkpoint, launched back to back -- classification of the
 * queries still active, the all-shapes kernel on trials [T_{k-1}, T_k), and a kernel that applies the rule, records trials of
 * the queries it retires and plans the next round's work items from the number left.  NPK_ERR_INVALID_ARGUMENT for a
 * max_stderr that is not finite or <= 0, min_trials < 1 or min_trials > max_trials is returned before the device is touched.
 *   workspace   npk_equity_adaptive_workspace_bytes(Q) bytes of device memory, private to this call until it completes
 */
int64_t npk_equity_adaptive_workspace_bytes(int64_t Q);
int npk_equity_batch_adaptive(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q,
                              int64_t min_trials, int64_t max_trials, double max_stderr, uint64_t shape_mask, uint64_t seed,
                              int64_t query_offset, int deal_mode, uint32_t flags, uint64_t* wins_strict, uint64_t* ties,
                              uint64_t* win_types, uint64_t* passes, uint64_t* trials, void* workspace, void* stream);

/*
 * Trial-sharded jobs (SURVEY 8e: one query spans several GPUs, e.g. 169 classes x 1,000,000 trials over 8 GPUs): the
 * count reduction is done by the Monte-Carlo kernel itself over NVLink-mapped peer memory; no NCCL call, no memset and no
 * pack kernel on the step path.  One process per GPU; the processes exchange 64-byte CUDA IPC handles once (any transport:
 * the Python host side uses torch.distributed.all_gather):
 *   npk_peer_create   allocates this rank's exchange buffer (2 parities x world slots x max_words u64) on the current
 *                     device and returns its IPC handle in handle[64] (HOST)
 *   npk_peer_connect  handles = all ranks' handles in rank order (HOST, world x 64 bytes): maps every peer's buffer
 *   npk_equity_batch_sharded  runs THIS rank's share of `trials_total` trials (rank r takes the r-th contiguous range) of
 *                     a uniform-shape batch and leaves in totals[2*Q] (device; wins [Q] then ties [Q]) the counters summed
 *                     over all ranks: the last warp of each rank's grid pushes the rank's counters into its slot on every
 *                     rank, publishes an epoch, waits for every rank's epoch and sums.  Every rank must make the same
 *                     sequence of calls; totals are bit-identical to the unsharded job.  Asynchronous on `stream`.
 *   npk_peer_error    HOST, synchronises: 1 if a peer's counters did not arrive within ~2 s in an earlier step
 */
int npk_peer_create(int rank, int world, int64_t max_words, void** group, uint8_t* handle);
int npk_peer_connect(void* group, const uint8_t* handles);
int npk_peer_destroy(void* group);
int npk_peer_error(void* group, int* error);
int npk_equity_batch_sharded(void* group, const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q,
                             int64_t trials_total, int players, int known, uint64_t seed, int64_t query_offset,
                             int deal_mode, uint64_t* totals, void* stream);

/* HOST buffers in, HOST buffers out: copies the queries to the device (pinned staging owned by the library), runs
 * npk_equity_batch with validation, copies the counters back and returns when they are valid.  wins/ties (and the
 * optional win_types [Q,9], passes [Q]) are overwritten. */
int npk_equity_host(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                    uint64_t seed, int deal_mode, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types,
                    uint64_t* passes);

/* HOST, pipelined: the two halves of npk_equity_host, so that a caller can keep several batches in flight -- the host-side
 * staging and the copies of batch i+1 overlap the kernel of batch i (each batch in flight owns pinned staging, device buffers
 * and a stream inside the library; kernels of consecutive batches fill each other's tails).
 *   npk_equity_host_submit  validates and stages the batch, enqueues H2D copy + kernels + D2H copy and returns a ticket >= 0
 *                           without waiting for the device (a negative NPK_ERR_* code on failure).  want bit 0: win types,
 *                           bit 1: passes.  At most NPK_HOST_SLOTS tickets per host thread may be outstanding.
 *   npk_equity_host_wait    blocks until that batch has finished and copies its counters out (same meaning as
 *                           npk_equity_host's outputs; win_types / passes may be NULL).  A ticket belongs to the thread that
 *                           submitted it and can be waited for once; tickets may be waited for in any order.
 * Results are bit-identical to npk_equity_host with the same arguments. */
#define NPK_HOST_SLOTS 4
int64_t npk_equity_host_submit(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int64_t trials,
                               uint64_t seed, int deal_mode, uint32_t want);
int npk_equity_host_wait(int64_t ticket, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes);

/* HOST, blocking: ONE query with as few arguments as a foreign-function call can have -- what the Python drop-in's get_equity
 * (montecarlo_python.py:401-406) calls.  packed = hole[0] | hole[1] << 8 | board[0] << 16 | ... | board[4] << 48 (card ids,
 * 0xFF = no card, known cards first); want bit 0: win types, bit 1: passes; out[12] (host) = wins, ties, win types[9],
 * passes.  One kernel launch, no copies, no stream synchronisation (the kernel publishes the result and the call's
 * sequence number in mapped host memory; the host spins on the number).  Validated like npk_equity_host. */
int npk_equity_one(uint64_t packed, int players, int64_t trials, uint64_t seed, int deal_mode, uint32_t want, uint64_t* out);

/* HOST.  Resident mode of the one-query path, per calling thread, opt-in.  npk_resident_start launches a persistent kernel on
 * `ctas` SMs (<= 0: all of them) that keeps the rank tables staged in shared memory and serves this thread's npk_equity_one /
 * one-query npk_equity_host calls (wins and ties only, fewer than 2^32 trials) out of a mailbox in mapped host memory: the call
 * posts the query (two 16-byte records), the kernel's polling thread picks it up over PCIe, the warps of all its CTAs run the
 * trials and the last CTA stores wins, ties and the call's sequence number back with one 16-byte store -- no kernel launch, no
 * CUDA call per query.  Results are bit-identical to the launch-per-call path (same Philox streams).
 * The kernel leaves on its own when no query has arrived for `idle_us` microseconds (<= 0: 200; at most 100,000) and is
 * started again by the next query, so it never holds the device for longer than that on its own; while it is resident, other
 * work submitted to the device waits for the SMs it occupies (libnpk's own host entry points of this thread stop it first).
 * One server per device and process: npk_resident_start fails (NPK_ERR_INVALID_ARGUMENT) while another thread runs one there.
 * npk_resident_stop makes the thread's calls launch a kernel per call again.  Both synchronise with the server only. */
int npk_resident_start(int ctas, int idle_us);
int npk_resident_stop(void);

/*
 * Monte-Carlo equity with RANGES (run_montecarlo's opponent_range / set-typed player cards / ghost_cards).
 * A starting-hand class is an unordered rank pair plus suitedness, numbered  suited hi*13+lo,  offsuit and pairs
 * lo*13+hi  (rank indices in "23456789TJQKA", hi >= lo); a range is a 169-bit mask in three uint64 words (HOST memory).
 *   opp_allowed   [3] host: classes every opponent's two cards must belong to
 *   hero_allowed  [3] host or NULL: if given, the hero's cards are drawn from this range every trial and `hole` is
 *                 ignored (may be NULL) -- the reference's "player_cards is a set" case
 *   ghost         [Q,2] device or NULL: cards removed from the deck before dealing (0xFF = none)
 * deal_mode NPK_DEAL_REFERENCE reproduces the reference dealer including the quirk that the range test looks at
 * deck[i1], deck[i2] before popping (montecarlo_python.py:173-179); NPK_DEAL_UNIFORM is the unbiased counterpart
 * (two distinct uniform cards, redrawn until the class is allowed).  passes [Q] counts the draw attempts of hero and
 * opponents in both modes -- a by-product of playing the reference's attempt loop literally, which only the generic kernel
 * does: with passes == NULL the call uses a sampler that lists the allowed pairs of every query's deck once and redraws
 * only on cards already dealt (same distribution of the dealt cards, several times faster; its Philox stream differs, so
 * the counters of the two variants agree statistically, not bit for bit).  One kernel handles every mix of player counts
 * and board sizes; the call is
 * asynchronous unless NPK_FLAG_VALIDATE is set, in which case the stream is synchronised and a range no remaining
 * hand can satisfy (one draw exceeded 65,536 attempts) is reported as NPK_ERR_RANGE.  Other arguments as above.
 */
int npk_equity_ranges_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                            int64_t Q, int64_t trials, const uint64_t* opp_allowed, const uint64_t* hero_allowed,
                            uint64_t seed, int64_t trial_offset, int64_t query_offset, int deal_mode, uint32_t flags,
                            uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes, void* workspace,
                            void* stream);
/* HOST buffers in and out, blocking, validated (NPK_ERR_INVALID_CARDS / NPK_ERR_RANGE): one run_montecarlo call with
 * ranges, or a batch of them sharing the same ranges.  hole may be NULL when hero_allowed is given; ghost [Q,2] or NULL. */
int npk_equity_ranges_host(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                           int64_t Q, int64_t trials, const uint64_t* opp_allowed, const uint64_t* hero_allowed,
                           uint64_t seed, int deal_mode, uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types,
                           uint64_t* passes);

/* The same two calls with opponents whose cards are KNOWN -- the reference's "several known hands in player_card_list" (its
 * provision for bots that share a table, tools/montecarlo_python.py:132-163): known_opp [Q, n_known, 2] (device for _batch,
 * host for _host) holds the hands of n_known (0..9) of the n_players - 1 opponents; their cards leave the deck before anything
 * is dealt and their hands take part in every showdown; the remaining n_players - 1 - n_known opponents are dealt from
 * opp_allowed as before.  The hero wins a trial when his hand is strictly best among all of them (ties are counted
 * separately, as everywhere).  Not combinable with hero_allowed: the reference draws a hero range BEFORE it removes the known
 * hands, so that case deals duplicate cards there.  n_known = 0 is npk_equity_ranges_batch / _host. */
int npk_equity_ranges_known_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                                  const uint8_t* known_opp, int n_known, int64_t Q, int64_t trials,
                                  const uint64_t* opp_allowed, const uint64_t* hero_allowed, uint64_t seed,
                                  int64_t trial_offset, int64_t query_offset, int deal_mode, uint32_t flags,
                                  uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes,
                                  void* workspace, void* stream);
/*
 * Monte-Carlo equity with ranges to a target PRECISION: npk_equity_batch_adaptive's contract (checkpoints T_0 = min_trials,
 * doubling, capped at max_trials; a query stops after checkpoint T_k when var <= max_stderr^2 with p = (wins_strict + ties +
 * 1) / (T_k + 2), var = p (1 - p) / T_k in round-to-nearest double without FMA; trials [Q] out) applied to
 * npk_equity_ranges_known_batch.  Arguments as there, minus trials and trial_offset: the counters of a query are EXACTLY those
 * npk_equity_ranges_known_batch computes with trials = T_stop, trial_offset = 0 and the same seed, query_offset, ranges,
 * ghost cards, known hands and sampler (the generic kernel when passes is given, the pair-list sampler when it is NULL).
 * The call zeroes its outputs; an invalid query is left at 0 with trials = 0, or with NPK_FLAG_VALIDATE is an error
 * (NPK_ERR_INVALID_CARDS) reported after one small device->host read, before any trial runs.  Each round runs the range
 * kernel on trials [T_{k-1}, T_k) of the queries still active, then a kernel that applies the rule, lists the queries left
 * and plans the next round's work items on the device.  A draw that needs more than 65,536 attempts stops that round and
 * every later one; with NPK_FLAG_VALIDATE it is reported as NPK_ERR_RANGE after the last round.  Without the flag the call is
 * asynchronous and free of host round trips (CUDA-graph capturable).  The rule's argument errors (NPK_ERR_INVALID_ARGUMENT)
 * are returned before the device is touched; the other argument errors are those of npk_equity_ranges_known_batch.
 *   workspace   npk_equity_adaptive_workspace_bytes(Q) bytes of device memory, private to this call until it completes
 */
int npk_equity_ranges_batch_adaptive(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                                     const uint8_t* known_opp, int n_known, int64_t Q, int64_t min_trials, int64_t max_trials,
                                     double max_stderr, const uint64_t* opp_allowed, const uint64_t* hero_allowed,
                                     uint64_t seed, int64_t query_offset, int deal_mode, uint32_t flags,
                                     uint64_t* wins_strict, uint64_t* ties, uint64_t* win_types, uint64_t* passes,
                                     uint64_t* trials, void* workspace, void* stream);
int npk_equity_ranges_known_host(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, const uint8_t* ghost,
                                 const uint8_t* known_opp, int n_known, int64_t Q, int64_t trials, const uint64_t* opp_allowed,
                                 const uint64_t* hero_allowed, uint64_t seed, int deal_mode, uint64_t* wins_strict,
                                 uint64_t* ties, uint64_t* win_types, uint64_t* passes);

/*
 * The evaluator entry points below take `flags`: with NPK_FLAG_VALIDATE the inputs are checked on the device first (every card
 * id < 52, no card twice in a row, n_players in range, a shape the kernel implements) and a violation is reported as
 * NPK_ERR_INVALID_CARDS / NPK_ERR_INVALID_ARGUMENT before anything is computed -- the stream is synchronised once.  Without
 * the flag the CALLER guarantees valid inputs: the kernels stay memory-safe for any byte values (ids are clamped to the
 * 64-slot descriptor table) but the results for invalid rows are meaningless.  The reference's error behaviour for this
 * case is a ValueError / RuntimeError("Card Type error!") (montecarlo_python.py:127-128, Montecarlo.cpp:233).
 */
/* rank ids of N 7-card hands */
int npk_rank7_batch(const uint8_t* cards /*[N,7]*/, int64_t N, uint16_t* ranks /*[N]*/, uint32_t flags, void* stream);
/* rank ids of the 7-card hands number first..first+count-1 in colexicographic order of C(52,7) = 133,784,560 hands
 * (c0<...<c6, index = sum C(c_i, i+1)) -- no input traffic; for the exhaustive parity check */
int npk_rank7_colex(int64_t first, int64_t count, uint16_t* ranks, void* stream);

/* Exact enumeration: heads-up (n_players = 2) with 0..5 known board cards, or three players on a complete board.
 * win/tie/lose [Q] u64 are overwritten: hero strictly best / tied / beaten, over all completions x opponent hands
 * (ordered pairs of disjoint hands for three players).  A query of any other shape gets 0 / 0 / 0 (NPK_FLAG_VALIDATE
 * reports it as NPK_ERR_INVALID_ARGUMENT instead). */
int npk_enum_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, uint64_t* win,
                   uint64_t* tie, uint64_t* lose, uint32_t flags, void* stream);

/* Exact enumeration under a chosen dealer: the shapes, validation and outputs of npk_enum_batch, which is this call with
 * NPK_DEAL_UNIFORM.  A deal_mode other than NPK_DEAL_UNIFORM / NPK_DEAL_REFERENCE is NPK_ERR_INVALID_ARGUMENT before the
 * device is touched.
 * NPK_DEAL_REFERENCE weights every deal by how often the reference's dealer (montecarlo_python.py:165-189) makes it, so
 * that the counts are integers.  R = the n unseen cards in ascending id order, m = missing board cards.
 *   opponent hand, slots a < b of R: weight w = 2 - [b == a + 1].  The dealer draws i1 in [0,n), i2 in [0,n-1), redraws
 *       while i1 == i2 and pops i1, then i2 from the shortened list: all (n-1)^2 accepted pairs are equally likely and the
 *       second card is never the successor of the first.  sum w = (n-1)^2.
 *   board: each card is pop(randint(0, len-1)), so the last card of the list is never dealt; every m-subset of R minus
 *       the opponents' cards minus its highest card has weight 1.
 *   three players (complete board): the ordered pair of hands has weight w(o1) * w(o2 | o1), with the adjacency of o2
 *       tested in R minus o1's cards.
 * Totals win + tie + lose: heads-up (n-1)^2 C(n-3, m); three players (n-1)^2 (n-3)^2.  The value get_equity converges to
 * with this dealer (ties count as wins) = (win + tie) / (win + tie + lose). */
int npk_enum_dealer_batch(const uint8_t* hole, const uint8_t* board, const uint8_t* n_players, int64_t Q, int deal_mode,
                          uint64_t* win, uint64_t* tie, uint64_t* lose, uint32_t flags, void* stream);

/* Batched showdown: holes [N,maxp,2], n_players [N] (1..maxp), board [N,5] complete.  winner [N] = first index among the
 * best hands (hand_evaluator.py:23 stable sort), wtype [N] = its hand type 0..8, ranks [N,maxp] or NULL. */
int npk_showdown_batch(const uint8_t* holes, const uint8_t* n_players, const uint8_t* board, int64_t N, int maxp,
                       int32_t* winner, uint8_t* wtype, uint16_t* ranks, uint32_t flags, void* stream);

/*
 * Exact showdown equity of KNOWN hands: for every spot, every completion of the board from the unseen cards is enumerated
 * once and scored for every player.
 *   holes [N,maxp,2]  the hands of players 0..n_players[s]-1 (maxp 1..10)   n_players [N]   board [N,5] 0xFF padding
 *   dead  [N] or NULL  one bit per card id removed from the deck (the reference's ghost cards)
 * The unseen cards U are the 52 minus hands, board and dead cards.  NPK_DEAL_UNIFORM enumerates every m-subset of U
 * (m = missing board cards); NPK_DEAL_REFERENCE leaves the highest id of U out when m >= 1 -- the reference deals a board
 * card with pop(randint(0, len-1)) from its id-ordered list (montecarlo_python.py:185-189) and so never deals the last one.
 * Per completion, with best = the highest rank id and k = the number of players holding it, each of those k players gets
 * win += (k == 1), tie += (k > 1), share += NPK_SHARE_UNIT / k.  Outputs (u64) are OVERWRITTEN; entries p >= n_players[s] are 0:
 *   win, tie, share [N,maxp]   completions [N] = C(|U'|, m)     sum_p share = NPK_SHARE_UNIT * completions
 *   split-pot equity = share / (NPK_SHARE_UNIT * completions); the reference's equity (ties count as wins) = (win + tie) / completions
 * workspace: npk_showdown_equity_workspace_bytes(N) bytes, private to the call until it completes.  Asynchronous and free of host
 * round trips (graph-capturable) unless NPK_FLAG_VALIDATE is set: NPK_ERR_INVALID_CARDS for an id >= 52, a card twice across
 * hands, board and dead mask, a gap in the board or a dead bit >= 52; NPK_ERR_INVALID_ARGUMENT for n_players outside 1..maxp or
 * fewer cards left than missing board cards.  Without the flag such a spot is memory-safe, and one with fewer cards left than
 * missing gets completions = 0 and zero counters.
 */
#define NPK_SHARE_UNIT 2520   /* lcm(1..10): a pot split k ways gives each of the k players 2520 / k */
int64_t npk_showdown_equity_workspace_bytes(int64_t N);
int npk_showdown_equity_batch(const uint8_t* holes, const uint8_t* n_players, const uint8_t* board, const uint64_t* dead,
                              int64_t N, int maxp, int deal_mode, uint32_t flags, uint64_t* win, uint64_t* tie, uint64_t* share,
                              uint64_t* completions, void* workspace, void* stream);
/* npk_showdown_equity_batch plus the hand types of the wins: win_types [N,maxp,9] (u64, OVERWRITTEN), where
 * win_types[s][p][t] = the completions in which player p holds the best rank, alone or tied, and that rank has hand type t
 * (0 high card .. 8 straight flush, as npk_showdown_batch's wtype).  sum_t win_types[s][p][t] = win[s][p] + tie[s][p].
 * Player 0's bins over completions are run_montecarlo's winTypesDict (montecarlo_python.py:226-231) when every hand is known.
 * Same arguments, validation, workspace and other outputs as npk_showdown_equity_batch, which is this call with
 * win_types = NULL. */
int npk_showdown_equity_win_types_batch(const uint8_t* holes, const uint8_t* n_players, const uint8_t* board,
                                        const uint64_t* dead, int64_t N, int maxp, int deal_mode, uint32_t flags, uint64_t* win,
                                        uint64_t* tie, uint64_t* share, uint64_t* completions, uint64_t* win_types,
                                        void* workspace, void* stream);

/*
 * Exact equity against one or two UNKNOWN opponents, with known opponent hands and dead cards: run_montecarlo with entries of
 * player_card_list beyond the hero known (montecarlo_python.py:132-163) and ghost cards (:206-208), without sampling.
 *   holes [N,maxk,2]  the hero, then the known opponents (maxk 1..8)   n_known [N] hands of `holes` in the spot, hero included
 *   n_random [N] unknown opponents k (1..2), n_known + k <= 10        board [N,5] 0xFF padding
 *   dead [N] or NULL  one bit per card id removed from the deck
 * R = the unseen cards (52 minus hands, board and dead cards) in ascending id order, n = |R|, m = missing board cards.  Outputs
 * (u64, OVERWRITTEN) are counts from the hero's side: win (hero strictly best of all players), tie (hero tied for best), lose.
 * (win + tie) / (win + tie + lose) is run_montecarlo's equity, where ties count as wins.
 *   NPK_DEAL_UNIFORM    every ordered tuple of disjoint unknown hands counts once, and so does every m-subset of what is left:
 *                       totals C(n,2) C(n-2,m) for k = 1, C(n,2) C(n-2,2) C(n-4,m) for k = 2.
 *   NPK_DEAL_REFERENCE  the weights of npk_enum_dealer_batch, applied to R (the list left after the known hands and the dead
 *                       cards): the first unknown hand, slots a < b, has weight 2 - [b == a + 1]; the second 2 - [every slot
 *                       strictly between a2 and b2 belongs to the first hand]; a completion holding x = max(R minus the unknown
 *                       hands' cards) counts 0.  Totals (n-1)^2 C(n-3,m) for k = 1, (n-1)^2 (n-3)^2 C(n-5,m) for k = 2.
 * With no known opponent and k = 1, or k = 2 on a complete board, the counts equal npk_enum_dealer_batch's in both modes.
 * A deal_mode other than NPK_DEAL_UNIFORM / NPK_DEAL_REFERENCE or maxk outside 1..8 is NPK_ERR_INVALID_ARGUMENT before the device
 * is touched.  workspace: npk_exact_equity_workspace_bytes(N) bytes, private to the call until it completes.  Asynchronous and
 * free of host round trips (graph-capturable) unless NPK_FLAG_VALIDATE is set: NPK_ERR_INVALID_CARDS for an id >= 52, a card twice
 * across hands, board and dead mask, a gap in the board or a dead bit >= 52; NPK_ERR_INVALID_ARGUMENT for n_known outside
 * 1..maxk, n_random outside 1..2, more than 10 players, or too few cards: n < 2k + m, or n < 2k + m + 1 under REFERENCE when
 * m >= 1.  Without the flag such a spot is memory-safe and gets zero counters.
 */
int64_t npk_exact_equity_workspace_bytes(int64_t N);
int npk_exact_equity_batch(const uint8_t* holes, const uint8_t* n_known, const uint8_t* n_random, const uint8_t* board,
                           const uint64_t* dead, int64_t N, int maxk, int deal_mode, uint32_t flags, uint64_t* win, uint64_t* tie,
                           uint64_t* lose, void* workspace, void* stream);
/* npk_exact_equity_batch plus the hand types of the hero's wins: win_types [N,9] (u64, OVERWRITTEN), where win_types[s][t] =
 * the weighted count (the same weights as win and tie, in either deal_mode) of the deals in which the hero is strictly best or
 * tied for best with a rank of hand type t (0 high card .. 8 straight flush).  sum_t win_types[s][t] = win[s] + tie[s].
 * win_types[s][t] / (win + tie + lose) is what run_montecarlo's winTypesDict (montecarlo_python.py:226-231) converges to.
 * Same arguments, validation, workspace and other outputs as npk_exact_equity_batch, which is this call with
 * win_types = NULL. */
int npk_exact_equity_win_types_batch(const uint8_t* holes, const uint8_t* n_known, const uint8_t* n_random, const uint8_t* board,
                                     const uint64_t* dead, int64_t N, int maxk, int deal_mode, uint32_t flags, uint64_t* win,
                                     uint64_t* tie, uint64_t* lose, uint64_t* win_types, void* workspace, void* stream);

/* Integer-issue microbenchmark on the current device (the roofline denominator of the Monte-Carlo kernel):
 * variant 0 = LOP3 chains (alu pipe), 1 = IMAD chains (fma pipe), 2 = both interleaved.  Reports executed
 * thread-instructions per second (best of 3 timed launches after a warm-up) and that launch's duration. */
int npk_int_peak(int variant, int iters, double* thread_instr_per_s, float* ms);

/* HOST, synchronises the device.  checked_build = 1 when the library was compiled with -DNPK_CHECKED (bounds checks on every
 * shared-memory gather, deck slot and decoded index of the kernels, deck-restored check after every work item: the stand-in
 * for compute-sanitizer where that tool is unavailable); first_failure = highest code of a failed check since npk_init
 * (0 = none; codes in csrc/npk_device.cuh).  Always 0 in the normal build. */
int npk_checked_status(int* checked_build, uint32_t* first_failure);

/* Philox4x32-10 known-answer hook: out[4i..4i+3] = philox(counter ctr[4i..4i+3], key (k0,k1)) */
int npk_philox_debug(const uint32_t* ctr, uint32_t k0, uint32_t k1, int n, uint32_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NPK_H */
