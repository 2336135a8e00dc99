/* Exact showdown equity of KNOWN hands, enumerated literally on the CPU: the checker of libnpk's npk_showdown_equity_batch.
 *
 * Every m-subset (m = 5 - nb) of the unseen cards U' is one completion of the board, scored for each of the P players with
 * `rank7` (the oracle's oracle_rank7_fast, passed in by the caller).  U' = the 52 cards minus holes[2P], board[nb] and the dead
 * mask; deal_mode 1 (the reference's dealer, which never deals the last card of its id-ordered list, montecarlo_python.py:185-189)
 * removes the highest id of U' when m >= 1.  Per completion, the k players holding the best rank id get win += (k == 1),
 * tie += (k > 1), share += 2520 / k.
 * out = win[P] tie[P] share[P] completions.  Returns -1 for P outside 1..10, nb outside 0..5 or fewer cards than missing. */
#include <stdint.h>

typedef int (*rank7_fn)(const uint8_t *cards);

static void showdown_rec(rank7_fn rank7, const uint8_t *u, int nu, int start, uint8_t *table, int nt, const uint8_t *holes,
                         int P, int64_t *out)
{
    if (nt == 5) {
        int v[10], best = -1, k = 0;
        for (int p = 0; p < P; p++) {
            uint8_t h7[7] = {holes[2 * p], holes[2 * p + 1], table[0], table[1], table[2], table[3], table[4]};
            v[p] = rank7(h7);
            if (v[p] > best) best = v[p];
        }
        for (int p = 0; p < P; p++) k += v[p] == best;
        for (int p = 0; p < P; p++) {
            if (v[p] != best) continue;
            if (k == 1) out[p]++; else out[P + p]++;
            out[2 * P + p] += 2520 / k;
        }
        out[3 * P]++;
        return;
    }
    for (int i = start; i < nu; i++) {
        table[nt] = u[i];
        showdown_rec(rank7, u, nu, i + 1, table, nt + 1, holes, P, out);
    }
}

int showdown_equity(rank7_fn rank7, const uint8_t *holes, int P, const uint8_t *board, int nb, uint64_t dead_mask,
                    int deal_mode, int64_t *out)
{
    if (P < 1 || P > 10 || nb < 0 || nb > 5) return -1;
    uint64_t seen = dead_mask;
    for (int i = 0; i < 2 * P; i++) seen |= 1ull << holes[i];
    for (int i = 0; i < nb; i++) seen |= 1ull << board[i];
    uint8_t u[52], table[5];
    int nu = 0;
    for (int c = 0; c < 52; c++) if (!(seen >> c & 1u)) u[nu++] = (uint8_t)c;
    if (deal_mode == 1 && nb < 5 && nu > 0) nu--;
    for (int i = 0; i < 3 * P + 1; i++) out[i] = 0;
    if (nu < 5 - nb) return -1;
    for (int i = 0; i < nb; i++) table[i] = board[i];
    showdown_rec(rank7, u, nu, 0, table, nb, holes, P, out);
    return 0;
}
