/* The exact expectation of the reference's dealer, computed on the CPU two ways: the checkers of libnpk's weighted enumeration
 * (npk_enum_dealer_batch with NPK_DEAL_REFERENCE).
 *
 * enum_reference_literal plays the dealer of montecarlo_python.py:165-189 literally over every index sequence it can draw.
 * The deck is the 52 ids in ascending order; the known board and the hero's cards are popped first.  Per opponent: every
 * i1 in [0,n), i2 in [0,n-1) with i1 != i2, then pop(i1) and pop(i2) from the shortened list.  Per missing board card: every
 * j in [0,len-1), then pop(j).  Every accepted sequence is equally likely, so the counts are sequence counts; the m! orders of
 * the same m board cards score the same, and the board sequences are divided by m! at the end.
 *
 * enum_reference_weighted states the same expectation with the weights of include/npk.h: an opponent hand (slots a < b of
 * the unseen cards R) has weight 2 - [b == a + 1], the board is every m-subset of R minus the opponents' cards minus its
 * highest card, and a second opponent's adjacency is tested in R minus the first opponent's cards.
 *
 * Both return out = {win, tie, lose} (hero strictly best / tied for best / beaten) and 0, or -1 for a shape they do not
 * handle (players 2..3, nb 0..5).  Hands are scored with `rank7` (the oracle's oracle_rank7_fast, passed in by the caller). */
#include <stdint.h>
#include <string.h>

typedef int (*rank7_fn)(const uint8_t *cards);

static int pop(uint8_t *deck, int *n, int idx)
{
    int v = deck[idx];
    memmove(deck + idx, deck + idx + 1, (size_t)(*n - idx - 1));
    (*n)--;
    return v;
}

static void score(rank7_fn rank7, const uint8_t *hero, const uint8_t (*opp)[2], int nopp, const uint8_t *table, int64_t w,
                  int64_t *out)
{
    uint8_t h7[7] = {hero[0], hero[1], table[0], table[1], table[2], table[3], table[4]};
    const int hv = rank7(h7);
    int best = -1;
    for (int o = 0; o < nopp; o++) {
        h7[0] = opp[o][0]; h7[1] = opp[o][1];
        const int v = rank7(h7);
        if (v > best) best = v;
    }
    out[hv > best ? 0 : hv == best ? 1 : 2] += w;
}

/* ---- the literal dealer ---------------------------------------------------------------------------------------------- */
static void literal_board(rank7_fn rank7, const uint8_t *deck, int n, uint8_t *table, int nt, const uint8_t *hero,
                          const uint8_t (*opp)[2], int nopp, int64_t *out)
{
    if (nt == 5) { score(rank7, hero, opp, nopp, table, 1, out); return; }
    for (int j = 0; j < n - 1; j++) {                        /* pop(randint(0, len(deck) - 1)) */
        uint8_t d[52];
        int m = n;
        memcpy(d, deck, (size_t)n);
        table[nt] = (uint8_t)pop(d, &m, j);
        literal_board(rank7, d, m, table, nt + 1, hero, opp, nopp, out);
    }
}

static void literal_opp(rank7_fn rank7, const uint8_t *deck, int n, int o, uint8_t *table, int nt, const uint8_t *hero,
                        uint8_t (*opp)[2], int nopp, int64_t *out)
{
    if (o == nopp) { literal_board(rank7, deck, n, table, nt, hero, (const uint8_t (*)[2])opp, nopp, out); return; }
    for (int i1 = 0; i1 < n; i1++)
        for (int i2 = 0; i2 < n - 1; i2++) {
            if (i1 == i2) continue;                          /* redrawn */
            uint8_t d[52];
            int m = n;
            memcpy(d, deck, (size_t)n);
            opp[o][0] = (uint8_t)pop(d, &m, i1);
            opp[o][1] = (uint8_t)pop(d, &m, i2);
            literal_opp(rank7, d, m, o + 1, table, nt, hero, opp, nopp, out);
        }
}

int enum_reference_literal(rank7_fn rank7, const uint8_t *hero, const uint8_t *board, int nb, int players, int64_t *out)
{
    if (players < 2 || players > 3 || nb < 0 || nb > 5) return -1;
    uint8_t deck[52], table[5], opp[2][2];
    int n = 52;
    for (int i = 0; i < 52; i++) deck[i] = (uint8_t)i;
    for (int i = 0; i < nb; i++) {
        int ix = 0;
        while (ix < n && deck[ix] != board[i]) ix++;
        if (ix == n) return -1;
        table[i] = (uint8_t)pop(deck, &n, ix);
    }
    for (int k = 0; k < 2; k++) {
        int ix = 0;
        while (ix < n && deck[ix] != hero[k]) ix++;
        if (ix == n) return -1;
        pop(deck, &n, ix);
    }
    out[0] = out[1] = out[2] = 0;
    literal_opp(rank7, deck, n, 0, table, nb, hero, opp, players - 1, out);
    int64_t orders = 1;
    for (int i = 2; i <= 5 - nb; i++) orders *= i;
    for (int k = 0; k < 3; k++) {
        if (out[k] % orders) return -2;                      /* cannot happen: every board set comes in m! orders */
        out[k] /= orders;
    }
    return 0;
}

/* ---- the weights -------------------------------------------------------------------------------------------------------- */
/* every m-subset of the usable slots of R (ascending), completing the table */
static void weighted_board(rank7_fn rank7, const uint8_t *r, const int *usable, int nu, int start, uint8_t *table, int nt,
                           const uint8_t *hero, const uint8_t (*opp)[2], int nopp, int64_t w, int64_t *out)
{
    if (nt == 5) { score(rank7, hero, opp, nopp, table, w, out); return; }
    for (int i = start; i < nu; i++) {
        table[nt] = r[usable[i]];
        weighted_board(rank7, r, usable, nu, i + 1, table, nt + 1, hero, opp, nopp, w, out);
    }
}

int enum_reference_weighted(rank7_fn rank7, const uint8_t *hero, const uint8_t *board, int nb, int players, int64_t *out)
{
    if (players < 2 || players > 3 || nb < 0 || nb > 5) return -1;
    uint64_t seen = (1ull << hero[0]) | (1ull << hero[1]);
    for (int i = 0; i < nb; i++) seen |= 1ull << board[i];
    uint8_t r[52], table[5], opp[2][2];
    int n = 0;
    for (int c = 0; c < 52; c++) if (!(seen >> c & 1u)) r[n++] = (uint8_t)c;
    for (int i = 0; i < nb; i++) table[i] = board[i];
    out[0] = out[1] = out[2] = 0;
    const int nopp = players - 1;
    for (int a1 = 0; a1 < n; a1++)
        for (int b1 = a1 + 1; b1 < n; b1++) {
            const int64_t w1 = 2 - (b1 == a1 + 1);
            opp[0][0] = r[a1]; opp[0][1] = r[b1];
            /* second opponent (three players): unordered slots a2 < b2 of R minus {a1, b1}; each ordered pair of hands is
             * visited once, the first hand in the outer loop.  Heads-up, these two loops make one pass. */
            const int n2 = nopp == 2 ? n : 1;
            for (int a2 = 0; a2 < n2; a2++)
                for (int b2 = nopp == 2 ? a2 + 1 : 0; b2 < (nopp == 2 ? n : 1); b2++) {
                    int64_t w = w1;
                    if (nopp == 2) {
                        if (a2 == a1 || a2 == b1 || b2 == a1 || b2 == b1) continue;
                        int gap = 0;                         /* slots of R - {a1, b1} strictly between a2 and b2 */
                        for (int s = a2 + 1; s < b2; s++) gap += s != a1 && s != b1;
                        w *= 2 - (gap == 0);
                        opp[1][0] = r[a2]; opp[1][1] = r[b2];
                    }
                    /* the board: R minus every opponent card minus the highest remaining slot */
                    int usable[52], nu = 0;
                    for (int s = 0; s < n; s++) {
                        const int held = s == a1 || s == b1 || (nopp == 2 && (s == a2 || s == b2));
                        if (!held) usable[nu++] = s;
                    }
                    if (nb < 5) nu--;
                    weighted_board(rank7, r, usable, nu, 0, table, nb, hero, (const uint8_t (*)[2])opp, nopp, w, out);
                }
        }
    return 0;
}
