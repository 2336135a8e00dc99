/* Exact equity against one or two unknown opponents, with known hands and dead cards, computed on the CPU two ways: the checkers
 * of libnpk's npk_exact_equity_batch.
 *
 * A spot: the hero's hand, nknown known opponent hands, k unknown opponents (1..2), nb board cards and a dead-card mask.  The
 * deck the dealer works on is the 52 ids in ascending order minus hero, known hands, board and dead cards: R, n cards.
 *
 * exact_equity_literal plays the reference's dealer (montecarlo_python.py:165-189) literally over every index sequence it can
 * draw.  Per unknown opponent: every i1 in [0,n), i2 in [0,n-1) with i1 != i2, then pop(i1) and pop(i2) from the shortened list.
 * Per missing board card: every j in [0,len-1), then pop(j).  Every accepted sequence is equally likely, so the counts are
 * sequence counts; the m! orders of the same m board cards score the same, and the board sequences are divided by m! at the end.
 *
 * exact_equity_weighted states the same expectation with the weights of include/npk.h (deal_mode 1): an unknown hand at slots
 * a < b of R has weight 2 - [b == a + 1], a second unknown hand 2 - [every slot strictly between a2 and b2 belongs to the first],
 * and the board is every m-subset of R minus the unknown hands' cards minus its highest card.  deal_mode 0 counts every ordered
 * tuple of disjoint unknown hands and every m-subset of what is left once.
 *
 * Both return out = {win, tie, lose} (hero strictly best of all players / tied for best / beaten) and 0, or -1 for a shape they
 * do not handle (k outside 1..2, nknown outside 0..7, nb outside 0..5, a card twice).  Hands are scored with `rank7` (the
 * oracle's oracle_rank7_fast, passed in by the caller). */
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

struct spot {
    rank7_fn rank7;
    const uint8_t *hero;
    const uint8_t *known;      /* [nknown][2] */
    int nknown, k;
};

static void score(const struct spot *sp, const uint8_t (*unk)[2], const uint8_t *table, int64_t w, int64_t *out)
{
    uint8_t h7[7] = {sp->hero[0], sp->hero[1], table[0], table[1], table[2], table[3], table[4]};
    const int hv = sp->rank7(h7);
    int best = -1;
    for (int o = 0; o < sp->nknown + sp->k; o++) {
        const uint8_t *h = o < sp->nknown ? sp->known + 2 * o : unk[o - sp->nknown];
        h7[0] = h[0]; h7[1] = h[1];
        const int v = sp->rank7(h7);
        if (v > best) best = v;
    }
    out[hv > best ? 0 : hv == best ? 1 : 2] += w;
}

/* R, the table's known part; -1 for a bad shape or a card twice */
static int setup(const struct spot *sp, const uint8_t *board, int nb, uint64_t dead, uint8_t *r, uint8_t *table)
{
    if (sp->k < 1 || sp->k > 2 || sp->nknown < 0 || sp->nknown > 7 || nb < 0 || nb > 5 || (dead >> 52)) return -1;
    uint64_t seen = dead;
    int cnt = __builtin_popcountll(dead);
    for (int i = 0; i < 2; i++) { seen |= 1ull << sp->hero[i]; cnt++; }
    for (int i = 0; i < 2 * sp->nknown; i++) { seen |= 1ull << sp->known[i]; cnt++; }
    for (int i = 0; i < nb; i++) { seen |= 1ull << board[i]; cnt++; table[i] = board[i]; }
    if (__builtin_popcountll(seen) != cnt) return -1;
    int n = 0;
    for (int c = 0; c < 52; c++) if (!(seen >> c & 1u)) r[n++] = (uint8_t)c;
    return n;
}

/* ---- the literal dealer ---------------------------------------------------------------------------------------------- */
static void literal_board(const struct spot *sp, const uint8_t *deck, int n, uint8_t *table, int nt, const uint8_t (*unk)[2],
                          int64_t *out)
{
    if (nt == 5) { score(sp, unk, table, 1, out); return; }
    for (int j = 0; j < n - 1; j++) {                        /* pop(randint(0, len(deck) - 1)) */
        uint8_t d[52];
        int m = n;
        memcpy(d, deck, (size_t)n);
        table[nt] = (uint8_t)pop(d, &m, j);
        literal_board(sp, d, m, table, nt + 1, unk, out);
    }
}

static void literal_opp(const struct spot *sp, const uint8_t *deck, int n, int o, uint8_t *table, int nt, uint8_t (*unk)[2],
                        int64_t *out)
{
    if (o == sp->k) { literal_board(sp, deck, n, table, nt, (const uint8_t (*)[2])unk, out); return; }
    for (int i1 = 0; i1 < n; i1++)
        for (int i2 = 0; i2 < n - 1; i2++) {
            if (i1 == i2) continue;                          /* redrawn */
            uint8_t d[52];
            int m = n;
            memcpy(d, deck, (size_t)n);
            unk[o][0] = (uint8_t)pop(d, &m, i1);
            unk[o][1] = (uint8_t)pop(d, &m, i2);
            literal_opp(sp, d, m, o + 1, table, nt, unk, out);
        }
}

int exact_equity_literal(rank7_fn rank7, const uint8_t *hero, const uint8_t *known, int nknown, int k, const uint8_t *board,
                         int nb, uint64_t dead, int64_t *out)
{
    const struct spot sp = {rank7, hero, known, nknown, k};
    uint8_t deck[52], table[5], unk[2][2];
    const int n = setup(&sp, board, nb, dead, deck, table);
    if (n < 0) return -1;
    out[0] = out[1] = out[2] = 0;
    literal_opp(&sp, deck, n, 0, table, nb, unk, out);
    int64_t orders = 1;
    for (int i = 2; i <= 5 - nb; i++) orders *= i;
    for (int j = 0; j < 3; j++) {
        if (out[j] % orders) return -2;                      /* cannot happen: every board set comes in m! orders */
        out[j] /= orders;
    }
    return 0;
}

/* ---- the weights -------------------------------------------------------------------------------------------------------- */
/* every m-subset of the usable slots of R (ascending), completing the table */
static void weighted_board(const struct spot *sp, const uint8_t *r, const int *usable, int nu, int start, uint8_t *table, int nt,
                           const uint8_t (*unk)[2], int64_t w, int64_t *out)
{
    if (nt == 5) { score(sp, unk, table, w, out); return; }
    for (int i = start; i < nu; i++) {
        table[nt] = r[usable[i]];
        weighted_board(sp, r, usable, nu, i + 1, table, nt + 1, unk, w, out);
    }
}

int exact_equity_weighted(rank7_fn rank7, const uint8_t *hero, const uint8_t *known, int nknown, int k, const uint8_t *board,
                          int nb, uint64_t dead, int deal_mode, int64_t *out)
{
    const struct spot sp = {rank7, hero, known, nknown, k};
    uint8_t r[52], table[5], unk[2][2];
    const int n = setup(&sp, board, nb, dead, r, table);
    if (n < 0) return -1;
    const int ref = deal_mode == 1;
    out[0] = out[1] = out[2] = 0;
    for (int a1 = 0; a1 < n; a1++)
        for (int b1 = a1 + 1; b1 < n; b1++) {
            const int64_t w1 = ref ? 2 - (b1 == a1 + 1) : 1;
            unk[0][0] = r[a1]; unk[0][1] = r[b1];
            /* second unknown hand: every pair a2 < b2 of R minus {a1, b1}, each ordered pair of hands once (the first hand in the
             * outer loop); with one unknown opponent these two loops make one pass */
            for (int a2 = 0; a2 < (k == 2 ? n : 1); a2++)
                for (int b2 = k == 2 ? a2 + 1 : 0; b2 < (k == 2 ? n : 1); b2++) {
                    int64_t w = w1;
                    if (k == 2) {
                        if (a2 == a1 || a2 == b1 || b2 == a1 || b2 == b1) continue;
                        int gap = 0;                         /* slots of R - {a1, b1} strictly between a2 and b2 */
                        for (int s = a2 + 1; s < b2; s++) gap += s != a1 && s != b1;
                        if (ref) w *= 2 - (gap == 0);
                        unk[1][0] = r[a2]; unk[1][1] = r[b2];
                    }
                    /* the board: R minus every unknown card, minus its highest card under the reference's dealer */
                    int usable[52], nu = 0;
                    for (int s = 0; s < n; s++) {
                        const int held = s == a1 || s == b1 || (k == 2 && (s == a2 || s == b2));
                        if (!held) usable[nu++] = s;
                    }
                    if (ref && nb < 5) nu--;
                    weighted_board(&sp, r, usable, nu, 0, table, nb, (const uint8_t (*)[2])unk, w, out);
                }
        }
    return 0;
}
