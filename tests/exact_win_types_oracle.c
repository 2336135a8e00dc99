/* Win-type histograms of the exact enumerations, computed on the CPU: the checkers of libnpk's npk_exact_equity_win_types_batch
 * and npk_showdown_equity_win_types_batch.
 *
 * exact_wt_literal and exact_wt_weighted are the two enumerators of tests/exact_equity_oracle.c (the reference's dealer replayed
 * over every index sequence it can draw, and the weights of include/npk.h), with the hero's hand type binned beside the counts:
 * out[0..2] = {win, tie, lose} and out[3 + t] = the part of win + tie in which the hero's rank has hand type t.  A rank id's type
 * is the number of type_start[1..8] (libnpk's table: first rank id of each type) at or below it.
 *
 * showdown_wt enumerates every board completion of a spot whose hands are all known (the highest unseen id left out under the
 * reference's dealer) and gives, per player p, win[p], tie[p] and bins[9 p + t] = completions in which p holds the best rank,
 * alone or tied, with hand type t.
 *
 * All return 0, or -1 for a shape they do not handle (k outside 1..2, nknown outside 0..7, nb outside 0..5, a card twice,
 * players outside 1..10).  Hands are scored with `rank7` (the oracle's oracle_rank7_fast, passed in by the caller). */
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

static int hand_type(const uint16_t *type_start, int v)
{
    int t = 0;
    for (int i = 1; i < 9; i++) t += v >= type_start[i];
    return t;
}

struct spot {
    rank7_fn rank7;
    const uint16_t *type_start;
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
    if (hv >= best) out[3 + hand_type(sp->type_start, hv)] += w;
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

int exact_wt_literal(rank7_fn rank7, const uint16_t *type_start, const uint8_t *hero, const uint8_t *known, int nknown, int k,
                     const uint8_t *board, int nb, uint64_t dead, int64_t *out)
{
    const struct spot sp = {rank7, type_start, hero, known, nknown, k};
    uint8_t deck[52], table[5], unk[2][2];
    const int n = setup(&sp, board, nb, dead, deck, table);
    if (n < 0) return -1;
    memset(out, 0, 12 * sizeof(int64_t));
    literal_opp(&sp, deck, n, 0, table, nb, unk, out);
    int64_t orders = 1;
    for (int i = 2; i <= 5 - nb; i++) orders *= i;
    for (int j = 0; j < 12; j++) {
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

int exact_wt_weighted(rank7_fn rank7, const uint16_t *type_start, const uint8_t *hero, const uint8_t *known, int nknown, int k,
                      const uint8_t *board, int nb, uint64_t dead, int deal_mode, int64_t *out)
{
    const struct spot sp = {rank7, type_start, hero, known, nknown, k};
    uint8_t r[52], table[5], unk[2][2];
    const int n = setup(&sp, board, nb, dead, r, table);
    if (n < 0) return -1;
    const int ref = deal_mode == 1;
    memset(out, 0, 12 * sizeof(int64_t));
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

/* ---- every hand known ----------------------------------------------------------------------------------------------- */
struct known_spot {
    rank7_fn rank7;
    const uint16_t *type_start;
    const uint8_t *holes;      /* [players][2] */
    int players;
    int64_t *win, *tie, *bins;
};

static void showdown_board(const struct known_spot *ks, const uint8_t *u, int nu, int start, uint8_t *table, int nt)
{
    if (nt == 5) {
        int v[10], best = -1, cnt = 0;
        for (int q = 0; q < ks->players; q++) {
            const uint8_t h7[7] = {ks->holes[2 * q], ks->holes[2 * q + 1], table[0], table[1], table[2], table[3], table[4]};
            v[q] = ks->rank7(h7);
            if (v[q] > best) best = v[q];
        }
        for (int q = 0; q < ks->players; q++) cnt += v[q] == best;
        const int t = hand_type(ks->type_start, best);
        for (int q = 0; q < ks->players; q++) {
            if (v[q] != best) continue;
            if (cnt == 1) ks->win[q]++; else ks->tie[q]++;
            ks->bins[9 * q + t]++;
        }
        return;
    }
    for (int i = start; i < nu; i++) {
        table[nt] = u[i];
        showdown_board(ks, u, nu, i + 1, table, nt + 1);
    }
}

int showdown_wt(rank7_fn rank7, const uint16_t *type_start, const uint8_t *holes, int players, const uint8_t *board, int nb,
                uint64_t dead, int deal_mode, int64_t *win, int64_t *tie, int64_t *bins)
{
    if (players < 1 || players > 10 || nb < 0 || nb > 5 || (dead >> 52)) return -1;
    uint64_t seen = dead;
    int cnt = __builtin_popcountll(dead);
    uint8_t table[5], u[52];
    for (int i = 0; i < 2 * players; i++) { seen |= 1ull << holes[i]; cnt++; }
    for (int i = 0; i < nb; i++) { seen |= 1ull << board[i]; cnt++; table[i] = board[i]; }
    if (__builtin_popcountll(seen) != cnt) return -1;
    int nu = 0;
    for (int c = 0; c < 52; c++) if (!(seen >> c & 1u)) u[nu++] = (uint8_t)c;
    if (deal_mode == 1 && nb < 5) nu--;                      /* the reference's dealer never deals the last unseen card */
    memset(win, 0, (size_t)players * sizeof(int64_t));
    memset(tie, 0, (size_t)players * sizeof(int64_t));
    memset(bins, 0, (size_t)players * 9 * sizeof(int64_t));
    const struct known_spot ks = {rank7, type_start, holes, players, win, tie, bins};
    showdown_board(&ks, u, nu, 0, table, nb);
    return 0;
}
