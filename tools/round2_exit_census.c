/* Round-2 dominance exit census (tools/round2_exit_census.py drives it).
 *
 * Full round-2 DP of every read against left + motif^T (map-ont in doubled units, the low bit of a word = "started
 * after the left anchor"), one column at a time.  From column `start` on, the DP column is kept every P columns
 * (P = the kernel's period: a multiple of 16 and of |motif|) and compared with the column P later; the first column
 * that is <= the kept one in every word (H, E1, E2 of every row) ends the sweep: nothing to its right can beat the
 * record (DESIGN.md section 4.9).  Input on stdin:
 *     R <left> <motif> <T> <n_reads> <start_offset>      then n_reads lines, one read each
 * where start_offset is added to |left| + (length of the read) to give the first checked column (the host's rule).
 * Output: one line per region, "cells <n> skipped <n> exit_cols <sum of exit columns - |left|> reads <n>".
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static int code(char c) { switch (c) { case 'A': return 0; case 'C': return 1; case 'G': return 2; case 'T': return 3; } return 4; }
enum { kMatch = 2, kMismatch = 4, kAmbiguous = 1, kOE1 = 6, kOE2 = 25, kExt1 = 2, kExt2 = 1 };
typedef int64_t w_t;
static inline w_t mx(w_t a, w_t b) { return a > b ? a : b; }
static int gcd(int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; }

int main(void) {
    static char L[1 << 20], mot[4096], core[1 << 20];
    int T, n, off;
    while (scanf(" R %s %s %d %d %d", L, mot, &T, &n, &off) == 5) {
        const int nl = (int)strlen(L), m = (int)strlen(mot), tlen = nl + m * T, P = 16 * m / gcd(16, m);
        char* tpl = malloc(tlen + 1);
        memcpy(tpl, L, nl);
        for (int k = 0; k < T; ++k) memcpy(tpl + nl + k * m, mot, m);
        long long cells = 0, skipped = 0, exit_cols = 0;
        for (int r = 0; r < n; ++r) {
            if (scanf(" %s", core) != 1) return 1;
            const int q = (int)strlen(core);
            w_t *H = malloc(sizeof(w_t) * (q + 1)), *E1 = malloc(sizeof(w_t) * (q + 1)), *E2 = malloc(sizeof(w_t) * (q + 1));
            w_t *kH = malloc(sizeof(w_t) * (q + 1)), *kE1 = malloc(sizeof(w_t) * (q + 1)), *kE2 = malloc(sizeof(w_t) * (q + 1));
            for (int i = 0; i <= q; ++i) { H[i] = 0; E1[i] = -2 * kOE1; E2[i] = -2 * kOE2; }
            int start = nl + q + off;
            if (start < nl + 1) start = nl + 1;
            start = (start + 15) / 16 * 16;
            int kept = 0, exit_at = tlen;
            for (int j = 1; j <= tlen; ++j) {       /* column j (1-based) of the template */
                const int tc = code(tpl[j - 1]);
                const w_t fresh = j > nl ? 1 : 0;
                w_t hd = H[0], f1 = fresh - 2 * kOE1, f2 = fresh - 2 * kOE2;
                H[0] = fresh;
                for (int i = 1; i <= q; ++i) {
                    const int qc = code(core[i - 1]);
                    const int s = qc > 3 ? -kAmbiguous : tc == qc ? kMatch : -kMismatch;
                    const w_t e1 = E1[i], e2 = E2[i];
                    w_t h = mx(mx(hd + 2 * s, fresh), mx(mx(e1, e2), mx(f1, f2)));
                    hd = H[i];
                    H[i] = h;
                    E1[i] = mx(h - 2 * kOE1, e1 - 2 * kExt1);
                    E2[i] = mx(h - 2 * kOE2, e2 - 2 * kExt2);
                    f1 = mx(h - 2 * kOE1, f1 - 2 * kExt1);
                    f2 = mx(h - 2 * kOE2, f2 - 2 * kExt2);
                }
                if (j >= start && (j - start) % P == 0) {
                    if (kept) {
                        int dom = 1;
                        for (int i = 0; i <= q && dom; ++i) dom = H[i] <= kH[i] && E1[i] <= kE1[i] && E2[i] <= kE2[i];
                        if (dom) { exit_at = j; break; }
                    }
                    memcpy(kH, H, sizeof(w_t) * (q + 1)); memcpy(kE1, E1, sizeof(w_t) * (q + 1)); memcpy(kE2, E2, sizeof(w_t) * (q + 1));
                    kept = 1;
                }
            }
            cells += (long long)q * tlen;
            skipped += (long long)q * (tlen - exit_at);
            exit_cols += exit_at - nl;
            free(H); free(E1); free(E2); free(kH); free(kE1); free(kE2);
        }
        printf("cells %lld skipped %lld exit_cols %lld reads %d\n", cells, skipped, exit_cols, n);
        fflush(stdout);
        free(tpl);
    }
    return 0;
}
