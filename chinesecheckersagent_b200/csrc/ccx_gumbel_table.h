/* ccx_gumbel_table.h — the sequential-halving schedule of the Gumbel search's root (mctx, seq_halving.py,
 * get_sequence_of_considered_visits), host-side and C-compatible.
 *
 * out[k], k < S, is the visit count an edge must have to be chosen at root simulation k when m edges are considered and
 * S simulations are made.  Visits of the considered edges stay equal to each other within a phase, so a phase of e extra
 * visits over c edges appends e runs of c copies of the common count. */
#pragma once
#include <stdint.h>

static inline void ccx_considered_visits(int32_t m, int32_t S, int32_t *out)
{
    if (m <= 1) {
        for (int32_t k = 0; k < S; k++) out[k] = k;
        return;
    }
    int32_t log2max = 0;
    while (((int64_t)1 << log2max) < m) log2max++;           /* ceil(log2(m)) */
    int32_t len = 0, visits = 0, considered = m;
    while (len < S) {
        int32_t extra = S / (log2max * considered);          /* int(S / (log2max * considered)) for positive integers */
        if (extra < 1) extra = 1;
        for (int32_t e = 0; e < extra; e++) {
            for (int32_t i = 0; i < considered && len < S; i++) out[len++] = visits;
            visits++;
        }
        considered = considered / 2 > 2 ? considered / 2 : 2;
    }
}
