/* The pairs of the striped-parity census (ps_make_pair of oracle/parasail_striped.c, which is compiled in here
 * unchanged), exported so that the device tests can replay exactly the pairs the CPU fuzz checks.
 * TEST INFRASTRUCTURE ONLY: built by tests/pair_census.py into a temporary directory. */
#include "../../oracle/parasail_striped.c"

/* pairs first .. first+n-1 of stream `seed`, concatenated: q[qoff[k] .. qoff[k+1]), t[toff[k] .. toff[k+1]);
 * q must hold n * qmax bytes and t n * tmax bytes */
int pc_gen_pairs(uint64_t seed, int64_t first, int64_t n, int qmax, int tmax, char *q, int64_t *qoff, char *t,
                 int64_t *toff)
{
    if (qmax < 8 || qmax > 500 || tmax < 8 || tmax > 2000 || n < 0) return -1;
    qoff[0] = toff[0] = 0;
    for (int64_t k = 0; k < n; ++k) {
        int ql, tl;
        ps_make_pair(seed, first + k, qmax, tmax, q + qoff[k], &ql, t + toff[k], &tl);
        qoff[k + 1] = qoff[k] + ql;
        toff[k + 1] = toff[k] + tl;
    }
    return 0;
}
