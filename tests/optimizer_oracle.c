/* C restatement of the Momentum / Adagrad / RMSProp updates of the PS data plane
 * (test infrastructure; loaded by tests/optimizer_oracle.py).
 *
 * TF r0.12 training_ops.cc functors, one IEEE-754 rounding per operation: compiled
 * with -ffp-contract=off, so a*b+c is never fused, the same value sequence as the
 * numpy restatement in optimizer_oracle.py and the CUDA kernels.  hyper[4] is the
 * shard header's {lr, b1, b2, eps}:
 *   MOMENTUM {lr, momentum}: a = a*mu + g; x = x - a*lr
 *   ADAGRAD  {lr, init}:     a = a + g*g; x = x - (g*lr) * (1/sqrt(a))
 *   RMSPROP  {lr, decay, momentum, eps}:
 *            ms = ms + (g*g - ms)*(1-decay); mom = mom*mu + (g*lr)/sqrt(ms+eps); x = x - mom
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

enum { OPT_MOMENTUM = 2, OPT_ADAGRAD = 3, OPT_RMSPROP = 4 };
enum { ASYNC_ORDERED = 0, SUM = 1, SYNC_MEAN = 2 };

int opt_oracle_apply(int opt, float *x, float *m, float *v, const float *g, size_t n,
                     const float *hyper)
{
    const float lr = hyper[0], b1 = hyper[1], b2 = hyper[2], eps = hyper[3];
    const float omb1 = 1.0f - b1;
    switch (opt) {
    case OPT_MOMENTUM:
        for (size_t i = 0; i < n; ++i) {
            m[i] = m[i] * b1 + g[i];
            x[i] = x[i] - m[i] * lr;
        }
        return 0;
    case OPT_ADAGRAD:
        for (size_t i = 0; i < n; ++i) {
            m[i] = m[i] + g[i] * g[i];
            x[i] = x[i] - (g[i] * lr) * (1.0f / sqrtf(m[i]));
        }
        return 0;
    case OPT_RMSPROP:
        for (size_t i = 0; i < n; ++i) {
            m[i] = m[i] + (g[i] * g[i] - m[i]) * omb1;
            v[i] = v[i] * b2 + (g[i] * lr) / sqrtf(m[i] + eps);
            x[i] = x[i] - v[i];
        }
        return 0;
    default:
        return -1;
    }
}

/* One round over W gradient slots (row stride `stride`).  ASYNC_ORDERED applies
 * slot after slot; SUM / SYNC_MEAN reduce ((g0 + g1) + g2) + ..., divide by W for
 * SYNC_MEAN, and apply once.  global_step advances per apply. */
int opt_oracle_round(int opt, float *x, float *m, float *v, const float *slots, size_t stride,
                     int W, size_t n, const float *hyper, int mode, float *scratch, int64_t *step)
{
    if (W < 1) return -1;
    if (mode == ASYNC_ORDERED) {
        for (int w = 0; w < W; ++w)
            if (opt_oracle_apply(opt, x, m, v, slots + (size_t)w * stride, n, hyper)) return -1;
        *step += W;
        return 0;
    }
    for (size_t i = 0; i < n; ++i) scratch[i] = slots[i];
    for (int w = 1; w < W; ++w)
        for (size_t i = 0; i < n; ++i) scratch[i] = scratch[i] + slots[(size_t)w * stride + i];
    if (mode == SYNC_MEAN)
        for (size_t i = 0; i < n; ++i) scratch[i] = scratch[i] / (float)W;
    if (opt_oracle_apply(opt, x, m, v, scratch, n, hyper)) return -1;
    *step += 1;
    return 0;
}

static long find_row(const int64_t *idx, long n, int64_t key)
{
    long lo = 0, hi = n;
    while (lo < hi) {
        long mid = (lo + hi) / 2;
        if (idx[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return (lo < n && idx[lo] == key) ? lo : -1;
}

/* Index-list round on an [n_rows, d] shard: a row pushed by several workers gets
 * ((g_w + g_w') + ...) in worker order, / W for mean, and ONE update; untouched
 * rows keep var and their state (TF's SparseApply* semantics).  -1 on an index
 * list that is not strictly ascending or leaves the matrix. */
int opt_oracle_rows_round(int opt, float *x, float *m, float *v, size_t n_rows, size_t d, int W,
                          const int64_t *const *idx, const float *const *rows, const size_t *k,
                          int mean, const float *hyper, float *scratch)
{
    for (int w = 0; w < W; ++w)
        for (size_t j = 0; j < k[w]; ++j) {
            if (idx[w][j] < 0 || (size_t)idx[w][j] >= n_rows) return -1;
            if (j > 0 && idx[w][j] <= idx[w][j - 1]) return -1;
        }
    for (int w = 0; w < W; ++w)
        for (size_t j = 0; j < k[w]; ++j) {
            const int64_t r = idx[w][j];
            int first = 1;
            for (int w2 = 0; w2 < w && first; ++w2)
                if (find_row(idx[w2], (long)k[w2], r) >= 0) first = 0;
            if (!first) continue;
            for (size_t e = 0; e < d; ++e) scratch[e] = rows[w][j * d + e];
            for (int w2 = w + 1; w2 < W; ++w2) {
                long p = find_row(idx[w2], (long)k[w2], r);
                if (p < 0) continue;
                for (size_t e = 0; e < d; ++e) scratch[e] = scratch[e] + rows[w2][(size_t)p * d + e];
            }
            if (mean)
                for (size_t e = 0; e < d; ++e) scratch[e] = scratch[e] / (float)W;
            const size_t at = (size_t)r * d;
            if (opt_oracle_apply(opt, x + at, m + at, v + at, scratch, d, hyper)) return -1;
        }
    return 0;
}
