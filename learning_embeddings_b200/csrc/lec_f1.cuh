// The best-F1 row of EmbeddingMetrics.calculate_metrics, 'val' phase (order_embeddings.py:272-287 = oe.py:380-395),
// shared by the sweep over sorted energies (lec_metrics.cu) and the streaming reconstruction check (lec_recon.cu).
#pragma once
#include <stdint.h>

namespace lec {

__host__ __device__ __forceinline__ bool f1_better(double fa, int64_t ia, double fb, int64_t ib) {
    // higher F1 wins; ties go to the lower threshold (np.argmax returns the first maximum)
    return fa > fb || (fa == fb && ia < ib);
}

// metrics of threshold t with cp = #{positives E <= t} and cn = #{negatives E > t}: the reference's expression tree in
// fp64.  NaN energies (the zero label row of the reference's off-by-one, SURVEY F9) satisfy neither E <= t nor E > t:
// they count in n_pos / n_neg only, and a NaN threshold has cp = cn = 0.
__device__ __forceinline__ void f1_row(float t, int64_t cp, int64_t cn, int64_t n_pos, int64_t n_neg, double* row) {
    if (t != t) { cp = 0; cn = 0; }
    const double acc = (double)(cp + cn) / (double)(n_pos + n_neg);
    const double prec = (double)cp / (double)(cp + (n_neg - cn));   // 0/0 -> NaN (the reference raises ZeroDivisionError)
    const double rec = (double)cp / (double)n_pos;
    const double f1 = (prec + rec == 0.0) ? 0.0 : (2.0 * prec * rec) / (prec + rec);
    row[0] = f1; row[1] = (double)t; row[2] = acc; row[3] = prec; row[4] = rec; row[5] = (double)cp; row[6] = (double)cn;
}

}  // namespace lec
