// Host side of the fast scoring kernel: builds the work-unit table (label segments x image groups) and
// dispatches to the per-geometry translation units (lec_score_fast_{hyp,euc,oe,poincare,lorentz}.cu).
#include "lec_score_fast_impl.cuh"

namespace lec {

int score_fast_hyp(FastArgs& a, cudaStream_t st);
int score_fast_euc(FastArgs& a, cudaStream_t st);
int score_fast_oe(FastArgs& a, cudaStream_t st);
int score_fast_poincare(FastArgs& a, cudaStream_t st);
int score_fast_lorentz(FastArgs& a, cudaStream_t st);

bool score_fast_supported(int geom, int precision, int D, int64_t L) {
    (void)geom;
    return precision == LEC_PREC_F32 && D <= 64 && L < (1LL << 28);
}

// level ranges must be ascending and disjoint (they are: consecutive label ranges of the hierarchy levels)
int score_fast_launch(int geom, const float* labels, int64_t L, const float* images, int64_t N, int D, float K,
                      const int32_t* level_start, const int32_t* level_stop, int n_levels, int k, float* scores,
                      int64_t s_img, int64_t s_lab, int32_t* topk_idx, float* topk_val, cudaStream_t st) {
    FastArgs a{};
    a.labels = labels; a.images = images; a.L = L; a.N = N; a.D = D; a.K = K; a.k = topk_idx ? k : 1;
    a.n_levels = n_levels; a.scores = scores; a.s_img = s_img; a.s_lab = s_lab; a.topk_idx = topk_idx; a.topk_val = topk_val;
    if (N == 0 || L == 0) return 0;
    // segments: the levels (clipped to [0, L)), plus the gaps when the full matrix is wanted
    int ns = 0;
    int64_t cursor = 0;
    for (int i = 0; i < n_levels; ++i) {
        int64_t s = level_start[i], e = level_stop[i];
        if (s < cursor || e < s) return LEC_E_K;  // not ascending / disjoint
        if (e > L) e = L;
        if (s > L) s = L;
        if (scores && s > cursor) { a.seg_start[ns] = (int)cursor; a.seg_stop[ns] = (int)s; a.seg_level[ns] = -1; ++ns; }
        a.seg_start[ns] = (int)s; a.seg_stop[ns] = (int)e; a.seg_level[ns] = i; ++ns;  // empty levels still write -1 / inf
        cursor = e;
    }
    if (scores && cursor < L) { a.seg_start[ns] = (int)cursor; a.seg_stop[ns] = (int)L; a.seg_level[ns] = -1; ++ns; }
    // largest first
    for (int i = 1; i < ns; ++i)
        for (int j = i; j > 0 && (a.seg_stop[j] - a.seg_start[j]) > (a.seg_stop[j - 1] - a.seg_start[j - 1]); --j) {
            int t;
            t = a.seg_start[j]; a.seg_start[j] = a.seg_start[j - 1]; a.seg_start[j - 1] = t;
            t = a.seg_stop[j]; a.seg_stop[j] = a.seg_stop[j - 1]; a.seg_stop[j - 1] = t;
            t = a.seg_level[j]; a.seg_level[j] = a.seg_level[j - 1]; a.seg_level[j - 1] = t;
        }
    a.n_seg = ns;
    if (ns == 0) return 0;
    switch (geom) {
        case LEC_GEOM_EUC: return score_fast_euc(a, st);
        case LEC_GEOM_HYP: return score_fast_hyp(a, st);
        case LEC_GEOM_OE: return score_fast_oe(a, st);
        case LEC_GEOM_POINCARE: return score_fast_poincare(a, st);
        case LEC_GEOM_LORENTZ: return score_fast_lorentz(a, st);
    }
    return LEC_E_ENUM;
}

}  // namespace lec
