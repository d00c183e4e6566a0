// Evaluation bookkeeping of the cone path on the device (SURVEY 8(a) rows a13 / a14, 8(f) items 1 and 4).
//
// 1. Best-F1 threshold sweep -- EmbeddingMetrics.calculate_metrics, 'val' phase (order_embeddings.py:272-287 =
//    oe.py:380-395): every unique energy is a candidate threshold t; F1(t) from cp = #{E+ <= t}, cn = #{E- > t}; the
//    first arg-max wins.  The reference evaluates each t with two full passes over the energies in a process pool
//    (O(T n)); here the caller sorts all energies once (ascending, NaN last) together with the running count of
//    positives, and one pass evaluates every run end.  The fp64 expression tree is the reference's
//    (precision = cp / (cp + fp); recall = cp / n_pos; f1 = 2 p r / (p + r)), so F1 values -- and therefore the
//    arg-max under ties -- are bit-identical to the Python floats.
//
// 2. Classification counts -- the per-image bookkeeping of JointEmbeddings.calculate_classification_metrics
//    (oe.py:1775-1796, oe_h.py:2030-2051): from the per-level top-k label ids of every image and its true label
//    per level, hit@k per true label and the tp / fp / fn per label; tn follows from the number of correct
//    predictions of the label's level.  Integer atomics only: bit-exact.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <atomic>

#include "../../include/lec_b200.h"
#include "lec_f1.cuh"

namespace lec {
extern std::atomic<unsigned long long> g_launches;  // lec_api.cu

namespace {

constexpr int kF1Blocks = 592;   // 4 x 148
constexpr int kF1Threads = 256;

struct F1Best { double f1; int64_t idx; };

// number of non-NaN energies: the sort puts NaNs last, so "is NaN" is monotone over the array
__device__ __forceinline__ int64_t first_nan(const float* sorted, int64_t n) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const float v = sorted[mid];
        if (v != v) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// metrics of threshold sorted[i] (a run end): counts from the positive prefix, then lec_f1.cuh's expression tree
__device__ __forceinline__ void sorted_f1_row(const float* sorted, const int64_t* pos_prefix, int64_t i, int64_t n_pos,
                                              int64_t n_neg, int64_t n_fin, double* row) {
    const float t = sorted[i];
    int64_t cp = 0, cn = 0;   // NaN threshold: no comparison holds
    if (t == t) {
        cp = pos_prefix[i];                                              // positives with E <= t
        const int64_t pos_fin = n_fin > 0 ? pos_prefix[n_fin - 1] : 0;   // positives that are not NaN
        const int64_t neg_fin = n_fin - pos_fin;
        cn = neg_fin - ((i + 1) - cp);                                   // negatives with E > t
    }
    f1_row(t, cp, cn, n_pos, n_neg, row);
}

__global__ void __launch_bounds__(kF1Threads) f1_sweep_kernel(const float* __restrict__ sorted, const int64_t* __restrict__ pos_prefix,
                                                               int64_t n, int64_t n_pos, int64_t n_neg, F1Best* __restrict__ block_best) {
    F1Best best{-1.0, INT64_MAX};
    const int64_t n_fin = first_nan(sorted, n);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float t = sorted[i];
        // run end: the last occurrence of a value (all NaNs form one run at the end, like np.unique)
        bool end = (i + 1 == n);
        if (!end) {
            const float nx = sorted[i + 1];
            end = (t == t) ? !(nx == t) : false;
        }
        if (!end) continue;
        double row[7];
        sorted_f1_row(sorted, pos_prefix, i, n_pos, n_neg, n_fin, row);
        double f1 = row[0];
        if (f1 != f1) f1 = -1.0;   // NaN never wins
        if (f1_better(f1, i, best.f1, best.idx)) { best.f1 = f1; best.idx = i; }
    }
    __shared__ F1Best sh[kF1Threads];
    sh[threadIdx.x] = best;
    __syncthreads();
    for (int o = kF1Threads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            const F1Best b = sh[threadIdx.x + o];
            if (f1_better(b.f1, b.idx, sh[threadIdx.x].f1, sh[threadIdx.x].idx)) sh[threadIdx.x] = b;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) block_best[blockIdx.x] = sh[0];
}

__global__ void __launch_bounds__(kF1Threads) f1_final_kernel(const float* __restrict__ sorted, const int64_t* __restrict__ pos_prefix,
                                                               int64_t n, int64_t n_pos, int64_t n_neg, const F1Best* __restrict__ block_best,
                                                               int n_blocks, double* __restrict__ out7) {
    __shared__ F1Best sh[kF1Threads];
    F1Best best{-1.0, INT64_MAX};
    for (int b = threadIdx.x; b < n_blocks; b += blockDim.x) {
        const F1Best c = block_best[b];
        if (f1_better(c.f1, c.idx, best.f1, best.idx)) best = c;
    }
    sh[threadIdx.x] = best;
    __syncthreads();
    for (int o = kF1Threads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            const F1Best b = sh[threadIdx.x + o];
            if (f1_better(b.f1, b.idx, sh[threadIdx.x].f1, sh[threadIdx.x].idx)) sh[threadIdx.x] = b;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (sh[0].idx == INT64_MAX) { for (int j = 0; j < 7; ++j) out7[j] = nan(""); }
        else sorted_f1_row(sorted, pos_prefix, sh[0].idx, n_pos, n_neg, first_nan(sorted, n), out7);
    }
}

struct ClassifyArgs {
    const int32_t* topk_idx; const int32_t* truth; int64_t n_img; int n_levels, k;
    int n_kvals; int kvals[LEC_MAX_TOPK];
    int64_t L;
    unsigned long long* hit;      // [n_kvals, L]
    unsigned long long* counts;   // [3, L]  tp, fp, fn
    unsigned long long* level_correct;  // [n_levels]
};

__global__ void __launch_bounds__(256) classify_kernel(const ClassifyArgs a) {
    const int64_t total = a.n_img * a.n_levels;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int level = (int)(t % a.n_levels);
        const int32_t want = a.truth[t];
        if (want < 0 || want >= a.L) continue;
        const int32_t* top = a.topk_idx + t * a.k;
        for (int j = 0; j < a.n_kvals; ++j) {
            bool hit = false;
            for (int q = 0; q < a.kvals[j] && q < a.k; ++q) hit |= (top[q] == want);
            if (hit) atomicAdd(a.hit + (int64_t)j * a.L + want, 1ull);
        }
        const int32_t pred = top[0];
        if (pred == want) {
            atomicAdd(a.counts + want, 1ull);                 // tp
            atomicAdd(a.level_correct + level, 1ull);         // every other label of the level gets a tn
        } else {
            if (pred >= 0 && pred < a.L) atomicAdd(a.counts + a.L + pred, 1ull);   // fp
            atomicAdd(a.counts + 2 * a.L + want, 1ull);       // fn
        }
    }
}

// Caption-style ranking hinge (order_embeddings_images.py:533-542): one thread per positive walks its M negative
// energies; S_i = sum_j max(0, alpha + E+_i - E-_ij) and, when asked, its VJP scaled by the upstream gradient gS_i.
__global__ void __launch_bounds__(256) caption_hinge_kernel(const float* __restrict__ E_pos, const float* __restrict__ E_neg,
                                                            int64_t B, int M, float alpha, const float* __restrict__ gS,
                                                            float* __restrict__ S, float* __restrict__ gE_pos,
                                                            float* __restrict__ gE_neg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const float ep = E_pos[i];
    const float up = gS ? gS[i] : 1.f;
    float s = 0.f, cnt = 0.f;
    for (int j = 0; j < M; ++j) {
        const float m = (alpha + ep) - E_neg[i * M + j];   // the reference's order: (alpha - s+) + s-
        const bool act = m >= 0.f;                          // clamp(min=0) passes the gradient at equality; NaN: inactive
        s += act ? m : 0.f;
        cnt += act ? 1.f : 0.f;
        if (gE_neg) gE_neg[i * M + j] = act ? -up : 0.f;
        if (!(m == m)) s = m;                               // NaN energy propagates like torch.clamp
    }
    if (S) S[i] = s;
    if (gE_pos) gE_pos[i] = up * cnt;
}

}  // namespace
}  // namespace lec

extern "C" int64_t lec_f1_workspace_bytes(void) { return (int64_t)lec::kF1Blocks * (int64_t)sizeof(lec::F1Best); }

extern "C" int lec_f1_sweep(const float* sorted_energies, const int64_t* pos_prefix, int64_t n, int64_t n_pos, int64_t n_neg,
                            double* out7, void* workspace, int64_t workspace_bytes, void* stream) {
    using namespace lec;
    if (!sorted_energies || !pos_prefix || !out7 || !workspace) return LEC_E_NULL;
    if (n < 1 || n_pos < 0 || n_neg < 0 || n_pos + n_neg != n) return LEC_E_SIZE;
    if (workspace_bytes < lec_f1_workspace_bytes()) return LEC_E_SIZE;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t blocks = (n + kF1Threads - 1) / kF1Threads;
    if (blocks > kF1Blocks) blocks = kF1Blocks;
    F1Best* bb = static_cast<F1Best*>(workspace);
    f1_sweep_kernel<<<(int)blocks, kF1Threads, 0, st>>>(sorted_energies, pos_prefix, n, n_pos, n_neg, bb);
    ++g_launches;
    f1_final_kernel<<<1, kF1Threads, 0, st>>>(sorted_energies, pos_prefix, n, n_pos, n_neg, bb, (int)blocks, out7);
    ++g_launches;
    return (int)cudaGetLastError();
}

extern "C" int lec_classify_counts(const int32_t* topk_idx, const int32_t* truth, int64_t n_img, int n_levels, int k,
                                   const int32_t* k_vals, int n_kvals, int64_t L, uint64_t* hit, uint64_t* counts,
                                   uint64_t* level_correct, void* stream) {
    using namespace lec;
    if (!topk_idx || !truth || !k_vals || !hit || !counts || !level_correct) return LEC_E_NULL;
    if (n_img < 0 || L < 1) return LEC_E_SIZE;
    if (k < 1 || k > LEC_MAX_TOPK || n_levels < 1 || n_levels > LEC_MAX_LEVELS || n_kvals < 1 || n_kvals > LEC_MAX_TOPK) return LEC_E_K;
    if (n_img == 0) return 0;
    ClassifyArgs a{};
    a.topk_idx = topk_idx; a.truth = truth; a.n_img = n_img; a.n_levels = n_levels; a.k = k; a.n_kvals = n_kvals; a.L = L;
    for (int j = 0; j < n_kvals; ++j) a.kvals[j] = k_vals[j];
    a.hit = reinterpret_cast<unsigned long long*>(hit);
    a.counts = reinterpret_cast<unsigned long long*>(counts);
    a.level_correct = reinterpret_cast<unsigned long long*>(level_correct);
    int64_t blocks = (n_img * n_levels + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    classify_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(a);
    ++g_launches;
    return (int)cudaGetLastError();
}

extern "C" int lec_caption_hinge(const float* E_pos, const float* E_neg, int64_t B, int M, float alpha, const float* gS,
                                 float* S, float* gE_pos, float* gE_neg, void* stream) {
    if (B < 0 || M < 0) return LEC_E_SIZE;
    if (B == 0) return 0;
    if (!E_pos || (M > 0 && !E_neg)) return LEC_E_NULL;
    int64_t blocks = (B + 255) / 256;
    if (blocks > 0x7fffffffLL) return LEC_E_SIZE;
    lec::caption_hinge_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(E_pos, E_neg, B, M, alpha, gS, S, gE_pos, gE_neg);
    ++lec::g_launches;
    return (int)cudaGetLastError();
}
