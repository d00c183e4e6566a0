// Nickel & Kiela's softmax loss (lec_pairs_poincare, lec_pairs_lorentz, include/lec_b200.h): one team per positive
// (u, v) and its N negatives v'_j, the team sizing of the other pair kernels (chunk q = lane + T*j of a row per lane).
// The distance is a policy of the kernel (PoincareDist, LorentzDist): everything else -- the two passes, the replica
// scatter, u's register accumulation, the index checks -- is one body.
//
//   pass 1  d(u, w) for w = v, v'_1 .. v'_N (energies out), online max-subtracted log-sum-exp of -d: the loss
//   pass 2  the same rows again (they are L1/L2-resident), the same fp64 instructions (the same d), the softmax weight
//           p_w = exp(-d_w - lse) and dL/dd = [w == v] - p_w chained through dd/du, dd/dw: w's gradient leaves as one
//           vector reduction, u's is accumulated in registers over the 1 + N pairs and leaves once
//
// With A = |x|^2, B = |y|^2, s = |x - y|^2 (summed from the differences), p = <x, y>, all in fp64 from the fp32 rows:
// Poincare ball (Nickel & Kiela 2017)
//   delta = 2 s / ((1 - A)(1 - B)),  d = arcosh(1 + delta) = log1p(delta + sqrt(delta (delta + 2)))
//   dd/dx = 4 / ((1 - B) r) ((B - 2p + 1) / (1 - A)^2 x - y / (1 - A)),  r = sqrt(delta (delta + 2)), 0 where delta = 0
// and symmetrically for y.
// Lorentz model (Nickel & Kiela 2018), rows are the spatial parts of hyperboloid points, x0 = sqrt(1 + A), y0 = sqrt(1 + B):
//   w = -<X,Y>_L - 1 = (s - (x0 - y0)^2) / 2,  x0 - y0 = (A - B) / (x0 + y0),  A - B = <x - y, x + y> summed from the
//   differences,  w clamped at 0,  d = log1p(w + r),
//   r = sqrt(w (w + 2));  dd/dx = (y0 / x0 x - y) / r,  dd/dy = (x0 / y0 y - x) / r,  0 where w = 0.
// The difference form of w keeps its digits for nearby points far from the origin, where x0 y0 - 1 - p cancels them:
// every input of the final subtraction is accurate to a few ulp of s, so |dw| <= (3D + 12) eps64 s.
#include "lec_pairs_impl.cuh"

namespace lec {

// the pair terms of (x = u, y = w) with A = |u|^2 already known
struct PairTerms {
    double d;
    double cxx, cxy;  // dd/dx = cxx x + cxy y
    double cyy, cyx;  // dd/dy = cyy y + cyx x
};

struct PoincareDist {
    template <int T, int V, bool GRAD>
    static __device__ __forceinline__ PairTerms pair(const Vec<V>& X, const Vec<V>& Y, double A) {
        double bb = 0.0, ss = 0.0, pp = 0.0;
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float yv[4] = {Y.c[j].x, Y.c[j].y, Y.c[j].z, Y.c[j].w};
            const float xv[4] = {X.c[j].x, X.c[j].y, X.c[j].z, X.c[j].w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const double y = (double)yv[c], x = (double)xv[c], df = x - y;
                bb = fma(y, y, bb);
                ss = fma(df, df, ss);
                if (GRAD) pp = fma(x, y, pp);
            }
        }
        const double B = team_sum<T, double>(bb);
        const double S = team_sum<T, double>(ss);
        const double ia = 1.0 / (1.0 - A), ib = 1.0 / (1.0 - B);
        const double delta = 2.0 * S * ia * ib;
        const double r = sqrt(delta * (delta + 2.0));
        PairTerms o;
        o.d = log1p(delta + r);
        o.cxx = o.cxy = o.cyy = o.cyx = 0.0;
        if (GRAD) {
            const double P = team_sum<T, double>(pp);
            if (delta != 0.0) {
                const double kx = 4.0 * ib / r, ky = 4.0 * ia / r;
                o.cxx = kx * (B - 2.0 * P + 1.0) * ia * ia;
                o.cxy = -kx * ia;
                o.cyy = ky * (A - 2.0 * P + 1.0) * ib * ib;
                o.cyx = -ky * ib;
            }
        }
        return o;
    }
};

struct LorentzDist {
    template <int T, int V, bool GRAD>
    static __device__ __forceinline__ PairTerms pair(const Vec<V>& X, const Vec<V>& Y, double A) {
        double bb = 0.0, ss = 0.0, dd = 0.0;
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const float yv[4] = {Y.c[j].x, Y.c[j].y, Y.c[j].z, Y.c[j].w};
            const float xv[4] = {X.c[j].x, X.c[j].y, X.c[j].z, X.c[j].w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const double x = (double)xv[c], y = (double)yv[c], df = x - y;
                bb = fma(y, y, bb);
                ss = fma(df, df, ss);
                dd = fma(df, x + y, dd);
            }
        }
        const double B = team_sum<T, double>(bb);
        const double S = team_sum<T, double>(ss);
        const double AB = team_sum<T, double>(dd);   // A - B as <x - y, x + y>: no cancellation of A against B
        const double x0 = sqrt(1.0 + A), y0 = sqrt(1.0 + B);
        const double t = AB / (x0 + y0);             // x0 - y0
        double w = 0.5 * (S - t * t);
        w = w < 0.0 ? 0.0 : w;                  // NaN stays NaN
        const double r = sqrt(w * (w + 2.0));
        PairTerms o;
        o.d = log1p(w + r);
        o.cxx = o.cxy = o.cyy = o.cyx = 0.0;
        if (GRAD && w != 0.0) {
            const double ir = 1.0 / r;
            o.cxx = y0 / x0 * ir;
            o.cyy = x0 / y0 * ir;
            o.cxy = o.cyx = -ir;
        }
        return o;
    }
};

template <class Dist, int T, int V>
__global__ void __launch_bounds__(kGroupThreads) pairs_softmax_kernel(const SoftmaxArgs a) {
    pdl_launch_dependents();
    pdl_wait();   // rows and cleared replicas of the previous update are complete
    const int lane_t = threadIdx.x % T;
    constexpr int tpb = kGroupThreads / T;
    const int64_t n_teams = (int64_t)gridDim.x * tpb;
    const int64_t team = (int64_t)blockIdx.x * tpb + threadIdx.x / T;
    const int64_t iters = (a.B + n_teams - 1) / n_teams;   // the same in every team: team sums are warp-wide
    const int Q = a.ld >> 2, N = a.N;
    const int q_narrow = a.narrow_tail ? Q - 1 : -1;
    const bool grad = a.grad_rows != nullptr;
    float* const grad_base = grad ? a.grad_rows + (int64_t)(blockIdx.x % a.grad_replicas) * a.replica_stride : nullptr;
    double loss = 0.0;
    for (int64_t it = 0; it < iters; ++it) {
        const int64_t i = team + it * n_teams;
        const bool valid = i < a.B;
        const int64_t ic = valid ? i : a.B - 1;
        const bool writer = valid && lane_t == 0;
        bool ok_g = true;
        const int64_t iu = ld_index_checked(a.pos_from, ic, a.idx_bytes, a.n_rows, a.index_errors, writer, ok_g);
        const int64_t iv = ld_index_checked(a.pos_to, ic, a.idx_bytes, a.n_rows, a.index_errors, writer, ok_g);
        Vec<V> U;
        load_row<T, V>(U, a.rows, iu, a.ld, lane_t);
        double aa = 0.0;
#pragma unroll
        for (int j = 0; j < V; ++j) {
            aa = fma((double)U.c[j].x, (double)U.c[j].x, aa); aa = fma((double)U.c[j].y, (double)U.c[j].y, aa);
            aa = fma((double)U.c[j].z, (double)U.c[j].z, aa); aa = fma((double)U.c[j].w, (double)U.c[j].w, aa);
        }
        const double A = team_sum<T, double>(aa);
        const int64_t nbase = ic * (int64_t)N;
        // pair k = 0 is the positive, k = 1 .. N the negatives; a bad negative id is counted in pass 1 only
        auto row_of = [&](int k, bool count, bool& ok) -> int64_t {
            if (k == 0) return iv;
            return ld_index_checked(a.neg_to, nbase + k - 1, a.idx_bytes, a.n_rows, a.index_errors, count, ok);
        };
        // ---- pass 1: energies and the log-sum-exp of -d over the group
        double m = -INFINITY, S = 0.0, d_pos = 0.0;
        for (int k = 0; k <= N; ++k) {
            bool ok = ok_g;
            const int64_t iw = row_of(k, writer, ok);
            Vec<V> W;
            load_row<T, V>(W, a.rows, iw, a.ld, lane_t);
            const double d = Dist::template pair<T, V, false>(U, W, A).d;
            if (writer) {
                if (k == 0) a.E_pos[i] = ok ? (float)d : NAN;
                else a.E_neg[nbase + k - 1] = ok ? (float)d : NAN;
            }
            if (k == 0) d_pos = d;
            if (ok) {
                const double x = -d;
                if (x > m) { S = S * exp(m - x) + 1.0; m = x; }
                else S += exp(x - m);
            }
        }
        const double lse = m + log(S);
        if (writer && ok_g) loss += d_pos + lse;
        // ---- pass 2: softmax weights and the gradient
        if (!grad) continue;   // grid-uniform
        const bool g_ok = valid && ok_g;
        double su = 0.0;   // coefficient of u in u's gradient
        Vec<V> accU;       // the other endpoints' part of u's gradient
#pragma unroll
        for (int j = 0; j < V; ++j) accU.c[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int k = 0; k <= N; ++k) {
            bool ok = ok_g;
            const int64_t iw = row_of(k, false, ok);
            Vec<V> W;
            load_row<T, V>(W, a.rows, iw, a.ld, lane_t);
            const PairTerms t = Dist::template pair<T, V, true>(U, W, A);
            const double c = (k == 0 ? 1.0 : 0.0) - exp(-t.d - lse);   // dL/dd
            if (!(g_ok && ok)) continue;
            su += c * t.cxx;
            const float fxy = (float)(c * t.cxy), fyy = (float)(c * t.cyy), fyx = (float)(c * t.cyx);
            float* gw = grad_base + iw * (int64_t)a.ld;
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const int q = lane_t + T * j;
                fma4(accU.c[j], fxy, W.c[j]);
                if (q < Q) red_add_chunk(gw + 4 * q, axpby4(fyy, W.c[j], fyx, U.c[j]), q == q_narrow);
            }
        }
        if (g_ok) {
            float* gu = grad_base + iu * (int64_t)a.ld;
            const float fu = (float)su;
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const int q = lane_t + T * j;
                if (q < Q) {
                    float4 v = accU.c[j];
                    fma4(v, fu, U.c[j]);
                    red_add_chunk(gu + 4 * q, v, q == q_narrow);
                }
            }
        }
    }
    block_add_double(loss, a.loss_out);
}

template <class Dist, int T, int V>
static int launch_softmax_tv(const SoftmaxArgs& a, cudaStream_t st) {
    constexpr int block = kGroupThreads;
    const int grid = grid_for(a.B, block / T, 8 * kThreads / block);
    const cudaError_t e = launch_step_kernel(pairs_softmax_kernel<Dist, T, V>, grid, block, st, a);
    ++g_launches;
    return (int)(e != cudaSuccess ? e : cudaGetLastError());
}

template <class Dist>
static int launch_softmax(const SoftmaxArgs& a, cudaStream_t st) {
    const int Q = a.ld >> 2;   // DESIGN.md section 3: Q <= 4 -> T = 1, Q <= 16 -> T = 4, Q <= 64 -> T = 16, else T = 32
    if (Q == 1) return launch_softmax_tv<Dist, 1, 1>(a, st);
    if (Q == 2) return launch_softmax_tv<Dist, 1, 2>(a, st);
    if (Q == 3) return launch_softmax_tv<Dist, 1, 3>(a, st);
    if (Q == 4) return launch_softmax_tv<Dist, 1, 4>(a, st);
    if (Q <= 16) return launch_softmax_tv<Dist, 4, 4>(a, st);
    if (Q <= 64) return launch_softmax_tv<Dist, 16, 4>(a, st);
    return launch_softmax_tv<Dist, 32, 8>(a, st);
}

int launch_pairs_poincare(const SoftmaxArgs& a, cudaStream_t st) { return launch_softmax<PoincareDist>(a, st); }
int launch_pairs_lorentz(const SoftmaxArgs& a, cudaStream_t st) { return launch_softmax<LorentzDist>(a, st); }

}  // namespace lec
