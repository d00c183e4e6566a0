// Pair-energy kernels (flat list, training-layout groups, dense operands), templated on the scalar
// core.  Each lec_pairs_<core>.cu instantiates this header once for its core and exports three
// launchers that lec_api.cu dispatches to.
#pragma once
#include "lec_common.cuh"

namespace lec {

enum Core { CORE_EUC32 = 0, CORE_HYP32 = 1, CORE_HYP64 = 2, CORE_OE32 = 3 };

template <int CORE> struct CoreTraits;
template <> struct CoreTraits<CORE_EUC32> { using Acc = float;  static constexpr bool cone = true,  hyp = false; static constexpr int geom = LEC_GEOM_EUC; };
template <> struct CoreTraits<CORE_HYP32> { using Acc = float;  static constexpr bool cone = true,  hyp = true;  static constexpr int geom = LEC_GEOM_HYP; };
template <> struct CoreTraits<CORE_HYP64> { using Acc = double; static constexpr bool cone = true,  hyp = true;  static constexpr int geom = LEC_GEOM_HYP; };
template <> struct CoreTraits<CORE_OE32>  { using Acc = float;  static constexpr bool cone = false, hyp = false; static constexpr int geom = LEC_GEOM_OE; };

#ifndef LEC_FP32_MINBLOCKS
#define LEC_FP32_MINBLOCKS 3
#endif

struct FlatArgs {
    const float* rows; const double* aux; int ld;
    const void* from_idx; const void* to_idx; int idx_bytes;
    const float* w; const uint8_t* is_pos;
    int64_t P; float K, alpha;
    float* E_out; double* loss_out; float* grad_rows; int grad_replicas; int64_t replica_stride;
    int64_t n_rows; unsigned* index_errors;
};

struct GroupArgs {
    const float* rows; const double* aux; int ld;
    const void* pos_from; const void* pos_to; const void* neg_to; const void* neg_from; int idx_bytes;
    int64_t B; int N;
    const float* w_pos; const float* w_neg;
    float K, alpha;
    float* E_pos; float* E_neg; double* loss_out; float* grad_rows; int grad_replicas; int64_t replica_stride;
    int64_t n_rows; unsigned* index_errors;
    int split;  // teams per group (>= 1): team s of a group takes negatives p = s, s + split, ... of both lists
    int narrow_tail;       // the last float4 chunk of a row holds <= 2 live floats (D % 4 in {1, 2}): its reductions are 64-bit
    unsigned long long* trace;   // LEC_STEP_TRACE builds only
};

// Nickel & Kiela's softmax loss on the Poincare or Lorentz distance (lec_pairs_softmax.cu): B positives with N
// negatives each, neg_to only
struct SoftmaxArgs {
    const float* rows; int ld;
    const void* pos_from; const void* pos_to; const void* neg_to; int idx_bytes;
    int64_t B; int N;
    float* E_pos; float* E_neg; double* loss_out; float* grad_rows; int grad_replicas; int64_t replica_stride;
    int64_t n_rows; unsigned* index_errors;
    int narrow_tail;
};
int launch_pairs_poincare(const SoftmaxArgs& a, cudaStream_t st);
int launch_pairs_lorentz(const SoftmaxArgs& a, cudaStream_t st);

// Gradient reduction of chunk q of a row.  The L2 executes a vector reduction as one fp32 add per element and its add
// rate is what bounds the Euclidean kernels (cfg0, D = 2: 2.3 M REDG.128 per step = 340 G adds/s on a 92 KB target), so
// a chunk whose upper half is padding (D = 2: every chunk; D = 10, 50: the last of 3 / 13) goes out as REDG.64.
__device__ __forceinline__ void red_add_chunk(float* p, float4 v, bool narrow) {
    if (narrow) atomicAdd(reinterpret_cast<float2*>(p), make_float2(v.x, v.y));
    else red_add4(p, v);
}

struct DenseArgs {
    const float* x; const float* y; const float* gE;
    int64_t P; int D; float K;
    float* E_out; float* gx; float* gy;
};

__device__ __forceinline__ int64_t ld_index(const void* p, int64_t i, int idx_bytes) {
    if (idx_bytes == 4) return (int64_t)__ldg(reinterpret_cast<const int32_t*>(p) + i);
    if (idx_bytes == 2) return (int64_t)__ldg(reinterpret_cast<const unsigned short*>(p) + i);
    return (int64_t)__ldg(reinterpret_cast<const long long*>(p) + i);
}

// Row number with the range check nn.Embedding does on the host (IndexError in the reference): an id outside
// [0, n_rows) is counted in *errors (lec_index_errors), replaced by row 0 so that nothing is read or written out of
// bounds, and `ok` is cleared -- the caller then emits NaN for the pair and no gradient.
__device__ __forceinline__ int64_t ld_index_checked(const void* p, int64_t i, int idx_bytes, int64_t n_rows,
                                                    unsigned* errors, bool count, bool& ok) {
    const int64_t ix = ld_index(p, i, idx_bytes);
    if ((uint64_t)ix < (uint64_t)n_rows) return ix;
    if (count && errors) atomicAdd(errors, 1u);
    ok = false;
    return 0;
}

// z and (optionally) the dz/dx, dz/dy coefficients of one pair held by a team.
//   ax : per-row terms of the apex x;  By : |y|^2 (hyperbolic only)
template <int CORE, int T, int V, bool GRAD>
__device__ __forceinline__ void eval_pair(const Vec<V>& X, const Vec<V>& Y,
                                          const Aux<typename CoreTraits<CORE>::Acc>& ax,
                                          typename CoreTraits<CORE>::Acc By, PairGrad& o) {
    using Acc = typename CoreTraits<CORE>::Acc;
    if (CORE == CORE_EUC32) {
        const Acc DD = team_sum<T, Acc>(dist2_part<Acc, V>(Y, X));
        const Acc XD = team_sum<T, Acc>(dot_diff_part<Acc, V>(X, Y));
        euc_pair<Acc, GRAD>(ax, DD, XD, o);
    } else if (CORE == CORE_HYP32) {
        const Acc P = team_sum<T, Acc>(dot_part<Acc, V>(X, Y));
        const Acc S2 = team_sum<T, Acc>(dist2_part<Acc, V>(X, Y));
        hyp_pair<Acc, GRAD>(ax, By, P, S2, o);
    } else if (CORE == CORE_HYP64) {
        const double P = team_sum<T, double>(dot_exact_part<V>(X, Y));
        // |x-y|^2 = |x|^2 + |y|^2 - 2<x,y> is accurate to ~2^-52 (|x|^2+|y|^2)/|x-y|^2 in double; only for
        // nearly coincident points fall back to summing the squared differences directly.
        double S2 = (double)ax.A + (double)By - 2.0 * P;
        const bool close = S2 < 1e-6 * ((double)ax.A + (double)By);
        if (__any_sync(0xffffffffu, close)) {
            const double direct = team_sum<T, double>(dist2_part<double, V>(X, Y));
            if (close) S2 = direct;
        }
        hyp_pair<Acc, GRAD>(ax, By, (Acc)P, (Acc)S2, o);
    } else {
        o.z = (float)team_sum<T, Acc>(relu_diff2_part<Acc, V>(X, Y));
        o.zxx = o.zxy = o.zyx = o.zyy = 0.f;
    }
}

// ------------------------------------------------------------------------------------------------
// Flat pair list
// ------------------------------------------------------------------------------------------------
template <int CORE, int T, int V, bool GRAD>
__global__ void __launch_bounds__(kThreads) pairs_flat_kernel(const FlatArgs a) {
    using Tr = CoreTraits<CORE>;
    using Acc = typename Tr::Acc;
    const int lane_t = threadIdx.x % T;
    const int64_t n_teams = (int64_t)gridDim.x * (kThreads / T);
    const int64_t team = (int64_t)blockIdx.x * (kThreads / T) + threadIdx.x / T;
    const int64_t iters = (a.P + n_teams - 1) / n_teams;
    const int Q = a.ld >> 2;
    float* const grad_base = GRAD ? a.grad_rows + (int64_t)(blockIdx.x % a.grad_replicas) * a.replica_stride : nullptr;
    double loss = 0.0;
    for (int64_t it = 0; it < iters; ++it) {
        const int64_t p = team + it * n_teams;
        const bool valid = p < a.P;
        const int64_t pc = valid ? p : a.P - 1;
        bool ok = true;
        const int64_t ix = ld_index_checked(a.from_idx, pc, a.idx_bytes, a.n_rows, a.index_errors, valid && lane_t == 0, ok);
        const int64_t iy = ld_index_checked(a.to_idx, pc, a.idx_bytes, a.n_rows, a.index_errors, valid && lane_t == 0, ok);
        Vec<V> X, Y;
        load_row<T, V>(X, a.rows, ix, a.ld, lane_t);
        load_row<T, V>(Y, a.rows, iy, a.ld, lane_t);
        Aux<Acc> ax{};
        Acc By = 0;
        if (Tr::cone) ax = load_aux<Acc>(a.aux, ix);
        if (Tr::hyp) By = load_aux_A<Acc>(a.aux, iy);
        PairGrad g;
        eval_pair<CORE, T, V, GRAD>(X, Y, ax, By, g);
        const float w = a.w ? __ldg(a.w + pc) : 1.f;
        const bool pos = a.is_pos ? (__ldg(a.is_pos + pc) != 0) : true;
        float E;
        double l = 0.0;
        const float cf = hinge(g.z, pos, w, a.alpha, E, l);
        if (valid && lane_t == 0) {
            a.E_out[p] = ok ? E : NAN;
            if (ok) loss += l;
        }
        if (GRAD && valid && ok && cf != 0.f) {
            float* gx = grad_base + ix * (int64_t)a.ld;
            float* gy = grad_base + iy * (int64_t)a.ld;
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const int q = lane_t + T * j;
                if (q < Q) {
                    if (!Tr::cone) {
                        const float4 r = relu_diff4(X.c[j], Y.c[j]);
                        const float c2 = 2.f * cf;
                        red_add4(gx + 4 * q, make_float4(c2 * r.x, c2 * r.y, c2 * r.z, c2 * r.w));
                        red_add4(gy + 4 * q, make_float4(-c2 * r.x, -c2 * r.y, -c2 * r.z, -c2 * r.w));
                    } else {
                        red_add4(gx + 4 * q, axpby4(cf * g.zxx, X.c[j], cf * g.zxy, Y.c[j]));
                        red_add4(gy + 4 * q, axpby4(cf * g.zyx, X.c[j], cf * g.zyy, Y.c[j]));
                    }
                }
            }
        }
    }
    block_add_double(loss, a.loss_out);
}

// ------------------------------------------------------------------------------------------------
// Training layout: one team per positive and its 2N negatives.  The gradients of the two shared
// endpoints u_i, v_i are accumulated in registers and written with one vector reduction each; only
// the 2N corrupted rows need their own reduction.  When a batch has too few positives to fill the GPU
// (cfg4: 2 520 positives x 51 pairs), a group is split over `split` teams: team s evaluates the positive
// (s == 0 only) and every split-th negative of both lists, and flushes its own partial sums for u_i, v_i.
// ------------------------------------------------------------------------------------------------
// Block size: the fp64-core kernel needs ~166 registers per thread, i.e. one 256-thread block (8 warps) per SM;
// 128-thread blocks fit three (12 warps), which is what hides the gather / reduction latency.
constexpr int kGroupThreads = 128;
// Minimum resident 256-thread blocks per SM the register allocation must allow: 2 caps the kernel at 128 registers
// (fp64 core: 28 bytes of spill, against the 184 it asks for uncapped) and doubles the resident warps.  The fp32 cores
// with one float4 per row (D <= 4: cfg0) fit under a tighter cap without spilling and are gather-latency-bound -- r2x
// sweep on cfg0: cap 128 / 80 / 64 -> pair kernel 29.8 / 26.8 / 29.2 us; rows of three chunks (D = 10) spill at 80 and
// lose (18.0 -> 23.1 us).
template <int CORE, int V>
constexpr int kGroupedMinBlocks = (CORE != CORE_HYP64 && V == 1) ? LEC_FP32_MINBLOCKS : 2;

template <int CORE, int T, int V, bool GRAD>
__global__ void __launch_bounds__(kThreads, (kGroupedMinBlocks<CORE, V>)) pairs_grouped_kernel(const GroupArgs a) {
    using Tr = CoreTraits<CORE>;
    using Acc = typename Tr::Acc;
    pdl_launch_dependents();   // the update kernel may take its (few) SM slots now; it parks in pdl_wait()
    pdl_wait();                // rows / aux / cleared replicas of the previous update are complete
    if (threadIdx.x == 0) LEC_TRACE_MIN(a.trace, 0);
    const int lane_t = threadIdx.x % T;
    constexpr int tpb = kGroupThreads / T;   // teams per block
    const int64_t n_teams = (int64_t)gridDim.x * tpb;
    const int64_t team = (int64_t)blockIdx.x * tpb + threadIdx.x / T;
    const int split = a.split;
    const int64_t n_items = a.B * split;
    const int64_t iters = (n_items + n_teams - 1) / n_teams;
    const int Q = a.ld >> 2;
    const int N = a.N;
    const int q_narrow = a.narrow_tail ? Q - 1 : -1;   // chunk whose reductions are 64 bits wide
    float* const grad_base = GRAD ? a.grad_rows + (int64_t)(blockIdx.x % a.grad_replicas) * a.replica_stride : nullptr;
    double loss = 0.0;
    for (int64_t it = 0; it < iters; ++it) {
        const int64_t item = team + it * n_teams;
        const bool valid = item < n_items;
        const int64_t ic_item = valid ? item : n_items - 1;
        const int64_t gidx = ic_item / split;
        const int sub = (int)(ic_item - gidx * split);
        const int64_t gc = gidx;
        const bool writer = valid && lane_t == 0;
        bool ok_g = true;   // both shared endpoints inside the table
        const int64_t iu = ld_index_checked(a.pos_from, gc, a.idx_bytes, a.n_rows, a.index_errors, writer && sub == 0, ok_g);
        const int64_t iv = ld_index_checked(a.pos_to, gc, a.idx_bytes, a.n_rows, a.index_errors, writer && sub == 0, ok_g);
        Vec<V> U, W;
        load_row<T, V>(U, a.rows, iu, a.ld, lane_t);
        load_row<T, V>(W, a.rows, iv, a.ld, lane_t);
        Aux<Acc> au{};
        Acc AW = 0;
        if (Tr::cone) au = load_aux<Acc>(a.aux, iu);
        if (Tr::hyp) AW = load_aux_A<Acc>(a.aux, iv);
        float su_u = 0.f, su_w = 0.f, sw_u = 0.f, sw_w = 0.f;
        Vec<V> accU, accW;
#pragma unroll
        for (int j = 0; j < V; ++j) accU.c[j] = accW.c[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        bool touch_u = false, touch_w = false;

        PairGrad g;
        float E;
        double l = 0.0;
        // positive (x = u, y = v): evaluated by every team of a split group (eval_pair votes warp-wide, so it
        // cannot sit in a divergent branch), counted by team 0 only
        {
            const bool act = sub == 0;
            eval_pair<CORE, T, V, GRAD>(U, W, au, AW, g);
            const float w = a.w_pos ? __ldg(a.w_pos + gc) : 1.f;
            double lp = 0.0;
            const float cf = hinge(g.z, true, w, a.alpha, E, lp);
            if (act && ok_g) l += lp;
            if (writer && act) a.E_pos[gidx] = ok_g ? E : NAN;
            if (GRAD && valid && act && ok_g && cf != 0.f) {
                touch_u = touch_w = true;
                if (!Tr::cone) {
#pragma unroll
                    for (int j = 0; j < V; ++j) {
                        const float4 r = relu_diff4(U.c[j], W.c[j]);
                        fma4(accU.c[j], 2.f * cf, r);
                        fma4(accW.c[j], -2.f * cf, r);
                    }
                } else {
                    su_u += cf * g.zxx; su_w += cf * g.zxy; sw_u += cf * g.zyx; sw_w += cf * g.zyy;
                }
            }
        }
        const int64_t nbase = gc * (int64_t)N;
        const int64_t ebase = gc * (int64_t)(2 * N);
        // negatives with a corrupted child: (x = u, y = c)
        // every team of a warp runs the same number of trips (eval_pair votes warp-wide); surplus trips of a
        // split group re-evaluate the last negative with their writes masked off
        const int trips = (N + split - 1) / split;
        for (int pi = 0; pi < trips; ++pi) {
            const int pr = sub + pi * split;
            const bool act = pr < N;
            const int p = act ? pr : N - 1;
            bool ok = ok_g;
            const int64_t ic = ld_index_checked(a.neg_to, nbase + p, a.idx_bytes, a.n_rows, a.index_errors, writer && act, ok);
            Vec<V> C;
            load_row<T, V>(C, a.rows, ic, a.ld, lane_t);
            Acc AC = 0;
            if (Tr::hyp) AC = load_aux_A<Acc>(a.aux, ic);
            eval_pair<CORE, T, V, GRAD>(U, C, au, AC, g);
            const float w = a.w_neg ? __ldg(a.w_neg + ebase + p) : 1.f;
            double lp = 0.0;
            const float cf = hinge(g.z, false, w, a.alpha, E, lp);
            if (act && ok) l += lp;
            if (writer && act) a.E_neg[ebase + p] = ok ? E : NAN;
            if (GRAD && valid && act && ok && cf != 0.f) {
                touch_u = true;
                float* gcp = grad_base + ic * (int64_t)a.ld;
                if (Tr::cone) su_u += cf * g.zxx;
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int q = lane_t + T * j;
                    if (!Tr::cone) {
                        const float4 r = relu_diff4(U.c[j], C.c[j]);
                        const float c2 = 2.f * cf;
                        fma4(accU.c[j], c2, r);
                        if (q < Q) red_add_chunk(gcp + 4 * q, make_float4(-c2 * r.x, -c2 * r.y, -c2 * r.z, -c2 * r.w), q == q_narrow);
                    } else {
                        fma4(accU.c[j], cf * g.zxy, C.c[j]);
                        if (q < Q) red_add_chunk(gcp + 4 * q, axpby4(cf * g.zyx, U.c[j], cf * g.zyy, C.c[j]), q == q_narrow);
                    }
                }
            }
        }
        // negatives with a corrupted parent: (x = c, y = v)
        for (int pi = 0; pi < trips; ++pi) {
            const int pr = sub + pi * split;
            const bool act = pr < N;
            const int p = act ? pr : N - 1;
            bool ok = ok_g;
            const int64_t ic = ld_index_checked(a.neg_from, nbase + p, a.idx_bytes, a.n_rows, a.index_errors, writer && act, ok);
            Vec<V> C;
            load_row<T, V>(C, a.rows, ic, a.ld, lane_t);
            Aux<Acc> ac{};
            if (Tr::cone) ac = load_aux<Acc>(a.aux, ic);
            eval_pair<CORE, T, V, GRAD>(C, W, ac, AW, g);
            const float w = a.w_neg ? __ldg(a.w_neg + ebase + N + p) : 1.f;
            double lp = 0.0;
            const float cf = hinge(g.z, false, w, a.alpha, E, lp);
            if (act && ok) l += lp;
            if (writer && act) a.E_neg[ebase + N + p] = ok ? E : NAN;
            if (GRAD && valid && act && ok && cf != 0.f) {
                touch_w = true;
                float* gcp = grad_base + ic * (int64_t)a.ld;
                if (Tr::cone) sw_w += cf * g.zyy;
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int q = lane_t + T * j;
                    if (!Tr::cone) {
                        const float4 r = relu_diff4(C.c[j], W.c[j]);
                        const float c2 = 2.f * cf;
                        fma4(accW.c[j], -c2, r);
                        if (q < Q) red_add_chunk(gcp + 4 * q, make_float4(c2 * r.x, c2 * r.y, c2 * r.z, c2 * r.w), q == q_narrow);
                    } else {
                        fma4(accW.c[j], cf * g.zyx, C.c[j]);
                        if (q < Q) red_add_chunk(gcp + 4 * q, axpby4(cf * g.zxx, C.c[j], cf * g.zxy, W.c[j]), q == q_narrow);
                    }
                }
            }
        }
        if (writer) loss += l;
        if (GRAD && valid && ok_g) {
            float* gu = grad_base + iu * (int64_t)a.ld;
            float* gw = grad_base + iv * (int64_t)a.ld;
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const int q = lane_t + T * j;
                if (q < Q) {
                    if (touch_u) {
                        float4 v = accU.c[j];
                        if (Tr::cone) { fma4(v, su_u, U.c[j]); fma4(v, su_w, W.c[j]); }
                        red_add_chunk(gu + 4 * q, v, q == q_narrow);
                    }
                    if (touch_w) {
                        float4 v = accW.c[j];
                        if (Tr::cone) { fma4(v, sw_u, U.c[j]); fma4(v, sw_w, W.c[j]); }
                        red_add_chunk(gw + 4 * q, v, q == q_narrow);
                    }
                }
            }
        }
    }
    block_add_double(loss, a.loss_out);
    if (threadIdx.x == 0) LEC_TRACE_MAX(a.trace, 1);
}

// ------------------------------------------------------------------------------------------------
// Dense operands x, y [P, D] (row stride D): one thread per pair, per-row terms computed in line.
// ------------------------------------------------------------------------------------------------
template <int CORE, bool BWD>
__global__ void __launch_bounds__(kThreads) energy_dense_kernel(const DenseArgs a) {
    using Tr = CoreTraits<CORE>;
    using Acc = typename Tr::Acc;
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x; p < a.P; p += stride) {
        const float* x = a.x + p * a.D;
        const float* y = a.y + p * a.D;
        Acc s0 = 0, s1 = 0, s2 = 0, s3 = 0;
        for (int d = 0; d < a.D; ++d) {
            const float xv = __ldg(x + d), yv = __ldg(y + d);
            if (CORE == CORE_EUC32) {
                const Acc dv = (Acc)yv - (Acc)xv;
                s0 += (Acc)xv * (Acc)xv; s1 += dv * dv; s2 += (Acc)xv * dv;
            } else if (CORE == CORE_OE32) {
                const float r = fmaxf(xv - yv, 0.f);
                s0 += (Acc)r * (Acc)r;
            } else {
                const Acc dv = (Acc)xv - (Acc)yv;
                s0 += (Acc)xv * (Acc)xv; s1 += (Acc)yv * (Acc)yv; s2 += (Acc)xv * (Acc)yv; s3 += dv * dv;
            }
        }
        PairGrad g;
        g.zxx = g.zxy = g.zyx = g.zyy = 0.f;
        if (CORE == CORE_EUC32) euc_pair<Acc, BWD>(row_aux<Acc>(LEC_GEOM_EUC, s0, a.K), s1, s2, g);
        else if (CORE == CORE_OE32) g.z = (float)s0;
        else hyp_pair<Acc, BWD>(row_aux<Acc>(LEC_GEOM_HYP, s0, a.K), s1, s2, s3, g);
        if (!BWD) {
            a.E_out[p] = relu_nan(g.z);
        } else {
            const float cf = (g.z >= 0.f) ? __ldg(a.gE + p) : 0.f;
            float* gx = a.gx + p * a.D;
            float* gy = a.gy + p * a.D;
            for (int d = 0; d < a.D; ++d) {
                const float xv = __ldg(x + d), yv = __ldg(y + d);
                if (!Tr::cone) {
                    const float r = 2.f * cf * fmaxf(xv - yv, 0.f);
                    gx[d] = r; gy[d] = -r;
                } else {
                    gx[d] = cf * fmaf(g.zxx, xv, g.zxy * yv);
                    gy[d] = cf * fmaf(g.zyx, xv, g.zyy * yv);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Host-side launch helpers
// ------------------------------------------------------------------------------------------------
inline int grid_for(int64_t items, int teams_per_block, int blocks_per_sm) {
    int64_t need = (items + teams_per_block - 1) / teams_per_block;
    int64_t cap = (int64_t)sm_count() * blocks_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

template <int CORE, int T, int V>
int launch_flat_tv(const FlatArgs& a, cudaStream_t st) {
    const int grid = grid_for(a.P, kThreads / T, 8);
    if (a.grad_rows) pairs_flat_kernel<CORE, T, V, true><<<grid, kThreads, 0, st>>>(a);
    else pairs_flat_kernel<CORE, T, V, false><<<grid, kThreads, 0, st>>>(a);
    ++g_launches;
    return (int)cudaGetLastError();
}

// Teams per group.  A team's trip count is 1 + 2*ceil(N/s) pair evaluations (the positive is re-evaluated by every team
// of a split group), so splitting only pays while the batch cannot fill the GPU: s is the largest split that still
// fits one resident wave of `cap` teams.  cfg4 (2 569 positives x 51 pairs, cap 9 472) -> s = 3, measured 30.8 us against
// 71.7 us unsplit and 37.0 us at s = 5 (profiles/r1d_cfg4_split_sweep.md); a batch that already fills the GPU (cfg1: 190 650
// positives) stays at s = 1, where no pair is evaluated twice.
inline int choose_split(int64_t B, int N, int64_t cap) {
    if (B <= 0 || N <= 1 || cap <= 0) return 1;
    int64_t s = cap / B;
    if (s > N) s = N;
    return s < 1 ? 1 : (int)s;
}

template <int CORE, int T, int V>
int launch_grouped_tv(const GroupArgs& a0, cudaStream_t st) {
    GroupArgs a = a0;
    constexpr int block = kGroupThreads;
    static const int resident_blocks = [] {
        int nb = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, pairs_grouped_kernel<CORE, T, V, true>, block, 0);
        return nb > 0 ? nb : 1;
    }();
#ifdef LEC_STEP_TRACE
    a.trace = g_step_trace;
#endif
    a.split = choose_split(a.B, a.N, (int64_t)sm_count() * resident_blocks * (block / T));
    const int grid = grid_for(a.B * a.split, block / T, 8 * kThreads / block);
    const cudaError_t le = a.grad_rows ? launch_step_kernel(pairs_grouped_kernel<CORE, T, V, true>, grid, block, st, a)
                                       : launch_step_kernel(pairs_grouped_kernel<CORE, T, V, false>, grid, block, st, a);
    ++g_launches;
    return (int)(le != cudaSuccess ? le : cudaGetLastError());
}

#define LEC_DISPATCH_TV(FN, CORE, Q, ...)                                   \
    do {                                                                    \
        if ((Q) == 1) return FN<CORE, 1, 1>(__VA_ARGS__);                   \
        if ((Q) == 2) return FN<CORE, 1, 2>(__VA_ARGS__);                   \
        if ((Q) == 3) return FN<CORE, 1, 3>(__VA_ARGS__);                   \
        if ((Q) == 4) return FN<CORE, 1, 4>(__VA_ARGS__);                   \
        if ((Q) <= 16) return FN<CORE, 4, 4>(__VA_ARGS__);                  \
        if ((Q) <= 64) return FN<CORE, 16, 4>(__VA_ARGS__);                 \
        return FN<CORE, 32, 8>(__VA_ARGS__);                                \
    } while (0)

template <int CORE>
int launch_flat(const FlatArgs& a, cudaStream_t st) {
    LEC_DISPATCH_TV(launch_flat_tv, CORE, a.ld >> 2, a, st);
}
template <int CORE>
int launch_grouped(const GroupArgs& a, cudaStream_t st) {
    LEC_DISPATCH_TV(launch_grouped_tv, CORE, a.ld >> 2, a, st);
}
template <int CORE>
int launch_dense(const DenseArgs& a, bool bwd, cudaStream_t st) {
    const int grid = grid_for(a.P, kThreads, 8);
    if (bwd) energy_dense_kernel<CORE, true><<<grid, kThreads, 0, st>>>(a);
    else energy_dense_kernel<CORE, false><<<grid, kThreads, 0, st>>>(a);
    ++g_launches;
    return (int)cudaGetLastError();
}

#define LEC_DEFINE_CORE_TU(CORE, NAME)                                                                      \
    namespace lec {                                                                                         \
    int launch_flat_##NAME(const FlatArgs& a, cudaStream_t st) { return launch_flat<CORE>(a, st); }          \
    int launch_grouped_##NAME(const GroupArgs& a, cudaStream_t st) { return launch_grouped<CORE>(a, st); }   \
    int launch_dense_##NAME(const DenseArgs& a, bool bwd, cudaStream_t st) { return launch_dense<CORE>(a, bwd, st); } \
    }

}  // namespace lec
