// Shared device helpers for the entailment-cone kernels (sm_100a).
//
// Work decomposition used by every pair kernel: a TEAM of T lanes (T a power of two <= 32) owns one
// work item (a pair, or a positive with its 2N negatives).  A row of the transformed table is
// [ld] floats, ld % 4 == 0, and is held by the team as V float4 chunks per lane, chunk q = lane + T*j
// so that one load instruction of the team covers 16*T contiguous bytes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/lec_b200.h"

namespace lec {

constexpr int kThreads = 256;
constexpr float kNormEps = 1e-12f;   // F.normalize eps (order_embeddings.py:197, :965)
constexpr float kClampEps = 1e-5f;   // acos/asin clamp (order_embeddings_h.py:1113-1114)

extern std::atomic<unsigned long long> g_launches;  // host-side launch counter (lec_api.cu); callers may be on several threads

// Programmatic dependent launch.  lec_cone_step sets t_pdl around its launches: each kernel of the step is then
// launched with programmatic stream serialisation, i.e. its blocks may become resident while the previous kernel of the
// stream drains, and park in pdl_wait() -- which returns once that kernel has completed and flushed -- so the launch
// latency between the two or three kernels of a step is hidden.  A kernel launched without the attribute sees both
// instructions as no-ops.
extern thread_local int t_pdl;
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename Arg>
inline cudaError_t launch_step_kernel(void (*kern)(const Arg), int grid, int block, cudaStream_t st, const Arg& a, size_t smem = 0) {
    if (!t_pdl) {
        kern<<<grid, block, smem, st>>>(a);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, a);
}

template <int V>
struct Vec {
    float4 c[V];
};

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// d += a (vector float4 reduction into global memory: one REDG.E.ADD.F32x4 on sm_100a)
__device__ __forceinline__ void red_add4(float* p, float4 v) { atomicAdd(reinterpret_cast<float4*>(p), v); }

template <int T, typename S>
__device__ __forceinline__ S team_sum(S v) {
#pragma unroll
    for (int o = T / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <typename S>
__device__ __forceinline__ S warp_sum(S v) {
    return team_sum<32, S>(v);
}

template <int T, int V>
__device__ __forceinline__ void load_row(Vec<V>& r, const float* __restrict__ rows, int64_t row, int ld, int lane_t) {
    const float* base = rows + row * (int64_t)ld;
    const int Q = ld >> 2;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int q = lane_t + T * j;
        if (q < Q) r.c[j] = ldg4(base + 4 * q);
        else r.c[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

template <typename S, int V>
__device__ __forceinline__ S dot_part(const Vec<V>& a, const Vec<V>& b) {
    S s = 0;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        s += (S)a.c[j].x * (S)b.c[j].x;
        s += (S)a.c[j].y * (S)b.c[j].y;
        s += (S)a.c[j].z * (S)b.c[j].z;
        s += (S)a.c[j].w * (S)b.c[j].w;
    }
    return s;
}

// <a, b> to double accuracy without double copies of the operands: each fp32 product is split exactly
// into hi + lo (lo via FMA); hi parts are summed in double, lo parts (2^-24 smaller) in fp32.
template <int V>
__device__ __forceinline__ double dot_exact_part(const Vec<V>& a, const Vec<V>& b) {
    double s = 0.0;
    float lo = 0.f;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        float h;
        h = __fmul_rn(a.c[j].x, b.c[j].x); lo += __fmaf_rn(a.c[j].x, b.c[j].x, -h); s += (double)h;
        h = __fmul_rn(a.c[j].y, b.c[j].y); lo += __fmaf_rn(a.c[j].y, b.c[j].y, -h); s += (double)h;
        h = __fmul_rn(a.c[j].z, b.c[j].z); lo += __fmaf_rn(a.c[j].z, b.c[j].z, -h); s += (double)h;
        h = __fmul_rn(a.c[j].w, b.c[j].w); lo += __fmaf_rn(a.c[j].w, b.c[j].w, -h); s += (double)h;
    }
    return s + (double)lo;
}

// sum (a-b)^2; the subtraction is done in the accumulator type (fp32: exactly what torch.norm(x - y)
// sees in the reference's fp32 run; fp64: exact difference of the fp32 inputs)
template <typename S, int V>
__device__ __forceinline__ S dist2_part(const Vec<V>& a, const Vec<V>& b) {
    S s = 0;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        S d;
        d = (S)a.c[j].x - (S)b.c[j].x; s += d * d;
        d = (S)a.c[j].y - (S)b.c[j].y; s += d * d;
        d = (S)a.c[j].z - (S)b.c[j].z; s += d * d;
        d = (S)a.c[j].w - (S)b.c[j].w; s += d * d;
    }
    return s;
}

// <x, y - x> (Euclidean cone numerator)
template <typename S, int V>
__device__ __forceinline__ S dot_diff_part(const Vec<V>& x, const Vec<V>& y) {
    S s = 0;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        s += (S)x.c[j].x * ((S)y.c[j].x - (S)x.c[j].x);
        s += (S)x.c[j].y * ((S)y.c[j].y - (S)x.c[j].y);
        s += (S)x.c[j].z * ((S)y.c[j].z - (S)x.c[j].z);
        s += (S)x.c[j].w * ((S)y.c[j].w - (S)x.c[j].w);
    }
    return s;
}

// sum max(0, x - y)^2 (order-embedding energy)
template <typename S, int V>
__device__ __forceinline__ S relu_diff2_part(const Vec<V>& x, const Vec<V>& y) {
    S s = 0;
#pragma unroll
    for (int j = 0; j < V; ++j) {
        float d;
        d = fmaxf(x.c[j].x - y.c[j].x, 0.f); s += (S)d * (S)d;
        d = fmaxf(x.c[j].y - y.c[j].y, 0.f); s += (S)d * (S)d;
        d = fmaxf(x.c[j].z - y.c[j].z, 0.f); s += (S)d * (S)d;
        d = fmaxf(x.c[j].w - y.c[j].w, 0.f); s += (S)d * (S)d;
    }
    return s;
}

__device__ __forceinline__ float4 axpby4(float a, float4 x, float b, float4 y) {
    return make_float4(fmaf(a, x.x, b * y.x), fmaf(a, x.y, b * y.y), fmaf(a, x.z, b * y.z), fmaf(a, x.w, b * y.w));
}
__device__ __forceinline__ void fma4(float4& acc, float a, float4 x) {
    acc.x = fmaf(a, x.x, acc.x); acc.y = fmaf(a, x.y, acc.y); acc.z = fmaf(a, x.z, acc.z); acc.w = fmaf(a, x.w, acc.w);
}
__device__ __forceinline__ float4 relu_diff4(float4 x, float4 y) {
    return make_float4(fmaxf(x.x - y.x, 0.f), fmaxf(x.y - y.y, 0.f), fmaxf(x.z - y.z, 0.f), fmaxf(x.w - y.w, 0.f));
}

// clamp(v, min=0) with torch semantics (NaN propagates; fmaxf would swallow it)
template <typename S>
__device__ __forceinline__ S relu_nan(S v) { return v < (S)0 ? (S)0 : v; }

// ------------------------------------------------------------------------------------------------
// Scalar cores.
//
// Everything that depends on ONE endpoint only (its squared norm, 1/norm, the half-aperture psi(x) and
// the aperture's contribution to dz/dx) is computed once per table row by lec_rows_fwd and stored as
// four doubles per row ("aux"); the per-pair cores below only do the genuinely pairwise algebra.
//   hyperbolic: aux = { |x|^2, 1/|x|, psi(x) = asin(clamp(K(1-|x|^2)/|x|)), -psi'(h) * dh/d|x|^2 * 2 }
//   Euclidean : aux = { |x|^2, 1/max(|x|,1e-12), sqrt(1 - K^2/|x|^2), K^2 / (|x|^4 sqrt(1 - K^2/|x|^2)) }
// Output of a pair core: raw z (energy before the outer max(0,.)), and the four coefficients of
// dz/dx = zxx*x + zxy*y, dz/dy = zyx*x + zyy*y.
// ------------------------------------------------------------------------------------------------
struct PairGrad {
    float z;
    float zxx, zxy, zyx, zyy;
};

template <typename S>
struct Aux {
    S A, ria, t0, t1;
};

template <typename S> __device__ __forceinline__ S s_sqrt(S v);
template <> __device__ __forceinline__ float s_sqrt<float>(float v) { return sqrtf(v); }
template <> __device__ __forceinline__ double s_sqrt<double>(double v) { return sqrt(v); }
template <typename S> __device__ __forceinline__ S s_rsqrt(S v);
template <> __device__ __forceinline__ float s_rsqrt<float>(float v) { return rsqrtf(v); }
template <> __device__ __forceinline__ double s_rsqrt<double>(double v) { return rsqrt(v); }
template <typename S> __device__ __forceinline__ S s_asin(S v);
template <> __device__ __forceinline__ float s_asin<float>(float v) { return asinf(v); }
template <> __device__ __forceinline__ double s_asin<double>(double v) { return asin(v); }

// a*b - c*d with both products rounded before the subtraction (no FMA contraction)
__device__ __forceinline__ float diff_of_products(float a, float b, float c, float d) {
    return __fsub_rn(__fmul_rn(a, b), __fmul_rn(c, d));
}
__device__ __forceinline__ double diff_of_products(double a, double b, double c, double d) {
    return __dsub_rn(__dmul_rn(a, b), __dmul_rn(c, d));
}

template <typename S>
__device__ __forceinline__ S clamp_eps(S v, bool& inside) {
    const S lo = (S)(-1.0 + 1e-5), hi = (S)(1.0 - 1e-5);
    inside = (v >= lo && v <= hi);               // torch.clamp passes the gradient on the closed interval
    return v < lo ? lo : (v > hi ? hi : v);      // NaN falls through unchanged, like torch.clamp
}

// per-row terms from A = |x|^2 (geom: LEC_GEOM_*)
template <typename S>
__device__ __forceinline__ Aux<S> row_aux(int geom, S A, float Kf) {
    Aux<S> o;
    const S K = (S)Kf, one = (S)1;
    o.A = A;
    if (geom == LEC_GEOM_HYP) {
        const S a = s_sqrt<S>(A);
        o.ria = one / a;
        bool in;
        const S hc = clamp_eps<S>(K * (one - A) / a, in);  // order_embeddings_h.py:1114
        o.t0 = s_asin<S>(hc);
        const S h_A = -K * (one + A) / ((S)2 * a * A);
        o.t1 = in ? -(one / s_sqrt<S>((one - hc) * (one + hc))) * h_A * (S)2 : (S)0;
    } else if (geom == LEC_GEOM_EUC) {
        const S a = s_sqrt<S>(A);
        o.ria = one / (a > (S)kNormEps ? a : (S)kNormEps);
        const S root = s_sqrt<S>(one - K * K / A);           // order_embeddings.py:967 (NaN when |x| < K)
        o.t0 = root;
        o.t1 = K * K / (A * A * root);
    } else {
        o.ria = o.t0 = o.t1 = (S)0;
    }
    return o;
}

// The same terms for the per-ROW producers (lec_rows_fwd, lec_update_rows), which run this once per table row inside
// a latency-bound kernel: reciprocal square roots instead of the sqrt / three divisions, and psi = asin(h) evaluated as
// atan2f(h, sqrt(1 - h^2)) with sqrt(1 - h^2) formed in fp64 -- atan2 is well conditioned where asin is not (asin' = 224
// at the clamp), so the fp32 evaluation keeps ~1e-7 absolute accuracy, which is all the pair kernels use of psi (they
// subtract it from an fp32 angle).  A = 0 / NaN behave as in row_aux.
__device__ __forceinline__ Aux<double> row_aux_fast(int geom, double A, float Kf) {
    Aux<double> o;
    const double K = (double)Kf;
    o.A = A;
    if (geom == LEC_GEOM_HYP) {
        const double rA = rsqrt(A);                                  // 1 / |x|
        o.ria = rA;
        bool in;
        const double hc = clamp_eps<double>(K * (1.0 - A) * rA, in);  // order_embeddings_h.py:1114
        const double q = (1.0 - hc) * (1.0 + hc);
        const double rq = rsqrt(q);                                  // 1 / sqrt(1 - h^2)
        o.t0 = (double)atan2f((float)hc, (float)(q * rq));
        const double h_A = -0.5 * K * (1.0 + A) * rA * rA * rA;       // dh / d|x|^2
        o.t1 = in ? -rq * h_A * 2.0 : 0.0;
    } else if (geom == LEC_GEOM_EUC) {
        const double rA = rsqrt(A);
        o.ria = A * rA > (double)kNormEps ? rA : 1.0 / (double)kNormEps;
        const double q = 1.0 - K * K * rA * rA;                      // order_embeddings.py:967 (NaN when |x| < K)
        o.t0 = sqrt(q);
        o.t1 = K * K * rA * rA * rA * rA * rsqrt(q);
    } else {
        o.ria = o.t0 = o.t1 = 0.0;
    }
    return o;
}

template <typename S>
__device__ __forceinline__ Aux<S> load_aux(const double* __restrict__ aux, int64_t row) {
    const double2 p0 = __ldg(reinterpret_cast<const double2*>(aux + 4 * row));
    const double2 p1 = __ldg(reinterpret_cast<const double2*>(aux + 4 * row) + 1);
    Aux<S> o;
    o.A = (S)p0.x; o.ria = (S)p0.y; o.t0 = (S)p1.x; o.t1 = (S)p1.y;
    return o;
}
template <typename S>
__device__ __forceinline__ S load_aux_A(const double* __restrict__ aux, int64_t row) {
    return (S)__ldg(aux + 4 * row);
}

// Euclidean cone, cos-space (order_embeddings.py:954-969).  x = apex with aux ax; DD=<d,d>, XD=<x,d>, d=y-x.
template <typename S, bool GRAD>
__device__ __forceinline__ void euc_pair(const Aux<S>& ax, S DD, S XD, PairGrad& o) {
    const S b = s_sqrt<S>(DD);
    const S rb = (S)1 / (b > (S)kNormEps ? b : (S)kNormEps);
    const S inv_ab = ax.ria * rb;
    const S c = XD * inv_ab;
    o.z = (float)(ax.t0 - c);
    if (GRAD) {
        const S c_b2 = c * rb * rb;
        const S m = -inv_ab - c_b2;  // coefficient of x in dz/dy (and of y in dz/dx)
        o.zyx = (float)m;
        o.zyy = (float)c_b2;
        o.zxy = (float)m;
        o.zxx = (float)((S)2 * inv_ab + c * ax.ria * ax.ria + c_b2 + ax.t1);
    }
}

// Poincare cone (order_embeddings_h.py:1097-1120).  x = apex with aux ax; B=<y,y>, P=<x,y>, S2=|x-y|^2.
// One reciprocal square root of A*S2*w2 yields 1/den and, by multiplication, 1/w2 and 1/S2.
template <typename S, bool GRAD>
__device__ __forceinline__ void hyp_pair(const Aux<S>& ax, S B, S P, S S2, PairGrad& o) {
    const S one = (S)1;
    const S A = ax.A;
    const S w2 = one + A * B - (S)2 * P;
    const S AS = A * S2;
    const S rden = s_rsqrt<S>(AS * w2);
    // identical endpoints: the reference evaluates 0/0 here (NaN up to the rounding of its norms); we
    // return NaN deterministically.  A zero apex row gives 0 * inf = NaN by itself (SURVEY F9).
    const S g = (S2 == (S)0) ? (S)NAN : diff_of_products(P, one + A, A, one + B) * rden;
    bool in;
    const S gc = clamp_eps<S>(g, in);
    const S tg = (one - gc) * (one + gc);
    const S rsg = s_rsqrt<S>(tg);
    float theta;
    if (sizeof(S) == 8) theta = atan2f((float)(tg * rsg), (float)gc);  // angle from (sin, cos), both accurate
    else theta = acosf((float)gc);
    o.z = theta - (float)ax.t0;
    if (GRAD) {
        const S th = in ? -rsg : (S)0;  // d acos(clamp(g)) / dg
        const S rden2 = rden * rden;
        const S inv_w2 = rden2 * AS;
        const S inv_S2 = rden2 * A * w2;
        const S g_p = (one + A) * rden + g * inv_w2;
        const S g_A2 = (S)2 * (P - one - B) * rden - g * (ax.ria * ax.ria + B * inv_w2);  // 2 * dg/dA
        const S g_B2 = (S)-2 * A * rden - g * A * inv_w2;                                 // 2 * dg/dB
        const S gs = -g * inv_S2;                                                          // (dg/ds)/s
        const S cross = th * (g_p - gs);
        o.zxx = (float)(th * (g_A2 + gs) + ax.t1);
        o.zxy = (float)cross;
        o.zyx = (float)cross;
        o.zyy = (float)(th * (g_B2 + gs));
    }
}

// hinge: returns d loss / d z and adds this pair's loss term
//   positive: w*E            -> w*[z>=0]
//   negative: w*max(0,a-E)   -> -w*[a-E>=0]*[z>=0]
__device__ __forceinline__ float hinge(float z, bool is_pos, float w, float alpha, float& E, double& loss) {
    E = relu_nan(z);
    const float act = (z >= 0.f) ? 1.f : 0.f;
    if (is_pos) {
        loss += (double)(w * E);
        return w * act;
    }
    const float m = alpha - E;
    loss += (double)(w * relu_nan(m));
    return (m >= 0.f) ? -w * act : 0.f;
}

template <int IDXB>
__device__ __forceinline__ int64_t load_idx(const void* p, int64_t i) {
    if (IDXB == 4) return (int64_t) __ldg(reinterpret_cast<const int32_t*>(p) + i);
    return (int64_t) __ldg(reinterpret_cast<const long long*>(p) + i);
}

// block-level double sum -> one atomic per block
__device__ __forceinline__ void block_add_double(double v, double* out) {
    __shared__ double warp_part[kThreads / 32];
    v = warp_sum<double>(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) warp_part[wid] = v;
    __syncthreads();
    if (wid == 0) {
        double t = (lane < (blockDim.x >> 5)) ? warp_part[lane] : 0.0;
        t = warp_sum<double>(t);
        if (lane == 0 && out != nullptr && t != 0.0) atomicAdd(out, t);
    }
}

// Optional phase trace of a training step (build with -DLEC_STEP_TRACE): the kernels of a step stamp %globaltimer into
// a small device array (min / max over blocks), read and reset by lec_debug_step_trace (scripts/step_trace.py).
//   [0] min pair kernel past its dependency wait   [1] max pair kernel block end
//   [2] min update kernel past its dependency wait [3] max ... [4] max packets pushed [5] max packets reduced [6] max end
#ifdef LEC_STEP_TRACE
extern unsigned long long* g_step_trace;   // device pointer, NULL until the debug entry point allocates it
__device__ __forceinline__ unsigned long long trace_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void trace_min(unsigned long long* tr, int slot) { if (tr) atomicMin(tr + slot, trace_now()); }
__device__ __forceinline__ void trace_max(unsigned long long* tr, int slot) { if (tr) atomicMax(tr + slot, trace_now()); }
#define LEC_TRACE_MIN(tr, slot) trace_min(tr, slot)
#define LEC_TRACE_MAX(tr, slot) trace_max(tr, slot)
#else
#define LEC_TRACE_MIN(tr, slot)
#define LEC_TRACE_MAX(tr, slot)
#endif

inline int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

}  // namespace lec
