// Fused table update: everything a training step does to the parameter table between the pair kernel and the next
// step's pair kernel, in ONE launch, one team of TT lanes per table row, the row held in registers as V float4 chunks
// per lane (chunk q = lane + TT*j, the layout of the transformed table):
//
//   1. sum of the row's gradient replicas (d loss / d rows, scattered by the pair kernel), replicas cleared
//   2. world > 1: one-shot all-reduce of that row over NVLink / NVSwitch peer memory, low-latency protocol: every rank
//      stores its partial row into its source region of EVERY rank's exchange buffer as 16-byte packets
//      {value, tag, value, tag} (8-byte halves are written atomically, so the tag IS the arrival flag: no fence, no
//      separate flag store, one NVLink one-way latency), then polls its OWN buffer until the `world` packets of the chunk
//      carry this step's tag and adds them in rank order (identical bits on every rank)
//   3. vector-Jacobian product of the row transform (Embedder.forward): d loss / d table
//   4. the update rule on the raw row: Riemannian SGD (order_embeddings_h.py:764-775), SGD with momentum or Adam
//      (torch.optim, order_embeddings.py:563-565), Nickel & Kiela's rescaled step + retraction (Poincare embeddings) or
//      exponential map on the hyperboloid (Lorentz embeddings), optionally preceded by the conformal rescale ((1-|w|)/2)^2 and followed
//      by the shell projection of the joint hyperbolic trainer (oe_h.py:1765-1771)
//   5. the row transform of the UPDATED row -- the Embedder.forward the next iteration starts with -- and its per-row
//      aperture terms (aux), so the next pair kernel can start right away
//
// 12*D bytes per row at least (read w, read g, write w); with the fused transform ~24*D (+ optimizer state).
#include "lec_rowops.cuh"

#ifndef LEC_UPD_MINBLOCKS
#define LEC_UPD_MINBLOCKS 3   // resident 256-thread blocks per SM the specialised kernels are compiled for (register cap 80)
#endif

namespace lec {

struct UpdArgs {
    int rule, row_mode, geom, lambda_mode, hyp_rescale, project_shell;
    float K, lr, r_in, r_in_rows, c0;
    float momentum, beta1, beta2, eps, step_size, inv_bc2_sqrt;
    float* table; int64_t n; int D; int ld; int tv;   // tv: widest aligned vector access of a raw table row (4, 2, 1 floats)
    float* grad_rows; int replicas; int64_t replica_stride;
    float* m; float* v;
    float* rows_out; double* aux_out; float* grad_out;
    double* loss_acc; double* loss_step;
    int world, rank, slot; unsigned tag; int64_t slot_packets; uint4* peer[kMaxPeers];
    double* loss_global; int* error; unsigned long long timeout_ns;
    // two-shot exchange (large tables): rank r owns rows [r * rows_per_rank, (r + 1) * rows_per_rank)
    int64_t rows_per_rank; int tiles_per_rank; int phases;
    unsigned long long* trace;   // LEC_STEP_TRACE builds only
};

// ---- two-shot exchange: layout of one rank's buffer --------------------------------------------------------------------
//   float rs[2][world][rows_per_rank * ld]   partial gradients of MY rows, one region per source rank   (reduce-scatter)
//   float ag[2][world * rows_per_rank * ld]  updated raw rows of every OTHER owner, padded row layout    (all-gather)
//   u32   rs_flag[2][world][tiles_per_rank]  tag of the step whose partial tile has arrived
//   u32   ag_flag[2][world * tiles_per_rank] tag of the step whose updated tile has arrived
//   uint4 loss[2][world]                     loss packets
// A tile is the kThreads / TT rows one block handles per iteration; rows_per_rank is a whole number of tiles.
struct TwoShot {
    int64_t rs_floats, ag_floats, flag_words;   // per slot
    __host__ __device__ TwoShot(int world, int64_t rows_per_rank, int tiles_per_rank, int ld) {
        rs_floats = (int64_t)world * rows_per_rank * ld;
        ag_floats = rs_floats;
        flag_words = (int64_t)world * tiles_per_rank;
    }
    __host__ __device__ int64_t bytes(int world) const {
        return (2 * (rs_floats + ag_floats)) * 4 + ((2 * 2 * flag_words * 4 + 15) / 16) * 16 + 2 * (int64_t)world * 16;
    }
    __host__ __device__ float* rs(uint4* base, int slot) const { return reinterpret_cast<float*>(base) + slot * rs_floats; }
    __host__ __device__ float* ag(uint4* base, int slot) const { return reinterpret_cast<float*>(base) + 2 * rs_floats + slot * ag_floats; }
    __host__ __device__ unsigned* rs_flag(uint4* base, int slot) const {
        return reinterpret_cast<unsigned*>(reinterpret_cast<float*>(base) + 2 * (rs_floats + ag_floats)) + slot * flag_words;
    }
    __host__ __device__ unsigned* ag_flag(uint4* base, int slot) const { return rs_flag(base, 0) + 2 * flag_words + slot * flag_words; }
    __host__ __device__ uint4* loss(uint4* base, int slot, int world) const {
        return reinterpret_cast<uint4*>(reinterpret_cast<char*>(base) + (2 * (rs_floats + ag_floats)) * 4 +
                                        ((2 * 2 * flag_words * 4 + 15) / 16) * 16) + slot * world;
    }
};

// ---- low-latency packets -------------------------------------------------------------------------------------------
__device__ __forceinline__ void ll_store(uint4* p, unsigned a, unsigned b, unsigned tag) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(tag), "r"(b), "r"(tag) : "memory");
}
__device__ __forceinline__ uint4 ll_load(const uint4* p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_volatile_int(const int* p) {
    int v;
    asm volatile("ld.volatile.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// waits until *flag == tag; false (and *error raised) on timeout or when the exchange already failed elsewhere
__device__ __forceinline__ bool flag_wait(const unsigned* flag, unsigned tag, int* error, unsigned long long timeout_ns,
                                          unsigned long long& t0) {
    unsigned spins = 0;
    while (ld_acquire_sys(flag) != tag) {
        if ((++spins & 255u) == 0) {
            if (t0 == 0) t0 = global_ns();
            if ((error && ld_volatile_int(error) != 0) || global_ns() - t0 > timeout_ns) {
                if (error) atomicExch(error, 1);
                return false;
            }
        }
    }
    return true;
}

// Spins until the packet at p carries `tag` in both halves.  Returns false (and raises *error) when the peer does not
// deliver within timeout_ns, or when another thread already raised *error: the caller then drops the row's update.
__device__ __forceinline__ bool ll_wait(const uint4* p, unsigned tag, uint4& pk, int* error, unsigned long long timeout_ns,
                                        unsigned long long& t0) {
    unsigned spins = 0;
    while (pk.y != tag || pk.w != tag) {
        pk = ll_load(p);
        if ((++spins & 1023u) == 0) {
            if (t0 == 0) t0 = global_ns();
            if ((error && ld_volatile_int(error) != 0) || global_ns() - t0 > timeout_ns) {
                if (error) atomicExch(error, 1);
                return false;
            }
        }
    }
    return true;
}

// my partial chunk -> source region `rank` of every rank's buffer
__device__ __forceinline__ void ll_push_chunk(const UpdArgs& a, int64_t packet, float4 g) {
    const int64_t off = ((int64_t)a.slot * a.world + a.rank) * a.slot_packets + packet;
    for (int p = 0; p < a.world; ++p) {
        uint4* dst = a.peer[p] + off;
        ll_store(dst, __float_as_uint(g.x), __float_as_uint(g.y), a.tag);
        ll_store(dst + 1, __float_as_uint(g.z), __float_as_uint(g.w), a.tag);
    }
}

// sum over the ranks, in rank order, of the chunk at `packet` of my own buffer.  Up to eight sources (16 packets) are
// polled together: every round re-issues the loads of ALL packets that have not arrived yet and only then looks at
// them, so a round costs one L2 round trip however many packets are outstanding (polling them one after the other
// costs one round trip EACH, which at eight ranks is longer than the NVLink latency the protocol is built to hide).
__device__ __forceinline__ bool ll_reduce_chunk(const UpdArgs& a, int64_t packet, float4& out, unsigned long long& t0) {
    const uint4* mine = a.peer[a.rank] + (int64_t)a.slot * a.world * a.slot_packets + packet;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    bool ok = true;
    for (int p0 = 0; p0 < a.world && ok; p0 += 8) {
        const int cnt = a.world - p0 < 8 ? a.world - p0 : 8;
        uint4 pk[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (i < cnt) {
                const uint4* src = mine + (int64_t)(p0 + i) * a.slot_packets;
                pk[2 * i] = ll_load(src);
                pk[2 * i + 1] = ll_load(src + 1);
            }
        }
        unsigned rounds = 0;
        while (true) {
            bool all = true;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (i < cnt) {
                    const uint4* src = mine + (int64_t)(p0 + i) * a.slot_packets;
                    if (pk[2 * i].y != a.tag || pk[2 * i].w != a.tag) { pk[2 * i] = ll_load(src); all = false; }
                    if (pk[2 * i + 1].y != a.tag || pk[2 * i + 1].w != a.tag) { pk[2 * i + 1] = ll_load(src + 1); all = false; }
                }
            }
            if (all) break;
            if ((++rounds & 255u) == 0) {
                if (t0 == 0) t0 = global_ns();
                if ((a.error && ld_volatile_int(a.error) != 0) || global_ns() - t0 > a.timeout_ns) {
                    if (a.error) atomicExch(a.error, 1);
                    ok = false;
                    break;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (i < cnt) {
                acc.x += __uint_as_float(pk[2 * i].x); acc.y += __uint_as_float(pk[2 * i].z);
                acc.z += __uint_as_float(pk[2 * i + 1].x); acc.w += __uint_as_float(pk[2 * i + 1].z);
            }
        }
    }
    out = acc;
    return ok;
}

// ---- raw table rows (row stride D floats, so only D % 4 == 0 rows are 16-byte aligned) ------------------------------
template <int TT, int V>
__device__ __forceinline__ void load_raw(float (&e)[4 * V], const float* __restrict__ w, int D, int lane, int tv) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int d0 = 4 * (lane + TT * j);
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (d0 < D) {
            if (tv == 4) {
                x = *reinterpret_cast<const float4*>(w + d0);
            } else if (tv == 2) {
                const float2 lo = *reinterpret_cast<const float2*>(w + d0);
                x.x = lo.x; x.y = lo.y;
                if (d0 + 2 < D) { const float2 hi = *reinterpret_cast<const float2*>(w + d0 + 2); x.z = hi.x; x.w = hi.y; }
            } else {
                x.x = w[d0];
                if (d0 + 1 < D) x.y = w[d0 + 1];
                if (d0 + 2 < D) x.z = w[d0 + 2];
                if (d0 + 3 < D) x.w = w[d0 + 3];
            }
        }
        e[4 * j] = x.x; e[4 * j + 1] = x.y; e[4 * j + 2] = x.z; e[4 * j + 3] = x.w;
    }
}

template <int TT, int V>
__device__ __forceinline__ void store_raw(float* __restrict__ w, const float (&e)[4 * V], int D, int lane, int tv) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int d0 = 4 * (lane + TT * j);
        if (d0 < D) {
            if (tv == 4) {
                *reinterpret_cast<float4*>(w + d0) = make_float4(e[4 * j], e[4 * j + 1], e[4 * j + 2], e[4 * j + 3]);
            } else if (tv == 2) {
                *reinterpret_cast<float2*>(w + d0) = make_float2(e[4 * j], e[4 * j + 1]);
                if (d0 + 2 < D) *reinterpret_cast<float2*>(w + d0 + 2) = make_float2(e[4 * j + 2], e[4 * j + 3]);
            } else {
                w[d0] = e[4 * j];
                if (d0 + 1 < D) w[d0 + 1] = e[4 * j + 1];
                if (d0 + 2 < D) w[d0 + 2] = e[4 * j + 2];
                if (d0 + 3 < D) w[d0 + 3] = e[4 * j + 3];
            }
        }
    }
}

// padded [n, ld] buffers (optimizer state, transformed rows): whole float4 chunks
template <int TT, int V>
__device__ __forceinline__ void load_chunks(float (&x)[4 * V], const float* __restrict__ p, int Q, int lane) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int q = lane + TT * j;
        const float4 c = q < Q ? *reinterpret_cast<const float4*>(p + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        x[4 * j] = c.x; x[4 * j + 1] = c.y; x[4 * j + 2] = c.z; x[4 * j + 3] = c.w;
    }
}
template <int TT, int V>
__device__ __forceinline__ void store_chunks(float* __restrict__ p, const float (&x)[4 * V], int Q, int lane) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
        const int q = lane + TT * j;
        if (q < Q) *reinterpret_cast<float4*>(p + 4 * q) = make_float4(x[4 * j], x[4 * j + 1], x[4 * j + 2], x[4 * j + 3]);
    }
}

template <int TT, int V>
__device__ __forceinline__ float sumsq32(const float (&x)[4 * V]) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 4 * V; ++i) s = fmaf(x[i], x[i], s);
    return team_sum<TT, float>(s);
}

// ---- steps 3 + 4 for one row held by a team: VJP of the row transform, update rule; e becomes the new raw row (and is
//      stored to the table when valid), the optimizer state is advanced ------------------------------------------------
template <int TT, int V, int RULE_T>
__device__ __forceinline__ void row_rule(const UpdArgs& a, const int rule, const int row_mode, float (&g)[4 * V], float (&e)[4 * V],
                                         float (&mb)[4 * V], float (&vb)[4 * V], const int64_t row, const int64_t rc,
                                         const bool valid, const int lane) {
    const int D = a.D, Q = a.ld >> 2;
    const bool sgd_m = rule == LEC_UPD_SGD && a.m && a.momentum != 0.f;
    float* const w = a.table + rc * (int64_t)D;
    // ---- 3. raw row, VJP of the row transform: g <- d loss / d table ---------------------------------------------
    if (row_mode == LEC_ROWS_EUC_SOFTCLIP) {
        // out = e/|e| * (|e| + K)  (order_embeddings.py:195-200):  J^T g = (1 + K/r) g - K <e,g> / r^3 e
        float ss = 0.f, eg = 0.f;
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) { ss = fmaf(e[i], e[i], ss); eg = fmaf(e[i], g[i], eg); }
        ss = team_sum<TT, float>(ss); eg = team_sum<TT, float>(eg);
        const float r = sqrtf(ss);
        const float c_g = 1.f + a.K / r, c_e = -a.K * eg / (r * ss);
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) g[i] = fmaf(c_e, e[i], c_g * g[i]);
    } else if (row_mode == LEC_ROWS_HYP_TANH) {
        // out = tanh(clamp(c0 + r)) e'/r, e' = e + 1e-15 (oe_h.py:77-104); the projection behind it is straight-through
        float ss = 0.f, eg = 0.f;
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) {
            const int d = 4 * (lane + TT * (i >> 2)) + (i & 3);
            const float ev = d < D ? e[i] + 1e-15f : 0.f;
            ss = fmaf(ev, ev, ss); eg = fmaf(ev, g[i], eg);
        }
        ss = team_sum<TT, float>(ss); eg = team_sum<TT, float>(eg);
        const float r = sqrtf(ss);
        const float arg = a.c0 + r;
        const float t = tanhf(fminf(fmaxf(arg, -15.f), 15.f));
        const float tp = (arg >= -15.f && arg <= 15.f) ? (1.f - t * t) : 0.f;
        const float c_g = t / r, c_e = (tp - t / r) * eg / ss;
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) {
            const int d = 4 * (lane + TT * (i >> 2)) + (i & 3);
            g[i] = d < D ? fmaf(c_e, e[i] + 1e-15f, c_g * g[i]) : 0.f;
        }
    }
    // ---- 4. update rule ------------------------------------------------------------------------------------------
    if (RULE_T == LEC_UPD_RSGD_RETRACT) {
        // Nickel & Kiela (eq. 5-7): w <- proj(w - lr (1 - |w|^2)^2 / 4 g), proj: |w| >= 1 - 1e-5 -> norm 1 - 1e-5.  Only
        // this compile-time specialisation holds the rule (the generic kernels never see it; row_mode is NONE)
        double uu = 0.0;
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) uu = fma((double)e[i], (double)e[i], uu);
        uu = team_sum<TT, double>(uu);
        const double om = 1.0 - uu;
        const float gs = (float)(0.25 * om * om);
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) g[i] *= gs;                       // the Riemannian gradient
        if (valid && a.grad_out) store_raw<TT, V>(a.grad_out + row * (int64_t)D, g, D, lane, a.tv);
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) e[i] = fmaf(-a.lr, g[i], e[i]);
        double nn = 0.0;
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) nn = fma((double)e[i], (double)e[i], nn);
        const double nrm = sqrt(team_sum<TT, double>(nn));
        constexpr double kMaxNorm = 1.0 - 1e-5;
        if (nrm >= kMaxNorm) {
            const float sc = (float)(kMaxNorm / nrm);
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) e[i] *= sc;
        }
    } else if (RULE_T == LEC_UPD_RSGD_LORENTZ) {
        // Nickel & Kiela 2018: the exponential map on the hyperboloid along -lr times the Riemannian gradient, in the
        // spatial chart (include/lec_b200.h): c = <x,g>, r = g + c x, nu = sqrt(|g|^2 + c^2), t = lr nu,
        // x <- cosh(t) x - lr sinh(t)/t r.  Only this compile-time specialisation holds the rule (row_mode is NONE)
        double xg = 0.0, gg = 0.0;
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) {
            xg = fma((double)e[i], (double)g[i], xg);
            gg = fma((double)g[i], (double)g[i], gg);
        }
        xg = team_sum<TT, double>(xg);
        gg = team_sum<TT, double>(gg);
        const double nu = sqrt(fma(xg, xg, gg));
        const double t = (double)a.lr * nu;
        // cosh(t) and sinh(t) from one expm1: E = e^t = 1 + m, cosh = 1 + m^2 / 2E, sinh = m (m + 2) / 2E (no cancellation
        // as t -> 0, where sinh(t) / t -> 1)
        const double m = expm1(t), ie = 0.5 / (1.0 + m);
        const double ch = fma(m * m, ie, 1.0);
        const double sh = t > 0.0 ? (double)a.lr * (m * (m + 2.0) * ie / t) : (double)a.lr;   // lr sinh(t) / t
        if (valid && a.grad_out) {
            float r[4 * V];
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) r[i] = (float)fma(xg, (double)e[i], (double)g[i]);
            store_raw<TT, V>(a.grad_out + row * (int64_t)D, r, D, lane, a.tv);
        }
        if (nu > 0.0) {
            const double ce = fma(-sh, xg, ch);   // x <- (cosh(t) - lr sinh(t)/t c) x - lr sinh(t)/t g
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) e[i] = (float)fma(ce, (double)e[i], -sh * (double)g[i]);
        }
    } else if (rule == LEC_UPD_RSGD) {
        // One pass gives the five row sums every later quantity is an algebraic function of (v = -lr gs g + 1e-15,
        // t = th v/|v| + 1e-6, the Moebius sums <w,t>, |t|^2 and the norm of the result), carried in fp64:
        double uu = 0.0, gg = 0.0, eg = 0.0, se = 0.0, sg = 0.0;
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) {
            const double ed = (double)e[i], gd = (double)g[i];
            uu = fma(ed, ed, uu); gg = fma(gd, gd, gg); eg = fma(ed, gd, eg); se += ed; sg += gd;
        }
        uu = team_sum<TT, double>(uu); gg = team_sum<TT, double>(gg); eg = team_sum<TT, double>(eg);
        se = team_sum<TT, double>(se); sg = team_sum<TT, double>(sg);
        // conformal factor (order_embeddings_h.py:662-666; SURVEY F4: the norm, not its square): 1/lambda = (1 - |w|) / 2.
        // Only the cancelling quantities (1 - |w|, 1 - |w|^2, the Moebius denominator) need fp64; square roots and
        // quotients whose results end up as fp32 coefficients are taken in fp32 (as the reference takes all of them).
        const float wn = (float)sqrt(uu);
        const float inv = 0.5f * (1.f - (a.lambda_mode == 1 ? (float)uu : wn));
        const float gs = inv * inv;
        const double Dn = (double)D, e15 = 1e-15, e6 = 1e-6;
        const double av = -(double)a.lr * (double)gs;                     // v_d = av g_d + 1e-15
        const double vv = av * av * gg + 2.0 * av * e15 * sg + Dn * e15 * e15;
        const float vn = sqrtf((float)vv);
        const float th = tanhf(fminf(fmaxf(0.5f * vn / inv, -15.f), 15.f));   // lambda |v| / 2
        const double c = (double)(th / vn);
        const double al = c * av, be = c * e15 + e6;                      // t_d = al g_d + be
        const double tt = al * al * gg + 2.0 * al * be * sg + Dn * be * be;
        const double uv2 = 2.0 * (al * eg + be * se);
        const double den = 1.0 + uv2 + tt * uu;
        const double rden = (double)(1.f / (float)den);
        const double cw = (1.0 + uv2 + tt) * rden, ct = (1.0 - uu) * rden;
        const double cg = ct * al, cb = ct * be;                          // res_d = cw e_d + cg g_d + cb
        const double rr = cw * cw * uu + cg * cg * gg + Dn * cb * cb + 2.0 * (cw * cg * eg + cw * cb * se + cg * cb * sg);
        float mul, add, div;
        shell_factor(sqrtf((float)rr), a.r_in, false, mul, add, div);
        const float sc = (mul != 1.f || div != 1.f) ? mul / div : 1.f;
        const float f_w = (float)cw * sc, f_g = (float)cg * sc, f_b = (float)cb * sc;
        float* go = (valid && a.grad_out) ? a.grad_out + row * (int64_t)D : nullptr;
        if (go) {
            float rg[4 * V];
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) rg[i] = g[i] * gs;            // the Riemannian gradient, as left in weight.grad
            store_raw<TT, V>(go, rg, D, lane, a.tv);
        }
#pragma unroll
        for (int i = 0; i < 4 * V; ++i) {
            const int d = 4 * (lane + TT * (i >> 2)) + (i & 3);
            e[i] = d < D ? fmaf(f_w, e[i], fmaf(f_g, g[i], f_b)) : 0.f;
        }
    } else {
        if (a.hyp_rescale) {
            // Euclidean -> Riemannian gradient of the joint hyperbolic trainer: grad *= (1/lambda_x(w))^2, oe_h.py:1766
            const float wn = sqrtf(sumsq32<TT, V>(e));
            const float inv = (1.f - wn) * 0.5f;
            const float gs = inv * inv;
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) g[i] *= gs;
        }
        if (valid && a.grad_out) store_raw<TT, V>(a.grad_out + row * (int64_t)D, g, D, lane, a.tv);
        if (rule == LEC_UPD_SGD) {
            // torch.optim.SGD: buf = momentum * buf + g (buf starts at 0, which equals its first-step rule); p -= lr * buf
            if (sgd_m) {
#pragma unroll
                for (int i = 0; i < 4 * V; ++i) { mb[i] = fmaf(a.momentum, mb[i], g[i]); g[i] = mb[i]; }
                if (valid) store_chunks<TT, V>(a.m + rc * (int64_t)a.ld, mb, Q, lane);
            }
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) e[i] = fmaf(-a.lr, g[i], e[i]);
        } else if (rule == LEC_UPD_ADAM) {
            // torch.optim.Adam (_single_tensor_adam, no amsgrad / weight decay):
            //   m.lerp_(g, 1-b1); v = v*b2 + (1-b2) g g; p += -(lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
            float* mp = a.m + rc * (int64_t)a.ld;
            float* vp = a.v + rc * (int64_t)a.ld;
            const float w1 = 1.f - a.beta1, w2 = 1.f - a.beta2;
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) {
                mb[i] = fmaf(w1, g[i] - mb[i], mb[i]);
                vb[i] = fmaf(w2 * g[i], g[i], __fmul_rn(vb[i], a.beta2));
                const float den = sqrtf(vb[i]) * a.inv_bc2_sqrt + a.eps;
                e[i] = fmaf(-a.step_size, mb[i] / den, e[i]);
            }
            if (valid) { store_chunks<TT, V>(mp, mb, Q, lane); store_chunks<TT, V>(vp, vb, Q, lane); }
        }
        if (a.project_shell) {
            // soft_clip on the table itself (oe_h.py:1604-1618, called at :1771): |w| <= r_in -> r_in, |w| >= 1 -> 1 - 1e-5
            float mul, add, div;
            shell_factor(sqrtf(sumsq32<TT, V>(e)), a.r_in, false, mul, add, div);
            if (mul != 1.f || div != 1.f) {
#pragma unroll
                for (int i = 0; i < 4 * V; ++i) e[i] = (e[i] / div) * mul;
            }
        }
    }
    if (valid && rule != LEC_UPD_NONE) store_raw<TT, V>(w, e, D, lane, a.tv);
}

// ---- step 5: Embedder.forward of the (updated) raw row e -> rows_out, |row|^2 parked for the batched aperture terms ----
template <int TT, int V>
__device__ __forceinline__ void row_forward(const UpdArgs& a, const int row_mode, float (&e)[4 * V], const int64_t row,
                                            const bool valid, const int lane) {
    const int D = a.D, Q = a.ld >> 2;
    const bool hyp = row_mode >= LEC_ROWS_HYP_SHELL;
    // ---- 5. Embedder.forward of the updated row + its aperture terms ---------------------------------------------
    if (a.rows_out) {
        if (hyp) {
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) {
                const int d = 4 * (lane + TT * (i >> 2)) + (i & 3);
                e[i] = d < D ? __fadd_rn(e[i], 1e-15f) : 0.f;
            }
        }
        if (row_mode != LEC_ROWS_NONE) {
            const float r = sqrtf(sumsq32<TT, V>(e));
            if (row_mode == LEC_ROWS_EUC_SOFTCLIP) {
                const float rn = fmaxf(r, kNormEps), scale = r + a.K;
#pragma unroll
                for (int i = 0; i < 4 * V; ++i) e[i] = (e[i] / rn) * scale;
            } else {
                float r2 = r;
                if (row_mode != LEC_ROWS_HYP_SHELL) {
                    const float rn = fmaxf(r, kNormEps);
                    const float scale = tanhf(fminf(fmaxf(a.c0 + r, -15.f), 15.f));
#pragma unroll
                    for (int i = 0; i < 4 * V; ++i) e[i] = scale * (e[i] / rn);
                    r2 = sqrtf(sumsq32<TT, V>(e));
                }
                float mul, add, div;
                shell_factor(r2, a.r_in_rows, false, mul, add, div);
                if (mul != 1.f || div != 1.f) {
#pragma unroll
                    for (int i = 0; i < 4 * V; ++i) {
                        const int d = 4 * (lane + TT * (i >> 2)) + (i & 3);
                        e[i] = d < D ? __fmul_rn((add + e[i]) / div, mul) : 0.f;
                    }
                }
            }
        }
        if (valid) store_chunks<TT, V>(a.rows_out + row * (int64_t)a.ld, e, Q, lane);
        if (a.aux_out) {
            double A = 0.0;
#pragma unroll
            for (int i = 0; i < 4 * V; ++i) A = fma((double)e[i], (double)e[i], A);
            A = team_sum<TT, double>(A);
            // the aperture terms of the row, by every lane of its team (rsqrt-based: ~90 issue slots, no block barrier)
            const Aux<double> x = row_aux_fast(a.geom, A, a.K);
            if (valid && lane == 0) {
                double2* dst = reinterpret_cast<double2*>(a.aux_out + 4 * row);
                dst[0] = make_double2(x.A, x.ria);
                dst[1] = make_double2(x.t0, x.t1);
            }
        }
    }
}

// RULE_T / MODE_T >= 0 fix the update rule / row transform at compile time (the hot combinations get their own, much
// smaller, instruction stream); -1 reads them from the arguments.  The Lorentz rule's fp64 expm1 does not fit the
// register cap of LEC_UPD_MINBLOCKS (28 bytes of spill at 80 registers with four chunks per lane): it gets two blocks.
template <int V, bool XCHG, int RULE_T>
constexpr int kUpdMinBlocks =
    (V <= 4 && !XCHG && RULE_T >= 0) ? (RULE_T == LEC_UPD_RSGD_LORENTZ ? 2 : LEC_UPD_MINBLOCKS) : 1;

template <int TT, int V, bool XCHG, int RULE_T, int MODE_T>
__global__ void __launch_bounds__(kThreads, (kUpdMinBlocks<V, XCHG, RULE_T>)) update_rows_kernel(const UpdArgs a) {
    const int rule = RULE_T >= 0 ? RULE_T : a.rule;
    const int row_mode = MODE_T >= 0 ? MODE_T : a.row_mode;
    pdl_launch_dependents();
    pdl_wait();   // the pair kernel's reductions into the replicas (and its loss) are complete
    if (threadIdx.x == 0) { LEC_TRACE_MIN(a.trace, 2); LEC_TRACE_MAX(a.trace, 3); }
    // an earlier exchange failed: the table is left alone.  The flag is READ here but tested only after the row's loads
    // have been issued (below), so that its latency overlaps theirs instead of preceding them.
    const int failed_before = (XCHG && a.error) ? ld_volatile_int(a.error) : 0;
    const int lane = threadIdx.x % TT;
    const int tpb_rt = (int)blockDim.x / TT;   // the launcher picks the block size: small tables use small blocks on many SMs
    const int64_t n_teams = (int64_t)gridDim.x * tpb_rt;
    const int64_t team = (int64_t)blockIdx.x * tpb_rt + threadIdx.x / TT;
    const int64_t iters = (a.n + n_teams - 1) / n_teams;
    const int D = a.D, Q = a.ld >> 2;
    unsigned long long t0 = 0;
    double my_loss = 0.0;
    const bool loss_thread = blockIdx.x == 0 && threadIdx.x == 0;
    if (loss_thread && a.loss_acc) my_loss = *a.loss_acc;
    if (XCHG && blockIdx.x == 0 && (int)threadIdx.x < a.world && a.loss_acc) {
        // this rank's loss of the step travels as one more packet of its source region
        const double l = *a.loss_acc;
        const unsigned long long bits = (unsigned long long)__double_as_longlong(l);
        uint4* dst = a.peer[threadIdx.x] + ((int64_t)a.slot * a.world + a.rank) * a.slot_packets + a.n * (int64_t)Q * 2;
        ll_store(dst, (unsigned)(bits & 0xffffffffu), (unsigned)(bits >> 32), a.tag);
    }
    const bool hyp = row_mode >= LEC_ROWS_HYP_SHELL;
    const bool adam = rule == LEC_UPD_ADAM;
    const bool sgd_m = rule == LEC_UPD_SGD && a.m && a.momentum != 0.f;
    for (int64_t it = 0; it < iters; ++it) {
        const int64_t row = team + it * n_teams;
        bool valid = row < a.n;
        const int64_t rc = valid ? row : 0;
        // ---- 1. every load of the row is issued up front (the kernel lives on memory-level parallelism): gradient
        //         replicas, raw row, optimizer state; only then are the replicas cleared --------------------------------
        float g[4 * V], e[4 * V], mb[4 * V], vb[4 * V];
        float* const gr = a.grad_rows + rc * (int64_t)a.ld;
        const float* const w = a.table + rc * (int64_t)D;
        {
            float4 c[V];
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const int q = lane + TT * j;
                c[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (q < Q) c[j] = a.replicas == 1 ? *reinterpret_cast<const float4*>(gr + 4 * q)
                                                  : rsum4(gr + 4 * q, a.replicas, a.replica_stride);
            }
            load_raw<TT, V>(e, w, D, lane, a.tv);
            if (adam || sgd_m) load_chunks<TT, V>(mb, a.m + rc * (int64_t)a.ld, Q, lane);
            if (adam) load_chunks<TT, V>(vb, a.v + rc * (int64_t)a.ld, Q, lane);
#pragma unroll
            for (int j = 0; j < V; ++j) { g[4 * j] = c[j].x; g[4 * j + 1] = c[j].y; g[4 * j + 2] = c[j].z; g[4 * j + 3] = c[j].w; }
            if (XCHG && failed_before != 0) return;   // grid-uniform; nothing has been written yet
            if (valid) {
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int q = lane + TT * j;
                    if (q < Q)
                        for (int r = 0; r < a.replicas; ++r)
                            *reinterpret_cast<float4*>(gr + r * a.replica_stride + 4 * q) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
        // ---- 2. all-reduce over the ranks -----------------------------------------------------------------------------
        if (XCHG) {
            bool ok = true;
            if (valid) {
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int q = lane + TT * j;
                    if (q < Q) ll_push_chunk(a, (row * Q + q) * 2, make_float4(g[4 * j], g[4 * j + 1], g[4 * j + 2], g[4 * j + 3]));
                }
                if (lane == 0) LEC_TRACE_MAX(a.trace, 4);
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int q = lane + TT * j;
                    if (q < Q) {
                        float4 s;
                        ok = ll_reduce_chunk(a, (row * Q + q) * 2, s, t0) && ok;
                        g[4 * j] = s.x; g[4 * j + 1] = s.y; g[4 * j + 2] = s.z; g[4 * j + 3] = s.w;
                    }
                }
            }
            // a row whose exchange failed is left untouched (the host raises on *error); the vote keeps teams uniform
            if (__any_sync(0xffffffffu, !ok)) valid = false;
            if (lane == 0) LEC_TRACE_MAX(a.trace, 5);
        }
        row_rule<TT, V, RULE_T>(a, rule, row_mode, g, e, mb, vb, row, rc, valid, lane);
        row_forward<TT, V>(a, row_mode, e, row, valid, lane);
    }
    if (threadIdx.x == 0) LEC_TRACE_MAX(a.trace, 6);
    if (XCHG && blockIdx.x == 0 && threadIdx.x >= 32 && threadIdx.x < 64 && a.loss_acc && a.loss_global) {
        // the ranks' losses: lane p of the block's second warp polls source p's loss packet (all in parallel), lane 0
        // adds them in rank order.  AFTER the rows: polled before them (r2 trace), this warp sat on the peers' loss packets
        // while its own rows were still unsent -- one extra NVLink latency on the critical path of every rank.
        const int p = threadIdx.x - 32;
        double l = 0.0;
        bool ok = true;
        if (p < a.world) {
            const uint4* src = a.peer[a.rank] + ((int64_t)a.slot * a.world + p) * a.slot_packets + a.n * (int64_t)Q * 2;
            uint4 pk = ll_load(src);
            ok = ll_wait(src, a.tag, pk, a.error, a.timeout_ns, t0);
            l = __longlong_as_double((long long)(((unsigned long long)pk.z << 32) | (unsigned long long)pk.x));
        }
        ok = __all_sync(0xffffffffu, ok);
        double total = 0.0;
        for (int q = 0; q < a.world; ++q) total += __shfl_sync(0xffffffffu, l, q);
        if (p == 0 && ok) *a.loss_global = total;
    }
    if (loss_thread && a.loss_acc) {
        if (a.loss_step) *a.loss_step = my_loss;
        *a.loss_acc = 0.0;
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// Two-shot exchange for tables too large for the one-shot packets (cfg4: 82 K x 50 = 16.4 MB; one-shot would send the
// whole gradient to every peer).  Rank r OWNS a contiguous range of rows:
//   scatter   every rank sums its gradient replicas and stores each row into the OWNER's buffer (region [source rank]);
//             a tile of rows is followed by a release-store of the tile's flag                       -- reduce-scatter
//   owner     the owner waits for the `world` flags of a tile, adds the partial rows in rank order, applies the update
//             rule, writes table / rows / aux locally and stores the updated raw row into every peer's staging area
//             (+ tile flag)                                                                           -- update + all-gather
//   receiver  every rank waits for the tiles it does not own, copies the staged rows into its table and runs the row
//             transform on them
// 2 (W-1)/W of the table cross NVLink per rank and step instead of (W-1); the update rule runs once per row, so the
// replicas are bit-identical by construction.  Three launches: a kernel only ever waits for data produced by an EARLIER
// kernel of its peers, so no co-residency assumption is needed.
// ------------------------------------------------------------------------------------------------------------------------
template <int TT, int V>
__global__ void __launch_bounds__(kThreads) xchg_scatter_kernel(const UpdArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    if (a.error && ld_volatile_int(a.error) != 0) return;
    constexpr int kTeams = kThreads / TT;
    const int Q = a.ld >> 2;
    const TwoShot L(a.world, a.rows_per_rank, a.tiles_per_rank, a.ld);
    const int64_t n_tiles = (a.n + kTeams - 1) / kTeams;
    if (blockIdx.x == 0 && (int)threadIdx.x < a.world && a.loss_acc) {
        // this rank's loss of the step: one packet to every rank (gathered by the owner kernels, so that every wait of the
        // exchange is on something an EARLIER launch of the peers produced)
        const unsigned long long bits = (unsigned long long)__double_as_longlong(*a.loss_acc);
        ll_store(L.loss(a.peer[threadIdx.x], a.slot, a.world) + a.rank, (unsigned)(bits & 0xffffffffu), (unsigned)(bits >> 32), a.tag);
    }
    // A tile's rows are one contiguous slab of kTeams * ld floats in the replicas and in the owner's region alike: the
    // block moves it as a flat array, 512 contiguous bytes per warp store (whole NVLink packets, not 64-byte pieces)
    const int slab4 = kTeams * Q;                     // float4 per full tile
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int owner = (int)(tile / a.tiles_per_rank);
        const int64_t row0 = tile * kTeams;
        const int64_t rows_here = a.n - row0 < kTeams ? a.n - row0 : kTeams;
        const int n4 = (int)rows_here * Q;
        float* gr = a.grad_rows + row0 * (int64_t)a.ld;
        float* dst = L.rs(a.peer[owner], a.slot) + ((int64_t)a.rank * a.rows_per_rank + (row0 - (int64_t)owner * a.rows_per_rank)) * a.ld;
        for (int i0 = 0; i0 < slab4; i0 += 4 * kThreads) {
            float4 c[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = i0 + k * kThreads + (int)threadIdx.x;
                if (i < n4) c[k] = a.replicas == 1 ? *reinterpret_cast<const float4*>(gr + 4 * i)
                                                   : rsum4(gr + 4 * i, a.replicas, a.replica_stride);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = i0 + k * kThreads + (int)threadIdx.x;
                if (i < n4) {
                    *reinterpret_cast<float4*>(dst + 4 * i) = c[k];
                    for (int r = 0; r < a.replicas; ++r)
                        *reinterpret_cast<float4*>(gr + r * a.replica_stride + 4 * i) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
        __syncthreads();
        // release at system scope is cumulative: the block's stores above (ordered before this thread by the barrier) are
        // visible to the owner before the flag is
        if (threadIdx.x == 0)
            st_release_sys(L.rs_flag(a.peer[owner], a.slot) + (int64_t)a.rank * a.tiles_per_rank + (tile - (int64_t)owner * a.tiles_per_rank),
                           a.tag);
    }
}

template <int TT, int V, int RULE_T, int MODE_T>
__global__ void __launch_bounds__(kThreads, V <= 4 ? 2 : 1) update_owner_kernel(const UpdArgs a) {
    const int rule = RULE_T >= 0 ? RULE_T : a.rule;
    const int row_mode = MODE_T >= 0 ? MODE_T : a.row_mode;
    __shared__ int s_ok;
    extern __shared__ __align__(16) float s_stage[];   // [kThreads / TT rows][ld]
    pdl_launch_dependents();
    pdl_wait();
    if (a.error && ld_volatile_int(a.error) != 0) return;
    constexpr int kTeams = kThreads / TT;
    const int lane = threadIdx.x % TT, team = threadIdx.x / TT;
    const int D = a.D, Q = a.ld >> 2;
    const TwoShot L(a.world, a.rows_per_rank, a.tiles_per_rank, a.ld);
    unsigned long long t0 = 0;
    // losses: packets, as in the one-shot kernel
    double my_loss = 0.0;
    const bool loss_thread = blockIdx.x == 0 && threadIdx.x == 0;
    if (loss_thread && a.loss_acc) my_loss = *a.loss_acc;
    if (blockIdx.x == 0 && threadIdx.x >= 32 && threadIdx.x < 64 && a.loss_acc && a.loss_global) {
        const int p = threadIdx.x - 32;   // the losses were sent by the scatter kernels
        double l = 0.0;
        bool ok = true;
        if (p < a.world) {
            const uint4* src = L.loss(a.peer[a.rank], a.slot, a.world) + p;
            uint4 pk = ll_load(src);
            ok = ll_wait(src, a.tag, pk, a.error, a.timeout_ns, t0);
            l = __longlong_as_double((long long)(((unsigned long long)pk.z << 32) | (unsigned long long)pk.x));
        }
        ok = __all_sync(0xffffffffu, ok);
        double total = 0.0;
        for (int q = 0; q < a.world; ++q) total += __shfl_sync(0xffffffffu, l, q);
        if (p == 0 && ok) *a.loss_global = total;
    }
    const bool adam = rule == LEC_UPD_ADAM;
    const bool sgd_m = rule == LEC_UPD_SGD && a.m && a.momentum != 0.f;
    const int64_t row_lo = (int64_t)a.rank * a.rows_per_rank;
    int64_t my_rows = a.n - row_lo;
    if (my_rows > a.rows_per_rank) my_rows = a.rows_per_rank;
    const int64_t my_tiles = my_rows > 0 ? (my_rows + kTeams - 1) / kTeams : 0;
    const float* rs = L.rs(a.peer[a.rank], a.slot);
    for (int64_t tl = blockIdx.x; tl < my_tiles; tl += gridDim.x) {
        if (threadIdx.x == 0) s_ok = 1;
        __syncthreads();
        if ((int)threadIdx.x < a.world) {
            if (!flag_wait(L.rs_flag(a.peer[a.rank], a.slot) + (int64_t)threadIdx.x * a.tiles_per_rank + tl, a.tag, a.error,
                           a.timeout_ns, t0))
                s_ok = 0;
        }
        __syncthreads();
        const bool tile_ok = s_ok != 0;
        const int64_t lrow = tl * kTeams + team;
        const int64_t row = row_lo + lrow;
        const bool valid = lrow < my_rows && tile_ok;
        const int64_t rc = lrow < my_rows ? row : row_lo;
        const int64_t lrc = lrow < my_rows ? lrow : 0;
        float g[4 * V], e[4 * V], mb[4 * V], vb[4 * V];
        {
            float4 acc[V];
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int p = 0; p < a.world; ++p) {       // rank order: the sum does not depend on arrival order
                const float* src = rs + ((int64_t)p * a.rows_per_rank + lrc) * a.ld;
#pragma unroll
                for (int j = 0; j < V; ++j) {
                    const int q = lane + TT * j;
                    if (q < Q) acc[j] = add4(acc[j], __ldcv(reinterpret_cast<const float4*>(src + 4 * q)));
                }
            }
            load_raw<TT, V>(e, a.table + rc * (int64_t)D, D, lane, a.tv);
            if (adam || sgd_m) load_chunks<TT, V>(mb, a.m + rc * (int64_t)a.ld, Q, lane);
            if (adam) load_chunks<TT, V>(vb, a.v + rc * (int64_t)a.ld, Q, lane);
#pragma unroll
            for (int j = 0; j < V; ++j) { g[4 * j] = acc[j].x; g[4 * j + 1] = acc[j].y; g[4 * j + 2] = acc[j].z; g[4 * j + 3] = acc[j].w; }
        }
        row_rule<TT, V, RULE_T>(a, rule, row_mode, g, e, mb, vb, row, rc, valid, lane);
        // the tile's updated raw rows (pad columns zero) are staged in shared memory as the slab they form in every peer's
        // staging area ...
        {
            float4* st4 = reinterpret_cast<float4*>(s_stage) + team * Q;
#pragma unroll
            for (int j = 0; j < V; ++j) {
                const int q = lane + TT * j;
                if (q < Q) st4[q] = make_float4(e[4 * j], e[4 * j + 1], e[4 * j + 2], e[4 * j + 3]);
            }
        }
        row_forward<TT, V>(a, row_mode, e, row, valid, lane);
        __syncthreads();
        // ... and copied out flat: 512 contiguous bytes per warp store and peer
        if (tile_ok) {
            int64_t rows_here = my_rows - tl * kTeams;
            if (rows_here > kTeams) rows_here = kTeams;
            const int n4 = (int)rows_here * Q;
            const float4* src4 = reinterpret_cast<const float4*>(s_stage);
            for (int p = 0; p < a.world; ++p) {
                if (p == a.rank) continue;
                float4* dst4 = reinterpret_cast<float4*>(L.ag(a.peer[p], a.slot) + (row_lo + tl * kTeams) * (int64_t)a.ld);
                for (int i = threadIdx.x; i < n4; i += kThreads) dst4[i] = src4[i];
            }
        }
        __syncthreads();
        if ((int)threadIdx.x < a.world && (int)threadIdx.x != a.rank && tile_ok) {
            st_release_sys(L.ag_flag(a.peer[threadIdx.x], a.slot) + (int64_t)a.rank * a.tiles_per_rank + tl, a.tag);
        }
    }
    if (loss_thread && a.loss_acc) {
        if (a.loss_step) *a.loss_step = my_loss;
        *a.loss_acc = 0.0;
    }
}

template <int TT, int V>
__global__ void __launch_bounds__(kThreads) update_receiver_kernel(const UpdArgs a) {
    __shared__ int s_ok;
    pdl_launch_dependents();
    pdl_wait();
    if (a.error && ld_volatile_int(a.error) != 0) return;
    constexpr int kTeams = kThreads / TT;
    const int lane = threadIdx.x % TT, team = threadIdx.x / TT;
    const int D = a.D, Q = a.ld >> 2;
    const TwoShot L(a.world, a.rows_per_rank, a.tiles_per_rank, a.ld);
    unsigned long long t0 = 0;
    const float* ag = L.ag(a.peer[a.rank], a.slot);
    const int64_t n_tiles = (int64_t)a.world * a.tiles_per_rank;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int owner = (int)(tile / a.tiles_per_rank);
        const int64_t tl = tile - (int64_t)owner * a.tiles_per_rank;
        const int64_t row0 = (int64_t)owner * a.rows_per_rank + tl * kTeams;
        if (owner == a.rank || row0 >= a.n) continue;       // block-uniform
        if (threadIdx.x == 0)
            s_ok = flag_wait(L.ag_flag(a.peer[a.rank], a.slot) + tile, a.tag, a.error, a.timeout_ns, t0) ? 1 : 0;
        __syncthreads();
        const int64_t row = row0 + team;
        int64_t owner_end = (int64_t)(owner + 1) * a.rows_per_rank;
        if (owner_end > a.n) owner_end = a.n;
        const bool valid = row < owner_end && s_ok != 0;
        const int64_t rc = row < owner_end ? row : row0;
        float e[4 * V];
#pragma unroll
        for (int j = 0; j < V; ++j) {
            const int q = lane + TT * j;
            const float4 c = q < Q ? __ldcv(reinterpret_cast<const float4*>(ag + rc * (int64_t)a.ld + 4 * q)) : make_float4(0.f, 0.f, 0.f, 0.f);
            e[4 * j] = c.x; e[4 * j + 1] = c.y; e[4 * j + 2] = c.z; e[4 * j + 3] = c.w;
        }
        if (valid) store_raw<TT, V>(a.table + row * (int64_t)D, e, D, lane, a.tv);
        row_forward<TT, V>(a, a.row_mode, e, row, valid, lane);
        __syncthreads();
    }
}

constexpr int kUpdGridCap = 148 * 8;   // the same on every rank: a block's rows are the same rows everywhere

template <int TT, int V, int RULE_T, int MODE_T>
static int update_go2(const UpdArgs& a, cudaStream_t st) {
    // a label-sized table (ETHEC: 723 rows) is pure latency: 64-thread blocks spread its rows over ~4x as many SMs (more
    // load / store / packet slots in flight); the choice depends on n only, so every rank makes the same one
    int block = kThreads;
    while (block > 64 && (a.n + block / TT - 1) / (block / TT) < 96) block >>= 1;
    const int tpb = block / TT;
    int64_t need = (a.n + tpb - 1) / tpb;
    if (need < 1) need = 1;
    const int grid = (int)(need < kUpdGridCap ? need : kUpdGridCap);
    cudaError_t e;
    if (a.world > 1) e = launch_step_kernel(update_rows_kernel<TT, V, true, RULE_T, MODE_T>, grid, block, st, a);
    else e = launch_step_kernel(update_rows_kernel<TT, V, false, RULE_T, MODE_T>, grid, block, st, a);
    ++g_launches;
    return (int)(e != cudaSuccess ? e : cudaGetLastError());
}

template <int TT, int V, int RULE_T, int MODE_T>
static int two_shot_go2(const UpdArgs& a, cudaStream_t st) {
    const int tpb = kThreads / TT;
    const int64_t tiles = (a.n + tpb - 1) / tpb;
    auto grid_of = [](int64_t t) { return (int)(t < 1 ? 1 : (t < kUpdGridCap ? t : kUpdGridCap)); };
    const int ph = a.phases ? a.phases : (LEC_XCHG_SCATTER | LEC_XCHG_OWNER | LEC_XCHG_RECEIVER);
    cudaError_t e = cudaSuccess;
    if (ph & LEC_XCHG_SCATTER) { e = launch_step_kernel(xchg_scatter_kernel<TT, V>, grid_of(tiles), kThreads, st, a); ++g_launches; }
    if (e == cudaSuccess && (ph & LEC_XCHG_OWNER)) {
        const size_t stage = (size_t)tpb * a.ld * sizeof(float);
        if (stage > 48 * 1024) cudaFuncSetAttribute(update_owner_kernel<TT, V, RULE_T, MODE_T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stage);
        e = launch_step_kernel(update_owner_kernel<TT, V, RULE_T, MODE_T>, grid_of(a.tiles_per_rank), kThreads, st, a, stage);
        ++g_launches;
    }
    if (e == cudaSuccess && (ph & LEC_XCHG_RECEIVER)) { e = launch_step_kernel(update_receiver_kernel<TT, V>, grid_of(tiles), kThreads, st, a); ++g_launches; }
    return (int)(e != cudaSuccess ? e : cudaGetLastError());
}

template <int TT, int V>
static int two_shot_go(UpdArgs& a, cudaStream_t st) {
    const int tpb = kThreads / TT;
    const int64_t per = (a.n + a.world - 1) / a.world;
    a.tiles_per_rank = (int)((per + tpb - 1) / tpb);
    a.rows_per_rank = (int64_t)a.tiles_per_rank * tpb;
    if (a.rule == LEC_UPD_RSGD && a.row_mode == LEC_ROWS_HYP_SHELL) return two_shot_go2<TT, V, LEC_UPD_RSGD, LEC_ROWS_HYP_SHELL>(a, st);
    if (a.rule == LEC_UPD_RSGD_RETRACT) return two_shot_go2<TT, V, LEC_UPD_RSGD_RETRACT, LEC_ROWS_NONE>(a, st);
    if (a.rule == LEC_UPD_RSGD_LORENTZ) return two_shot_go2<TT, V, LEC_UPD_RSGD_LORENTZ, LEC_ROWS_NONE>(a, st);
    return two_shot_go2<TT, V, -1, -1>(a, st);
}

// bytes of one rank's two-shot exchange buffer (see TwoShot); the row tile follows the kernel configuration for ld
int64_t two_shot_bytes(int64_t n, int ld, int world) {
    const int Q = ld >> 2;
    const int tt = Q <= 16 ? 4 : (Q <= 64 ? 16 : 32);
    const int tpb = kThreads / tt;
    const int64_t per = (n + world - 1) / world;
    const int tiles_per_rank = (int)((per + tpb - 1) / tpb);
    return TwoShot(world, (int64_t)tiles_per_rank * tpb, tiles_per_rank, ld).bytes(world);
}

template <int TT, int V>
static int update_go(const UpdArgs& a, cudaStream_t st) {
    // the two training configurations of the benchmarks get specialised kernels; everything else the generic one
    if (a.rule == LEC_UPD_RSGD && a.row_mode == LEC_ROWS_HYP_SHELL) return update_go2<TT, V, LEC_UPD_RSGD, LEC_ROWS_HYP_SHELL>(a, st);
    if (a.rule == LEC_UPD_RSGD_RETRACT) return update_go2<TT, V, LEC_UPD_RSGD_RETRACT, LEC_ROWS_NONE>(a, st);   // row_mode NONE (checked)
    if (a.rule == LEC_UPD_RSGD_LORENTZ) return update_go2<TT, V, LEC_UPD_RSGD_LORENTZ, LEC_ROWS_NONE>(a, st);   // row_mode NONE (checked)
    if (a.rule == LEC_UPD_ADAM && a.row_mode == LEC_ROWS_EUC_SOFTCLIP && !a.hyp_rescale && !a.project_shell)
        return update_go2<TT, V, LEC_UPD_ADAM, LEC_ROWS_EUC_SOFTCLIP>(a, st);
    return update_go2<TT, V, -1, -1>(a, st);
}

int update_rows_launch(const lec_update_t& u, const lec_exchange_t* x, cudaStream_t st) {
    UpdArgs a{};
    a.rule = u.rule; a.row_mode = u.row_mode; a.geom = u.geom; a.lambda_mode = u.lambda_mode;
    a.hyp_rescale = u.hyp_rescale; a.project_shell = u.project_shell;
    a.K = u.K; a.lr = u.lr; a.r_in = u.r_in;
    hyp_constants(u.K, a.r_in_rows, a.c0);
    a.momentum = u.momentum; a.beta1 = u.beta1; a.beta2 = u.beta2; a.eps = u.eps;
    if (u.rule == LEC_UPD_ADAM) {
        const double t = (double)(u.opt_step < 1 ? 1 : u.opt_step);
        a.step_size = (float)((double)u.lr / (1.0 - pow((double)u.beta1, t)));
        a.inv_bc2_sqrt = (float)(1.0 / sqrt(1.0 - pow((double)u.beta2, t)));
    }
    a.table = u.table; a.n = u.n; a.D = u.D; a.ld = u.ld;
    const uintptr_t base = reinterpret_cast<uintptr_t>(u.table);
    uintptr_t go = reinterpret_cast<uintptr_t>(u.grad_out);
    a.tv = ((u.D & 3) == 0 && (base & 15) == 0 && (go & 15) == 0) ? 4 : (((u.D & 1) == 0 && (base & 7) == 0 && (go & 7) == 0) ? 2 : 1);
    a.grad_rows = u.grad_rows; a.replicas = u.grad_replicas; a.replica_stride = u.grad_stride > 0 ? u.grad_stride : u.n * (int64_t)u.ld;
    a.m = u.state_m; a.v = u.state_v;
    a.rows_out = u.rows_out; a.aux_out = u.aux_out; a.grad_out = u.grad_out;
    a.loss_acc = u.loss_acc; a.loss_step = u.loss_step;
#ifdef LEC_STEP_TRACE
    a.trace = g_step_trace;
#endif
    a.world = 0;
    if (x && x->world > 1) {
        a.world = x->world; a.rank = x->rank; a.slot = x->slot; a.tag = x->tag; a.slot_packets = x->slot_packets;
        for (int p = 0; p < x->world; ++p) a.peer[p] = static_cast<uint4*>(x->peer_bufs[p]);
        a.loss_global = x->loss_global; a.error = x->error;
        a.timeout_ns = (unsigned long long)(x->timeout_ms > 0 ? x->timeout_ms : 30000) * 1000000ull;
        a.phases = x->phases;
    }
    if (u.n == 0) return 0;
    const int Q = u.ld >> 2;
    if (a.world > 1 && x->mode == LEC_XCHG_TWO_SHOT) {
        if (Q <= 4) return two_shot_go<4, 1>(a, st);
        if (Q <= 16) return two_shot_go<4, 4>(a, st);
        if (Q <= 64) return two_shot_go<16, 4>(a, st);
        return two_shot_go<32, 8>(a, st);
    }
    if (Q <= 4) return update_go<4, 1>(a, st);
    if (Q <= 16) return update_go<4, 4>(a, st);
    if (Q <= 64) return update_go<16, 4>(a, st);
    return update_go<32, 8>(a, st);
}

}  // namespace lec
