// Fast all-pairs image x label scoring (fp32 core) with per-level top-k: the bandwidth/issue-bound tiled
// kernel of the scoring path (oe.py:1764-1779, oe_h.py:2018-2036 replaced; SURVEY 8 rows a13).
//
// Work unit = (label segment, image group).  A segment is one level's label range [start, stop) (its
// top-k is private to the unit) or, when the full matrix is wanted, a gap between levels.  Units are
// ordered largest segment first so the small levels fill the tail of the last wave.
//
// Thread mapping: a thread owns RI images (rows in registers, packed two images per 64-bit register
// pair) and walks the segment's labels, which are staged tile by tile in shared memory with every value
// duplicated ({x_d, x_d}) so that one broadcast LDS.128 feeds two packed FFMA2 (fma.rn.f32x2: two fp32
// FMAs per issue slot; the B200 FMA pipe does 128 FMA/clk/SM either way, the packing frees issue slots
// for the MUFU/ALU/LSU work of the epilogue).  Everything that depends on the label only (|x|^2, 1+|x|^2,
// the half-aperture) is computed once per tile in fp64 and staged next to the row.
//
// Hyperbolic energy per pair, from p = <x,y>, A = |x|^2, B = |y|^2 (order_embeddings_h.py:1097-1120):
//   num = p(1+A) - A(1+B);  s2 = A + B - 2p;  w2 = 1 + AB - 2p;  g = num * rsqrt(A s2 w2)
//   E = max(0, acos(clamp(g)) - psi),  acos(x) = sqrt(1-|x|) P7(|x|), reflected for x < 0
// (9 packed FMA-pipe ops + 2 MUFU + an 8-term polynomial; checked against the reference's fp64 run in
// tests/test_gpu_parity.py -- its error is below the reference's own fp32 error on the golden vectors).
// Poincare distance (LEC_GEOM_POINCARE, Nickel & Kiela): s = max(A + B - 2p, 0), delta = 2s / ((1-A)(1-B)),
//   E = log1p(delta + sqrt(delta (delta + 2))) = arcosh(1 + delta), 2/(1-A) and 1/(1-B) formed in fp64 per row.
// Lorentz distance (LEC_GEOM_LORENTZ, Nickel & Kiela 2018; rows are spatial parts, x0 = sqrt(1 + A)): per row, in fp64
//   and rounded once, x0 and e = x0 - 1 = A / (1 + x0);  per pair w = max(e_x y0 + (e_y - p), 0) = -<X,Y>_L - 1 and
//   E = log1p(w + sqrt(w (w + 2))).  Every term of w is a product of per-row constants or p itself, so its error is
//   |dw| <= (D + 8) 2^-24 (x0 y0 - 1 + |x||y|) (the dot product's gamma_D plus five roundings), small against w for
//   points apart at any radius; E then carries that error through arcosh(1 + w) plus a few ulp (DESIGN.md).
//
// Top-k: a thread cannot afford a sorted insertion per score (lanes diverge), so candidates that beat the
// current k-th best are appended, predicated and branch-free, to a small per-thread ring in shared
// memory; when any lane's ring is nearly full the whole warp merges its rings into the per-image sorted
// top-k lists (also in shared memory) and refreshes the thresholds.  NaN never passes `E < thr`.
//
// Deferred angle (hyperbolic, top-k only -- what the reference's caller consumes): acos is monotone, so
// E < thr  <=>  g > cos(thr + psi) = cos(thr) cos(psi) - sin(thr) sin(psi)  for thr + psi <= pi.  The main
// loop therefore tests g against that bound (2 packed FMAs, minus a 4e-6 slack so rounding can only let
// extra candidates through) and appends {g, label, -psi} to the ring; the acos polynomial runs only for
// ring entries inside merge(), with the same instruction sequence as the full-matrix path, so top-k
// values are bit-identical to the matrix entries.  thr > pi/2 or an unfilled list accepts everything.
#pragma once
#include "lec_common.cuh"
#include "lec_packed.cuh"

namespace lec {

constexpr int kMaxSeg = 2 * LEC_MAX_LEVELS + 1;
constexpr int kRing = 16;  // candidate ring entries per thread
constexpr int kTileLabels = 96;  // labels per shared-memory tile

struct FastArgs {
    const float* labels; const float* images; int64_t L, N; int D; float K;
    int k, n_levels;
    int n_seg;
    int seg_start[kMaxSeg], seg_stop[kMaxSeg], seg_level[kMaxSeg];
    float* scores; int64_t s_img, s_lab;  // element strides of the score matrix
    int32_t* topk_idx; float* topk_val;
    int64_t groups;  // image groups of NT*RI images
    int ring;        // candidate ring entries per thread (> RI)
    // evaluation passes (Pass below): labels = images = rows, row stride ld; a block evaluates the apex rows
    // [u_begin + c*chunk, ...) of chunk c against its image group
    int64_t ld, u_begin, u_end, chunk;
    const int32_t* tin; const int32_t* tout;
    const struct ReconState* rstate; const struct ReconOpen* ropen;
    unsigned long long* rhdr; unsigned long long* rhist;
    // extra intervals (DAG): apex u's extra preorder intervals [xlo[i], xhi[i]], i in [xptr[u], xptr[u+1])
    const int32_t* xptr; const int32_t* xlo; const int32_t* xhi;
    // rank passes (lec_rank.cu): block chunks index the apex list rapex[0, *rnapex); apex u's positives own slots
    // [rpos[u], rpos[u+1]); rxcum[i] = slots of u's primary interval and of its extra intervals before i
    const int32_t* rapex; const int* rnapex; const int64_t* rpos; const int32_t* rxcum;
    unsigned* rkey; int32_t* rval; const unsigned* rsorted; unsigned* rcnt; unsigned* req;
    // held-out passes: apex u's closure pairs own the closure slots [hptr[u], hptr[u+1]) (the layout of rpos for every
    // closure edge, extra intervals offset by rxcum); hmap[j] is the held-out slot of closure slot j, -1 for a pair that
    // is neither positive nor negative
    const int64_t* hptr; const int32_t* hmap;
};

// What a score_fast_kernel instantiation computes.  Score is the scoring kernel (top-k and / or the score matrix); the
// others are the all-pairs evaluation passes over the same energies, counted instead of stored.  The values appear in
// the kernels' mangled names.
//   F1            reconstruction F1 (lec_recon.cu): every pair's energy into the round's histograms
//   F1Dag         F1 on a DAG: a pair is also positive when tin[v] lies in one of the apex's extra intervals
//   RankKeys      reconstruction ranks (lec_rank.cu): the rank key of every positive pair into its slot (forest or DAG)
//   RankCounts    every negative pair at or below its apex's largest positive key into the bucket of its lower bound
//                 among the apex's sorted positive keys
//   F1Held, F1HeldDag  F1, F1Dag on a held-out set: a pair below its apex is positive only when its closure slot is
//                 held out and is skipped otherwise (only those pairs look the slot up); negatives are F1's
//   RankKeysHeld  RankKeys on a held-out set: the key of a held-out pair into its held-out slot hmap[closure slot]
enum class Pass : int { Score = 0, F1, F1Dag, RankKeys, RankCounts, F1Held, F1HeldDag, RankKeysHeld };
__host__ __device__ constexpr bool is_eval(Pass p) { return p != Pass::Score; }
__host__ __device__ constexpr bool is_rank(Pass p) {
    return p == Pass::RankKeys || p == Pass::RankCounts || p == Pass::RankKeysHeld;
}
__host__ __device__ constexpr bool is_f1(Pass p) { return is_eval(p) && !is_rank(p); }
// F1 passes with the extra-interval test compiled in (the rank passes test at run time: xptr may be NULL)
__host__ __device__ constexpr bool has_extra(Pass p) { return p == Pass::F1Dag || p == Pass::F1HeldDag; }
__host__ __device__ constexpr bool is_held(Pass p) {
    return p == Pass::F1Held || p == Pass::F1HeldDag || p == Pass::RankKeysHeld;
}

// Reconstruction check (lec_recon.cu).  Key of an energy = its fp32 bit pattern (energies are >= 0 or NaN, -0 is
// counted as 0); the coarse round histograms key >> kReconShift, a fine round counts every key of the open coarse bins.
constexpr int kReconShift = 16;
constexpr int kReconBins = 1 << (31 - kReconShift);  // coarse bins of a non-negative fp32 key (+inf included)
constexpr int kReconFine = 1 << kReconShift;         // fine bins (one fp32 value each) per coarse bin
struct ReconOpen { uint32_t bin, pad; unsigned long long cp_below, fp_below; };  // finite energies below the bin
struct ReconState {
    int phase, pad;                  // 0 coarse round, 1 fine rounds, 2 done
    long long n_open, next, m, batch;  // open coarse bins; first one and number of them in this round; bins per round
    unsigned long long n_pos, n_neg, nan_pos, nan_neg;
    double best_f1; unsigned long long best_cp, best_cn; unsigned best_key; int has_best;
};

// Reconstruction ranks (lec_rank.cu).  Rank key of an energy: its fp32 bits, -0 counted as 0, every NaN one value
// after +inf.  A staged tile counts the negatives of its apexes in up to kRankShared shared buckets {count, equal}
// (16 bits each: at most NT * RI images per block add to a bucket before the tile's flush); larger apexes count in
// global memory.
constexpr int kRankShared = 16384;
__device__ __forceinline__ unsigned rank_key(float e) {
    const unsigned k = __float_as_uint(e);
    return e != e ? 0x7fc00000u : (k == 0x80000000u ? 0u : k);
}

// per image: how many of an apex's extra intervals (xlo[xe.x, xe.x + xe.y), sorted starts, xe.y > 0) start at or before
// tin_v (binary lifting over the starts, the same ceil(log2(count + 1)) steps in every lane)
template <int RI>
__device__ __forceinline__ void extra_below(const int32_t* xlo, int2 xe, const int (&tin_v)[RI], int (&below)[RI]) {
#pragma unroll
    for (int r = 0; r < RI; ++r) below[r] = 0;
    for (int s = 1 << (31 - __clz(xe.y)); s > 0; s >>= 1) {
#pragma unroll
        for (int r = 0; r < RI; ++r) {
            const int i = below[r] + s;
            if (i <= xe.y && __ldg(xlo + xe.x + i - 1) <= tin_v[r]) below[r] = i;
        }
    }
}

// Shared-memory layout of one staged label: DQ float4 chunks of the row (zero padded), then one float4
// of constants.   hyp: {A, 1+A, A^2, -psi} {cos psi, sin psi, 0, 0}   euc: {A, t0, 0, 0}   oe: unused
// Label values enter the packed FMAs as scalar-broadcast operands (FFMA2 takes a .F32 operand that
// feeds both lanes), so nothing is duplicated in shared memory and an instruction reads two register
// pairs plus one scalar: the B200 register file sustains two pair reads per clock, three distinct pair
// operands cost three clocks (scripts/ubench_pipes.cu).
template <int V>
struct IntC {
    static constexpr int value = V;
};

template <int GEOM, int DH, int RI, int NT, int MINB, Pass PASS = Pass::Score>
__global__ void __launch_bounds__(NT, MINB) score_fast_kernel(const FastArgs a) {
    static_assert(RI % 2 == 0, "images are packed in pairs");
    constexpr bool EVAL = is_eval(PASS), RANK = is_rank(PASS), F1 = is_f1(PASS), XDAG = has_extra(PASS);
    constexpr bool HELD = is_held(PASS);
    constexpr int DQ = (DH + 1) / 2;     // float4 chunks per row
    constexpr int LS = 4 * DQ + 8;       // floats per staged label: row chunks + two float4 of constants
    constexpr int NP = RI / 2;           // packed image pairs per thread
    extern __shared__ __align__(16) float smem[];
    float* lab = smem;                                      // [kTileLabels][LS]
    float2* top = reinterpret_cast<float2*>(smem + kTileLabels * LS);  // [RI*k][NT]   {E, idx}
    float2* ring = top + (size_t)RI * a.k * NT;             // [a.ring][NT]  {E or g, (label << 3) | image slot}
    float* ringp = reinterpret_cast<float*>(ring + (size_t)a.ring * NT);  // [a.ring][NT]  -psi of a deferred entry
    float* psi_max_s = ringp + (size_t)a.ring * NT;         // largest half-aperture of the staged tile

    const int tid = threadIdx.x;
    const int seg = (int)(blockIdx.x / a.groups);
    const int64_t group = blockIdx.x % a.groups;
    const int l_begin = EVAL ? (int)(a.u_begin + (int64_t)seg * a.chunk) : a.seg_start[seg];
    const int l_end = EVAL ? (int)min(RANK ? (int64_t)*a.rnapex : a.u_end, a.u_begin + (int64_t)(seg + 1) * a.chunk)
                          : a.seg_stop[seg];
    if (RANK && l_begin >= l_end) return;  // the grid is sized for every apex row, the list holds those with P_u >= 1
    // row of staged label l: the apex list indexes the rows in the rank passes
    auto label_row = [&](int l) -> int64_t { return RANK ? (int64_t)a.rapex[l] : (int64_t)l; };
    const int level = EVAL ? -1 : a.seg_level[seg];
    const bool want_topk = (level >= 0) && (a.topk_idx != nullptr);
    const int k = a.k;
    const int D = a.D;

    // ---- image rows -> registers (two images per packed pair), per-image constants
    const int64_t img0 = group * (int64_t)(NT * RI) + tid;  // image of slot r: img0 + r*NT
    u64 y[NP][4 * DQ];
    u64 B2[NP], C2[NP];  // hyp: B, -(1+B) ; euc: B, unused
#pragma unroll
    for (int j = 0; j < NP; ++j) {
        const int64_t i0 = img0 + (2 * j) * NT, i1 = img0 + (2 * j + 1) * NT;
        const float* s0 = a.images + (i0 < a.N ? i0 : 0) * (EVAL ? a.ld : (int64_t)D);
        const float* s1 = a.images + (i1 < a.N ? i1 : 0) * (EVAL ? a.ld : (int64_t)D);
        float b0 = 0.f, b1 = 0.f;
        double e0 = 0.0, e1 = 0.0;  // Poincare, Lorentz: |y|^2 in fp64, as the labels' A
#pragma unroll
        for (int d = 0; d < 4 * DQ; ++d) {
            const float v0 = (d < D) ? __ldg(s0 + d) : 0.f;
            const float v1 = (d < D) ? __ldg(s1 + d) : 0.f;
            b0 = fmaf(v0, v0, b0);
            b1 = fmaf(v1, v1, b1);
            if (GEOM == LEC_GEOM_POINCARE || GEOM == LEC_GEOM_LORENTZ) {
                e0 += (double)v0 * (double)v0;
                e1 += (double)v1 * (double)v1;
            }
            y[j][d] = (GEOM == LEC_GEOM_OE) ? pack2(-v0, -v1) : pack2(v0, v1);
        }
        if (GEOM == LEC_GEOM_POINCARE) {  // B, 1 / (1 - B)
            B2[j] = pack2((float)e0, (float)e1);
            C2[j] = pack2((float)(1.0 / (1.0 - e0)), (float)(1.0 / (1.0 - e1)));
        } else if (GEOM == LEC_GEOM_LORENTZ) {  // y0, y0 - 1
            const double h0 = sqrt(1.0 + e0), h1 = sqrt(1.0 + e1);
            B2[j] = pack2((float)h0, (float)h1);
            C2[j] = pack2((float)(e0 / (1.0 + h0)), (float)(e1 / (1.0 + h1)));
        } else {
            B2[j] = pack2(b0, b1);
            C2[j] = pack2(-1.f - b0, -1.f - b1);
        }
    }

    // ---- top-k state: thresholds in registers, sorted lists and the candidate ring in shared memory
    float thr[RI];
#pragma unroll
    for (int r = 0; r < RI; ++r) thr[r] = INFINITY;
    const unsigned ring0 = (unsigned)__cvta_generic_to_shared(ring + tid);  // entry j of this thread: ring0 + j*NT*8
    unsigned rp = ring0;                                                     // next free entry
    const unsigned ring_trigger = ring0 + (unsigned)(a.ring - RI) * NT * 8;   // merge when rp > trigger
    if (want_topk) {
        for (int s = 0; s < RI * k; ++s) top[s * NT + tid] = make_float2(INFINITY, __int_as_float(-1));
    }
    const bool full = (group + 1) * (int64_t)(NT * RI) <= a.N;  // block-uniform: every image of the group exists

    // ---- reconstruction pass: coarse round = negatives per coarse bin in shared memory (positives, which are a
    // fraction of a percent of the pairs, go straight to global memory); fine rounds = the batch slot of every coarse
    // bin (or -1) in the same shared array.  Zeros, NaNs and the pair counts stay in registers until the block ends.
    unsigned* rsh = reinterpret_cast<unsigned*>(smem + kTileLabels * LS);
    int2* xsh = reinterpret_cast<int2*>(rsh + kReconBins);  // has_extra: [kTileLabels] {first extra interval, count}
    int rphase = 0;
    int tin_v[RI];
    unsigned c_np = 0, c_nn = 0, c_nanp = 0, c_nann = 0, c_zp = 0, c_zn = 0;
    // rank passes: per staged apex {first slot, P_u, smallest and largest sorted positive key}, {first extra interval,
    // count}, the first shared bucket (-1: global counters) and the prefix the flush searches; then the buckets
    int4* rsk = reinterpret_cast<int4*>(smem + kTileLabels * LS);
    int2* rxs = reinterpret_cast<int2*>(rsk + kTileLabels);
    int* rso = reinterpret_cast<int*>(rxs + kTileLabels);
    int* rpre = rso + kTileLabels;
    int* rused = rpre + kTileLabels;
    unsigned* rbk = reinterpret_cast<unsigned*>(rused + 4);
    if (F1) {
        rphase = a.rstate->phase;
        if (rphase == 2) return;
    }
    if (EVAL) {
#pragma unroll
        for (int r = 0; r < RI; ++r) {
            const int64_t v = img0 + r * NT;
            tin_v[r] = v < a.N ? a.tin[v] : 0;
        }
    }
    if (PASS == Pass::RankCounts)
        for (int b = tid; b < kRankShared; b += NT) rbk[b] = 0u;
    if (F1) {
        for (int b = tid; b < kReconBins; b += NT) rsh[b] = rphase == 0 ? 0u : ~0u;
        if (rphase == 1) {
            __syncthreads();
            const long long first = a.rstate->next, m = a.rstate->m;
            for (long long i = tid; i < m; i += NT) rsh[a.ropen[first + i].bin] = (unsigned)i;
        }
        // the tile loop's first barrier orders these stores before any use
    }
    // one ordered pair (x = label u, y = image v); valid excludes the diagonal and images past the table
    auto recon_count = [&](float e, bool valid, bool pos) {
        const bool fin = e == e;
        const bool zero = e == 0.f;
        const unsigned key = __float_as_uint(e);
        c_zp += valid & pos & zero;
        c_zn += valid & !pos & zero;
        if (rphase == 0) {
            c_np += valid & pos;
            c_nn += valid & !pos;
            c_nanp += valid & pos & !fin;
            c_nann += valid & !pos & !fin;
            if (valid && fin && !zero) {
                if (pos) atomicAdd(a.rhist + (key >> kReconShift), 1ull);
                else atomicAdd(rsh + (key >> kReconShift), 1u);
            }
        } else {
            int tag = -1;  // (slot, low key bits, positive) of a pair inside an open coarse bin
            if (valid && fin && !zero) {
                const int s = (int)rsh[key >> kReconShift];
                if (s >= 0) tag = (((s << kReconShift) | (int)(key & (kReconFine - 1))) << 1) | (int)pos;
            }
            // equal tags of a warp are added once: a heavily populated value costs one atomic per warp, not per pair
            if (__any_sync(0xffffffffu, tag >= 0)) {
                const unsigned peers = __match_any_sync(0xffffffffu, tag);
                if (tag >= 0 && (int)(tid & 31) == __ffs(peers) - 1) atomicAdd(a.rhist + tag, (unsigned long long)__popc(peers));
            }
        }
    };

    auto merge = [&]() {
        // insert this thread's ring entries into its sorted per-image lists (stable: ties keep the lower label)
        const int cnt = (int)((rp - ring0) / (NT * 8));
        for (int j = 0; j < cnt; ++j) {
            const float2 e = ring[j * NT + tid];
            const int code = __float_as_int(e.y);
            const int r = code & 7;
            float2* t = top + (size_t)(r * k) * NT + tid;
            if (e.x < t[(k - 1) * NT].x) {
                int pos = k - 1;
                while (pos > 0) {
                    const float2 prev = t[(pos - 1) * NT];
                    if (!(prev.x > e.x)) break;
                    t[pos * NT] = prev;
                    --pos;
                }
                t[pos * NT] = make_float2(e.x, __int_as_float(code >> 3));
            }
        }
        rp = ring0;
#pragma unroll
        for (int r = 0; r < RI; ++r) thr[r] = top[(size_t)(r * k + k - 1) * NT + tid].x;
    };

    // <x, y> of one staged label against this thread's packed image pairs.  Few pairs per thread (large D)
    // means few independent FMA chains, so the sum is split over NA partial accumulators per pair.
    auto dots = [&](const float4* lp, u64 (&acc)[NP]) {
        constexpr int NA = NP >= 4 ? 1 : (NP == 2 ? 2 : 4);
        u64 part[NP][NA];
#pragma unroll
        for (int j = 0; j < NP; ++j)
#pragma unroll
            for (int c = 0; c < NA; ++c) part[j][c] = 0ull;
#pragma unroll
        for (int q = 0; q < DQ; ++q) {
            const float4 v = lp[q];
            const float xv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (4 * q + c >= 2 * DH) continue;
                const u64 xb = pack2(xv[c], xv[c]);
#pragma unroll
                for (int j = 0; j < NP; ++j) part[j][c % NA] = ffma2(y[j][4 * q + c], xb, part[j][c % NA]);
            }
        }
#pragma unroll
        for (int j = 0; j < NP; ++j) {
            u64 t = part[j][0];
            if (NA == 2) t = fadd2(t, part[j][1]);
            if (NA == 4) t = fadd2(fadd2(t, part[j][1]), fadd2(part[j][2 % NA], part[j][3 % NA]));
            acc[j] = t;
        }
    };
    // cos of the cone angle for a packed pair: g = (p(1+A) - A(1+B)) * rsqrt(A (A+B-2p) (1+AB-2p))
    auto hyp_g = [&](u64 P, int j, const float4& cst) -> u64 {
        const u64 A2 = pack2(cst.x, cst.x), A12 = pack2(cst.y, cst.y), ASQ = pack2(cst.z, cst.z);
        const u64 M2 = pack2(-2.f, -2.f), ONE2 = pack2(1.f, 1.f);
        const u64 q = fmul2(P, M2);
        const u64 num = ffma2(P, A12, fmul2(A2, C2[j]));          // p(1+A) - A(1+B)
        const u64 w2 = fadd2(q, ffma2(A2, B2[j], ONE2));          // 1 + AB - 2p
        const u64 as2 = ffma2(A2, q, ffma2(A2, B2[j], ASQ));      // A (A + B - 2p)
        const u64 d2 = fmul2(as2, w2);
        float d0, d1;
        unpack2(d2, d0, d1);
        return fmul2(num, pack2(rsqrt_approx(d0), rsqrt_approx(d1)));
    };

    // ---- deferred-angle filter state (hyperbolic, top-k only): accept g >= cT cos(psi) - sT sin(psi) + off
    u64 cT2[NP], nsT2[NP], off2[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) { cT2[j] = 0ull; nsT2[j] = 0ull; off2[j] = pack2(-INFINITY, -INFINITY); }
    const unsigned ringp0 = (unsigned)__cvta_generic_to_shared(ringp + tid);
    // psi_max = largest half-aperture of the staged tile: the bound is only valid while thr + psi <= pi
    auto filter_terms = [&](float t, float psi_max, float& c, float& ns, float& off) {
        if (t <= 0.f) { c = 0.f; ns = 0.f; off = INFINITY; }                         // k zeros already: nothing can beat them
        else if (!(t + psi_max <= 3.1415f)) { c = 0.f; ns = 0.f; off = -INFINITY; }  // list not full / thr + psi may pass pi
        else { float sn, cs; __sincosf(t, &sn, &cs); c = cs; ns = -sn; off = -4e-6f; }  // MUFU sin/cos: |err| < 2e-6 on [0, pi]
    };
    auto refresh_filter = [&]() {
        const float psi_max = *psi_max_s;
#pragma unroll
        for (int j = 0; j < NP; ++j) {
            float c0, c1, n0, n1, o0, o1;
            filter_terms(top[(size_t)((2 * j) * k + k - 1) * NT + tid].x, psi_max, c0, n0, o0);
            filter_terms(top[(size_t)((2 * j + 1) * k + k - 1) * NT + tid].x, psi_max, c1, n1, o1);
            cT2[j] = pack2(c0, c1); nsT2[j] = pack2(n0, n1); off2[j] = pack2(o0, o1);
        }
    };
    auto merge_deferred = [&]() {
        const int cnt = (int)((rp - ring0) / (NT * 8));
        for (int j = 0; j < cnt; ++j) {
            const float2 e = ring[j * NT + tid];
            const float np = ringp[j * NT + tid];
            const int code = __float_as_int(e.y);
            const int r = code & 7;
            float z0, z1;
            unpack2(fadd2(acos_clamped2(pack2(e.x, e.x)), pack2(np, np)), z0, z1);
            const float Ev = max_nan(z0, 0.f);
            float2* t = top + (size_t)(r * k) * NT + tid;
            if (Ev < t[(k - 1) * NT].x) {
                int pos = k - 1;
                while (pos > 0) {
                    const float2 prev = t[(pos - 1) * NT];
                    if (!(prev.x > Ev)) break;
                    t[pos * NT] = prev;
                    --pos;
                }
                t[pos * NT] = make_float2(Ev, __int_as_float(code >> 3));
            }
        }
        rp = ring0;
        refresh_filter();
    };
    auto tile_loop_deferred = [&](int l0, int tl) {
        int lcode = l0 << 3;
#pragma unroll 2
        for (int t = 0; t < tl; ++t) {
            const float4* lp = reinterpret_cast<const float4*>(lab + t * LS);
            u64 acc[NP];
            dots(lp, acc);
            const float4 cst = lp[DQ];
            const float4 cs2 = lp[DQ + 1];
            const u64 CP = pack2(cs2.x, cs2.x), SP = pack2(cs2.y, cs2.y);
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                const u64 g = hyp_g(acc[j], j, cst);
                const u64 cb = ffma2(cT2[j], CP, ffma2(nsT2[j], SP, off2[j]));
                float g0, g1, b0, b1;
                unpack2(g, g0, g1);
                unpack2(cb, b0, b1);
                if (g0 >= b0) {
                    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(rp), "f"(g0), "r"(lcode + 2 * j) : "memory");
                    asm volatile("st.shared.b32 [%0], %1;" ::"r"(ringp0 + ((rp - ring0) >> 1)), "f"(cst.w) : "memory");
                    rp += NT * 8;
                }
                if (g1 >= b1) {
                    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(rp), "f"(g1), "r"(lcode + 2 * j + 1) : "memory");
                    asm volatile("st.shared.b32 [%0], %1;" ::"r"(ringp0 + ((rp - ring0) >> 1)), "f"(cst.w) : "memory");
                    rp += NT * 8;
                }
            }
            lcode += 8;
            if (__any_sync(0xffffffffu, rp > ring_trigger)) merge_deferred();
        }
    };

    // energies of one staged label against this thread's RI images
    auto energies = [&](const float* lrow, float (&E)[RI]) {
        const float4* lp = reinterpret_cast<const float4*>(lrow);
        u64 acc[NP];
#pragma unroll
        for (int j = 0; j < NP; ++j) acc[j] = 0ull;  // {0.f, 0.f}
        if (GEOM == LEC_GEOM_OE) {
#pragma unroll
            for (int q = 0; q < DQ; ++q) {
                const float4 v = lp[q];
                const float xv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (4 * q + c >= 2 * DH) continue;
#pragma unroll
                    for (int j = 0; j < NP; ++j) {
                        float d0, d1;
                        unpack2(fadd2(pack2(xv[c], xv[c]), y[j][4 * q + c]), d0, d1);  // x_d - y_d for the two images
                        const u64 dd = pack2(fmaxf(d0, 0.f), fmaxf(d1, 0.f));
                        acc[j] = ffma2(dd, dd, acc[j]);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < NP; ++j) unpack2(acc[j], E[2 * j], E[2 * j + 1]);
            return;
        }
        dots(lp, acc);
        const float4 cst = lp[DQ];
        if (GEOM == LEC_GEOM_HYP) {
            // cst = {A, 1+A, A^2, -psi};  q = -2p;  w2 = q + (AB + 1);  A*s2 = A q + (AB + A^2)
            const u64 npsi = pack2(cst.w, cst.w);
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                const u64 g = hyp_g(acc[j], j, cst);
                const u64 z = fadd2(acos_clamped2(g), npsi);
                float z0, z1;
                unpack2(z, z0, z1);
                E[2 * j] = max_nan(z0, 0.f);
                E[2 * j + 1] = max_nan(z1, 0.f);
            }
        } else if (GEOM == LEC_GEOM_POINCARE) {
            // cst = {A, 2 / (1 - A)};  s = max(A + B - 2p, 0);  delta = s 2/(1-A) 1/(1-B);  d = log1p(delta + sqrt(delta (delta + 2)))
            const u64 A2 = pack2(cst.x, cst.x), M2 = pack2(-2.f, -2.f), IA2 = pack2(cst.y, cst.y);
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                float s0, s1, i0, i1;
                unpack2(ffma2(M2, acc[j], fadd2(A2, B2[j])), s0, s1);
                unpack2(fmul2(IA2, C2[j]), i0, i1);
                const float d0 = max_nan(s0, 0.f) * i0, d1 = max_nan(s1, 0.f) * i1;
                E[2 * j] = log1pf(d0 + sqrtf(d0 * (d0 + 2.f)));
                E[2 * j + 1] = log1pf(d1 + sqrtf(d1 * (d1 + 2.f)));
            }
        } else if (GEOM == LEC_GEOM_LORENTZ) {
            // cst = {x0 - 1};  w = (x0 - 1) y0 + ((y0 - 1) - p);  d = log1p(w + sqrt(w (w + 2)))
            const u64 EX2 = pack2(cst.x, cst.x), M1 = pack2(-1.f, -1.f);
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                float w0, w1;
                unpack2(ffma2(EX2, B2[j], ffma2(M1, acc[j], C2[j])), w0, w1);
                w0 = max_nan(w0, 0.f);
                w1 = max_nan(w1, 0.f);
                E[2 * j] = log1pf(w0 + sqrtf(w0 * (w0 + 2.f)));
                E[2 * j + 1] = log1pf(w1 + sqrtf(w1 * (w1 + 2.f)));
            }
        } else {
            const float Af = cst.x, t0 = cst.y;
            const u64 A2 = pack2(Af, Af);
            const u64 M2 = pack2(-2.f, -2.f);
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                const u64 P = acc[j];
                const u64 s2 = ffma2(M2, P, fadd2(A2, B2[j]));            // |y - x|^2 = A + B - 2p
                float s0, s1, p0, p1;
                unpack2(s2, s0, s1);
                unpack2(P, p0, p1);
                // <x, y-x> / (max(|x|,eps) max(|y-x|,eps)); a vanishing |y-x| gives 0 like F.normalize
                const float q0 = Af * fmaxf(s0, 0.f), q1 = Af * fmaxf(s1, 0.f);
                const float c_0 = q0 > 0.f ? (p0 - Af) * rsqrt_approx(q0) : 0.f;
                const float c_1 = q1 > 0.f ? (p1 - Af) * rsqrt_approx(q1) : 0.f;
                E[2 * j] = max_nan(t0 - c_0, 0.f);
                E[2 * j + 1] = max_nan(t0 - c_1, 0.f);
            }
        }
    };

    // STORE (Pass::Score): 0 no matrix, 1 label-major and every image of the group exists, 2 generic strides / partial
    // group; an evaluation pass counts instead (STORE 0)
    auto tile_loop = [&](int l0, int tl, auto store_c, auto topk_c) {
        constexpr int STORE = decltype(store_c)::value;
        constexpr bool TOPK = decltype(topk_c)::value != 0;
        float* dst = nullptr;
        const int64_t s_lab = a.s_lab;
        if (STORE == 1) dst = a.scores + (int64_t)l0 * s_lab + img0;
        int lcode = l0 << 3;
#pragma unroll 2
        for (int t = 0; t < tl; ++t) {
            float E[RI];
            energies(lab + t * LS, E);
            if (STORE == 1) {
#pragma unroll
                for (int r = 0; r < RI; ++r) dst[r * NT] = E[r];
                dst += s_lab;
            } else if (STORE == 2) {
                float* row = a.scores + (int64_t)(l0 + t) * s_lab;
#pragma unroll
                for (int r = 0; r < RI; ++r) {
                    const int64_t i = img0 + r * NT;
                    if (i < a.N) row[i * a.s_img] = E[r];
                }
            } else if (F1 && !XDAG) {
                const int u = l0 + t;
                const int* ue = reinterpret_cast<const int*>(lab + t * LS + 4 * DQ + 6);  // Euler interval of u
                const int tin_u = ue[0], tout_u = ue[1];
#pragma unroll
                for (int r = 0; r < RI; ++r) {
                    const int64_t v = img0 + r * NT;
                    bool valid = v < a.N && v != u;
                    const bool pos = tin_u < tin_v[r] && tin_v[r] <= tout_u;
                    // held out: a pair below u loads the held-out slot of its closure slot (ue[-1]: u's first one); a
                    // training pair is skipped
                    if (HELD && valid && pos && __ldg(a.hmap + ue[-1] + tin_v[r] - tin_u - 1) < 0) valid = false;
                    recon_count(E[r], valid, pos);
                }
            } else if (XDAG) {
                const int u = l0 + t;
                const int* ue = reinterpret_cast<const int*>(lab + t * LS + 4 * DQ + 6);
                const int tin_u = ue[0], tout_u = ue[1];
                bool pos[RI];
                int cs[RI];  // held out: closure slot of a pair below u
#pragma unroll
                for (int r = 0; r < RI; ++r) {
                    pos[r] = tin_u < tin_v[r] && tin_v[r] <= tout_u;
                    if (HELD) cs[r] = ue[-1] + tin_v[r] - tin_u - 1;
                }
                const int2 xe = xsh[t];
                if (xe.y > 0) {  // block-uniform: every thread is on apex u
                    // the last extra interval starting at or before tin_v, then its end
                    int below[RI];
                    extra_below(a.xlo, xe, tin_v, below);
                    if (HELD) {
#pragma unroll
                        for (int r = 0; r < RI; ++r) {
                            const int i = xe.x + below[r] - 1;
                            if (below[r] > 0 && tin_v[r] <= __ldg(a.xhi + i)) {
                                pos[r] = true;
                                cs[r] = ue[-1] + __ldg(a.rxcum + i) + tin_v[r] - __ldg(a.xlo + i);
                            }
                        }
                    } else {
#pragma unroll
                        for (int r = 0; r < RI; ++r)
                            pos[r] |= below[r] > 0 && tin_v[r] <= __ldg(a.xhi + xe.x + below[r] - 1);
                    }
                }
#pragma unroll
                for (int r = 0; r < RI; ++r) {
                    const int64_t v = img0 + r * NT;
                    bool valid = v < a.N && v != u;
                    if (HELD && valid && pos[r] && __ldg(a.hmap + cs[r]) < 0) valid = false;  // as F1Held
                    recon_count(E[r], valid, pos[r]);
                }
            } else if (RANK) {
                constexpr bool KEYS = PASS != Pass::RankCounts;
                const int* ue = reinterpret_cast<const int*>(lab + t * LS + 4 * DQ + 6);
                const int tin_u = ue[0], tout_u = ue[1];
                const int4 rk = rsk[t];  // {first slot, P_u, smallest key, largest key}
                bool pos[RI];
                int slot[RI];
#pragma unroll
                for (int r = 0; r < RI; ++r) {
                    pos[r] = img0 + r * NT < a.N && tin_u < tin_v[r] && tin_v[r] <= tout_u;
                    slot[r] = tin_v[r] - tin_u - 1;
                }
                const int2 xe = rxs[t];
                if (xe.y > 0) {  // block-uniform: F1Dag's search of the apex's extra intervals
                    int below[RI];
                    extra_below(a.xlo, xe, tin_v, below);
#pragma unroll
                    for (int r = 0; r < RI; ++r) {
                        const int i = xe.x + below[r] - 1;
                        if (img0 + r * NT < a.N && below[r] > 0 && tin_v[r] <= __ldg(a.xhi + i)) {
                            pos[r] = true;
                            if (KEYS) slot[r] = __ldg(a.rxcum + i) + tin_v[r] - __ldg(a.xlo + i);
                        }
                    }
                }
                if (KEYS) {
#pragma unroll
                    for (int r = 0; r < RI; ++r) {
                        if (pos[r] && slot[r] < rk.y) {  // a slot past P_u would mean pos_ptr disagrees with the cover
                            const int j = HELD ? __ldg(a.hmap + rk.x + slot[r]) : rk.x + slot[r];
                            if (HELD && j < 0) continue;  // a training pair
                            a.rkey[j] = rank_key(E[r]);
                            a.rval[j] = j;
                        }
                    }
                } else {
                    unsigned key[RI];
                    bool neg[RI], srch = false;
                    int lb[RI];
#pragma unroll
                    for (int r = 0; r < RI; ++r) {
                        key[r] = rank_key(E[r]);
                        neg[r] = img0 + r * NT < a.N && tin_v[r] != tin_u && !pos[r] && key[r] <= (unsigned)rk.w;
                        lb[r] = 0;
                        srch |= neg[r] && key[r] > (unsigned)rk.z;
                    }
                    // lower bound among the sorted positive keys: the same ceil(log2(P_u + 1)) steps in every lane
                    const unsigned* sk = a.rsorted + rk.x;
                    if (__any_sync(0xffffffffu, srch)) {
                        for (int s = 1 << (31 - __clz(rk.y)); s > 0; s >>= 1) {
#pragma unroll
                            for (int r = 0; r < RI; ++r) {
                                const int i = lb[r] + s;
                                if (neg[r] && i <= rk.y && __ldg(sk + i - 1) < key[r]) lb[r] = i;
                            }
                        }
                    }
                    const int so = rso[t];
                    if (so >= 0) {  // block-uniform
#pragma unroll
                        for (int r = 0; r < RI; ++r)
                            if (neg[r]) atomicAdd(rbk + so + lb[r], __ldg(sk + lb[r]) == key[r] ? 0x10001u : 1u);
                    } else {
                        // equal buckets of a warp are added once, as in the fine round of the F1 pass
#pragma unroll
                        for (int r = 0; r < RI; ++r) {
                            const int tag = neg[r] ? rk.x + lb[r] : -1;
                            const bool eq = neg[r] && __ldg(sk + lb[r]) == key[r];
                            if (__any_sync(0xffffffffu, tag >= 0)) {
                                const unsigned peers = __match_any_sync(0xffffffffu, tag);
                                const unsigned eqm = __ballot_sync(0xffffffffu, eq);
                                if (tag >= 0 && (int)(tid & 31) == __ffs(peers) - 1) {
                                    atomicAdd(a.rcnt + tag, (unsigned)__popc(peers));
                                    const int ne = __popc(peers & eqm);
                                    if (ne) atomicAdd(a.req + tag, (unsigned)ne);
                                }
                            }
                        }
                    }
                }
            }
            if (TOPK) {
#pragma unroll
                for (int r = 0; r < RI; ++r) {
                    if (E[r] < thr[r]) {
                        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(rp), "f"(E[r]), "r"(lcode + r) : "memory");
                        rp += NT * 8;
                    }
                }
                lcode += 8;
                if (__any_sync(0xffffffffu, rp > ring_trigger)) merge();
            }
        }
    };

    const int store = (a.scores == nullptr) ? 0 : ((a.s_img == 1 && full) ? 1 : 2);
    for (int l0 = l_begin; l0 < l_end; l0 += kTileLabels) {
        const int tl = min(kTileLabels, l_end - l0);
        __syncthreads();
        // ---- stage the tile: rows zero-padded to whole float4 chunks
        for (int i = tid; i < tl * 4 * DQ; i += NT) {
            const int t = i / (4 * DQ), d = i - t * (4 * DQ);
            lab[t * LS + d] = (d < D) ? __ldg(a.labels + label_row(l0 + t) * (EVAL ? a.ld : (int64_t)D) + d) : 0.f;
        }
        // ---- per-label constants in fp64 (same terms as lec_rows_fwd's aux)
        if (GEOM != LEC_GEOM_OE) {
            for (int t = tid; t < tl; t += NT) {
                const float* src = a.labels + label_row(l0 + t) * (EVAL ? a.ld : (int64_t)D);
                double A = 0.0;
                for (int d = 0; d < D; ++d) { const double v = (double)__ldg(src + d); A += v * v; }
                const Aux<double> x = row_aux<double>(GEOM, A, a.K);
                float4 c, c2 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (GEOM == LEC_GEOM_POINCARE) {
                    c = make_float4((float)A, (float)(2.0 / (1.0 - A)), 0.f, 0.f);
                } else if (GEOM == LEC_GEOM_LORENTZ) {
                    c = make_float4((float)(A / (1.0 + sqrt(1.0 + A))), 0.f, 0.f, 0.f);  // x0 - 1
                } else if (GEOM == LEC_GEOM_HYP) {
                    c = make_float4((float)A, (float)(1.0 + A), (float)(A * A), (float)(-x.t0));
                    const double sp = sin(x.t0);  // = the clamped asin argument
                    c2 = make_float4((float)sqrt(fmax(0.0, 1.0 - sp * sp)), (float)sp, 0.f, 0.f);
                } else {
                    c = make_float4((float)A, (float)x.t0, 0.f, 0.f);
                }
                *reinterpret_cast<float4*>(lab + t * LS + 4 * DQ) = c;
                *reinterpret_cast<float4*>(lab + t * LS + 4 * DQ + 4) = c2;
            }
        }
        if (EVAL) {  // the apex's Euler interval in the last two constant slots (after the stores above, same thread)
            for (int t = tid; t < tl; t += NT) {
                int* ue = reinterpret_cast<int*>(lab + t * LS + 4 * DQ + 6);
                const int64_t u = label_row(l0 + t);
                ue[0] = a.tin[u];
                ue[1] = a.tout[u];
                if (F1 && HELD) ue[-1] = (int)a.hptr[u];  // the deferred top-k's sin(psi) slot
                if (XDAG) {
                    const int x0 = a.xptr[u];
                    xsh[t] = make_int2(x0, a.xptr[u + 1] - x0);
                }
                if (RANK) {
                    const int x0 = a.xptr ? a.xptr[u] : 0;
                    rxs[t] = make_int2(x0, a.xptr ? a.xptr[u + 1] - x0 : 0);
                    const int64_t* sp = HELD ? a.hptr : a.rpos;  // RankKeysHeld walks the closure slots
                    const int base = (int)sp[u], n = (int)(sp[u + 1] - base);
                    rsk[t] = PASS == Pass::RankCounts
                                 ? make_int4(base, n, (int)a.rsorted[base], (int)a.rsorted[base + n - 1])
                                 : make_int4(base, n, 0, 0);
                }
            }
        }
        __syncthreads();
        if (PASS == Pass::RankCounts) {
            // shared buckets for the tile's apexes in order while their P_u sum stays within kRankShared; an apex
            // larger than that, and every apex after the budget is spent, counts in global memory
            if (tid < 32) {
                static_assert(kTileLabels == 3 * 32, "three staged apexes per lane");
                int s[3], loc = 0;
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int t = 3 * tid + j;
                    const int n = t < tl ? rsk[t].y : 0;
                    s[j] = n <= kRankShared ? n : 0;
                    loc += s[j];
                }
                int inc = loc;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, inc, o);
                    if (tid >= o) inc += y;
                }
                int pre = inc - loc, used = 0;
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int t = 3 * tid + j;
                    const bool fits = s[j] > 0 && pre + s[j] <= kRankShared;
                    if (t < tl) { rpre[t] = pre; rso[t] = fits ? pre : -1; }
                    if (fits) used = pre + s[j];
                    pre += s[j];
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) used = max(used, __shfl_xor_sync(0xffffffffu, used, o));
                if (tid == 0) *rused = used;
            }
            __syncthreads();
        }
        if (GEOM == LEC_GEOM_HYP && want_topk && store == 0) {
            if (tid < 32) {
                float mx = -INFINITY;
                for (int t = tid; t < tl; t += 32) mx = fmaxf(mx, -lab[t * LS + 4 * DQ + 3]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                if (tid == 0) *psi_max_s = mx;
            }
            __syncthreads();
            refresh_filter();
        }
        if (RANK) {
            tile_loop(l0, tl, IntC<0>(), IntC<0>());
            if (PASS == Pass::RankCounts) {  // flush the tile's non-zero buckets and clear them for the next tile
                __syncthreads();
                const int used = *rused;
                for (int i = tid; i < used; i += NT) {
                    const unsigned c = rbk[i];
                    if (!c) continue;
                    rbk[i] = 0u;
                    int lo = 0, hi = tl - 1;  // owner: the last staged apex whose buckets start at or before i
                    while (lo < hi) {
                        const int mid = (lo + hi + 1) >> 1;
                        if (rpre[mid] <= i) lo = mid;
                        else hi = mid - 1;
                    }
                    const int g = rsk[lo].x + (i - rpre[lo]);
                    atomicAdd(a.rcnt + g, c & 0xffffu);
                    if (c >> 16) atomicAdd(a.req + g, c >> 16);
                }
            }
        } else if (F1) {
            tile_loop(l0, tl, IntC<0>(), IntC<0>());
        } else if (want_topk) {
            if (store == 0 && GEOM == LEC_GEOM_HYP) tile_loop_deferred(l0, tl);
            else if (store == 0) tile_loop(l0, tl, IntC<0>(), IntC<1>());
            else if (store == 1) tile_loop(l0, tl, IntC<1>(), IntC<1>());
            else tile_loop(l0, tl, IntC<2>(), IntC<1>());
        } else {
            if (store == 1) tile_loop(l0, tl, IntC<1>(), IntC<0>());
            else if (store == 2) tile_loop(l0, tl, IntC<2>(), IntC<0>());
        }
    }

    if (RANK) return;
    if (F1) {
        // register counters: one global add per warp; then the block's coarse negatives
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c_np += __shfl_xor_sync(0xffffffffu, c_np, o);
            c_nn += __shfl_xor_sync(0xffffffffu, c_nn, o);
            c_nanp += __shfl_xor_sync(0xffffffffu, c_nanp, o);
            c_nann += __shfl_xor_sync(0xffffffffu, c_nann, o);
            c_zp += __shfl_xor_sync(0xffffffffu, c_zp, o);
            c_zn += __shfl_xor_sync(0xffffffffu, c_zn, o);
        }
        if ((tid & 31) == 0) {
            if (rphase == 0) {
                if (c_np) atomicAdd(a.rhdr + 0, (unsigned long long)c_np);
                if (c_nn) atomicAdd(a.rhdr + 1, (unsigned long long)c_nn);
                if (c_nanp) atomicAdd(a.rhdr + 2, (unsigned long long)c_nanp);
                if (c_nann) atomicAdd(a.rhdr + 3, (unsigned long long)c_nann);
                if (c_zp) atomicAdd(a.rhist + 0, (unsigned long long)c_zp);
                if (c_zn) atomicAdd(a.rhist + kReconBins, (unsigned long long)c_zn);
            } else {
                const int s0 = (int)rsh[0];  // key 0 is fine bin 0 of coarse bin 0
                if (s0 >= 0) {
                    const int64_t z = (int64_t)s0 << (kReconShift + 1);
                    if (c_zp) atomicAdd(a.rhist + z + 1, (unsigned long long)c_zp);
                    if (c_zn) atomicAdd(a.rhist + z, (unsigned long long)c_zn);
                }
            }
        }
        if (rphase == 0) {
            __syncthreads();
            for (int b = tid; b < kReconBins; b += NT) {
                const unsigned c = rsh[b];
                if (c) atomicAdd(a.rhist + kReconBins + b, (unsigned long long)c);
            }
        }
        return;
    }

    if (want_topk) {
        if (store == 0 && GEOM == LEC_GEOM_HYP) merge_deferred();
        else merge();
#pragma unroll
        for (int r = 0; r < RI; ++r) {
            const int64_t i = img0 + r * NT;
            if (i >= a.N) continue;
            const int64_t o = (i * a.n_levels + level) * k;
            for (int j = 0; j < k; ++j) {
                const float2 e = top[(size_t)(r * k + j) * NT + tid];
                a.topk_idx[o + j] = __float_as_int(e.y);
                if (a.topk_val) a.topk_val[o + j] = e.x;
            }
        }
    }
}

// The <DH, RI> instantiation for a row width D, f(IntC<DH>(), IntC<RI>()): the scoring kernel and every evaluation pass
// share it, because the energy bits depend on RI (through the accumulator split of dots), and so every evaluation pass
// equals the SIMT score matrix bit for bit.
template <typename F>
static int dispatch_width(int D, F&& f) {
    const int dh = (D + 1) / 2;
    if (dh <= 1) return f(IntC<1>(), IntC<4>());
    if (dh <= 2) return f(IntC<2>(), IntC<4>());
    if (dh <= 5) return f(IntC<5>(), IntC<4>());
    if (dh <= 8) return f(IntC<8>(), IntC<4>());
    if (dh <= 16) return f(IntC<16>(), IntC<2>());
    if (dh <= 25) return f(IntC<25>(), IntC<2>());
    if (dh <= 32) return f(IntC<32>(), IntC<2>());
    return LEC_E_DIM;
}

// 128-thread blocks whose register allocation need only allow one resident block per SM; a thread holds RI images.
template <int GEOM, int DH, int RI>
static int fast_launch_dh(FastArgs& a, cudaStream_t st) {
    constexpr int NT = 128;
    static_assert(kRing > RI, "a thread appends up to RI candidates per label before the ring is merged");
    a.ring = kRing;
    constexpr int LS = 4 * ((DH + 1) / 2) + 8;
    const size_t smem = (size_t)kTileLabels * LS * sizeof(float) + ((size_t)RI * a.k + a.ring) * NT * sizeof(float2) +
                        (size_t)a.ring * NT * sizeof(float) + 16;
    static size_t configured = 0;
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(score_fast_kernel<GEOM, DH, RI, NT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        configured = smem;
    }
    a.groups = (a.N + (int64_t)NT * RI - 1) / ((int64_t)NT * RI);
    const int64_t blocks = a.groups * a.n_seg;
    if (blocks <= 0) return 0;
    if (blocks > 0x7fffffffLL) return LEC_E_SIZE;
    score_fast_kernel<GEOM, DH, RI, NT, 1><<<(unsigned)blocks, NT, smem, st>>>(a);
    ++g_launches;
    return (int)cudaGetLastError();
}

template <int GEOM>
static int fast_launch_geom(FastArgs& a, cudaStream_t st) {
    return dispatch_width(a.D, [&](auto dh, auto ri) {
        return fast_launch_dh<GEOM, decltype(dh)::value, decltype(ri)::value>(a, st);
    });
}

// Evaluation passes: one block per SM (128 KB of shared counters in the F1 passes), 16 warps where the image rows fit
// 128 registers, else 8 (D > 32 spills at 512 threads).  The block size does not change the energy bits.
constexpr int eval_threads(int dh) { return dh > 16 ? 256 : 512; }
constexpr int kEvalTarget = 148 * 16;    // blocks per pass to aim for (16 waves: the chunks balance)
constexpr int64_t kEvalMaxChunk = 4096;  // apex rows per block: the F1 passes' 32-bit shared counters cannot overflow

// dynamic shared memory of an evaluation pass: the staged tile, then the F1 passes' coarse counters (and the extra
// intervals of the staged apexes) or the rank passes' per-apex table (and the count's buckets)
constexpr size_t eval_smem_bytes(Pass p, int dh) {
    return (size_t)kTileLabels * (4 * ((dh + 1) / 2) + 8) * sizeof(float) +
           (is_rank(p) ? (size_t)kTileLabels * (sizeof(int4) + sizeof(int2) + 2 * sizeof(int)) + 4 * sizeof(int) +
                             (p == Pass::RankCounts ? (size_t)kRankShared * sizeof(unsigned) : 0)
                       : (size_t)kReconBins * sizeof(unsigned) + (has_extra(p) ? (size_t)kTileLabels * sizeof(int2) : 0));
}

// one pass over the apex rows [u_begin, u_end) (the rank passes: entries of the apex list, u_begin = 0)
template <int GEOM, int DH, int RI, Pass P>
static int eval_launch_dh(FastArgs& a, cudaStream_t st) {
    constexpr int NT = eval_threads(DH);
    constexpr size_t smem = eval_smem_bytes(P, DH);
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(score_fast_kernel<GEOM, DH, RI, NT, 1, P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        configured = true;
    }
    a.groups = (a.N + (int64_t)NT * RI - 1) / ((int64_t)NT * RI);
    const int64_t rows = a.u_end - a.u_begin;  // rank passes: an upper bound on the apex list; blocks past its end return
    int64_t chunks = (kEvalTarget + a.groups - 1) / a.groups;
    int64_t chunk = (rows + chunks - 1) / chunks;
    if (chunk < 32) chunk = 32;
    if (chunk > kEvalMaxChunk) chunk = kEvalMaxChunk;
    a.chunk = chunk;
    chunks = (rows + chunk - 1) / chunk;
    const int64_t blocks = a.groups * chunks;
    if (blocks > 0x7fffffffLL) return LEC_E_SIZE;
    score_fast_kernel<GEOM, DH, RI, NT, 1, P><<<(unsigned)blocks, NT, smem, st>>>(a);
    ++g_launches;
    return (int)cudaGetLastError();
}

template <int GEOM, Pass P>
static int eval_launch_geom(FastArgs& a, cudaStream_t st) {
    return dispatch_width(a.D, [&](auto dh, auto ri) {
        return eval_launch_dh<GEOM, decltype(dh)::value, decltype(ri)::value, P>(a, st);
    });
}

// evaluation pass P for a geometry the caller has validated
template <Pass P>
static int eval_launch(int geom, FastArgs& a, cudaStream_t st) {
    switch (geom) {
        case LEC_GEOM_EUC: return eval_launch_geom<LEC_GEOM_EUC, P>(a, st);
        case LEC_GEOM_HYP: return eval_launch_geom<LEC_GEOM_HYP, P>(a, st);
        case LEC_GEOM_POINCARE: return eval_launch_geom<LEC_GEOM_POINCARE, P>(a, st);
        case LEC_GEOM_LORENTZ: return eval_launch_geom<LEC_GEOM_LORENTZ, P>(a, st);
        default: return eval_launch_geom<LEC_GEOM_OE, P>(a, st);
    }
}

// Checks of the fields lec_recon_t and lec_rank_t share, in the order their entry points apply them: NULL (`set`: the
// caller's own pointers are set), DIM, ENUM, SIZE, then the caller's own checks `more()`, then ALIGN.
template <typename T, typename F>
static int eval_validate(const T* r, bool set, F&& more) {
    if (!r || !r->rows || !r->tin || !r->tout || !r->workspace || !set) return LEC_E_NULL;
    if (r->D < 1 || r->D > 64 || r->ld < r->D || (r->ld != r->D && r->ld % 4 != 0)) return LEC_E_DIM;
    if (r->geom != LEC_GEOM_EUC && r->geom != LEC_GEOM_HYP && r->geom != LEC_GEOM_OE && r->geom != LEC_GEOM_POINCARE &&
        r->geom != LEC_GEOM_LORENTZ)
        return LEC_E_ENUM;
    if (r->n < 0 || r->n > 0x7fffffffLL || r->u_begin < 0 || r->u_end < r->u_begin || r->u_end > r->n) return LEC_E_SIZE;
    if (const int e = more()) return e;
    if ((reinterpret_cast<uintptr_t>(r->rows) & 15) || (reinterpret_cast<uintptr_t>(r->workspace) & 15)) return LEC_E_ALIGN;
    return 0;
}

// arguments of a held-out set (lec_rank_run_heldout, lec_recon_pass_heldout); xcum is needed with extra intervals.
// closure_ptr[n] == n_closure is the caller's to keep, like pos_ptr's agreement with the cover: reading it would
// synchronise.
inline int heldout_validate(const lec_heldout_t* h, bool dag) {
    if (!h->closure_ptr || !h->slot_map || (dag && !h->xcum)) return LEC_E_NULL;
    if (h->n_closure < 0 || h->n_closure > 0x7fffffffLL) return LEC_E_SIZE;
    return 0;
}

}  // namespace lec
