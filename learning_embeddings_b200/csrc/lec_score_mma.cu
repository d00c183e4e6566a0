// Tensor-core path of the all-pairs image x label scoring (hyperbolic cones), sm_100a only.
//
// Replaces the per-image CPU loop of JointEmbeddings.calculate_classification_metrics
// (oe_h.py:2018-2036): e[i, l] = E(x = label_l, y = image_i), then per level topk(k, largest=False).
//
// With A = |x|^2 (label), B = |y|^2 (image), p = <x, y> the cosine of the cone angle is
//     g = num * rsqrt(as2 * w2),   num = p(1+A) - A(1+B),   w2 = 1 + AB - 2p,   as2 = A (A + B - 2p)
// (order_embeddings_h.py:1097-1120).  All three are BILINEAR in the augmented rows y' = [y, B, 1] and
//     x'_num = [(1+A) x, -A, -A]     x'_w2 = [-2 x, A, 1]     x'_as2 = [-2A x, A, A^2]
// so one tcgen05.mma (kind::tf32, M = 128 images, N = 3 x 32 label rows, K = D + 2, fp32 accumulators in TMEM)
// produces all three per pair and the FMA pipe is left with  g = num * rsqrt(as2 * w2), the clamped acos and the
// hinge -- 13 FMA-pipe operations per score instead of ~30 for the in-register algebra + dot product.  fp32
// accuracy comes from the 3xTF32 split
//     x' = x_hi + x_lo,  y' = y_hi + y_lo   (hi = tf32 round-to-nearest, lo = tf32(rest))
//     <x', y'> ~= y_hi.x_hi + y_hi.x_lo + y_lo.x_hi      (the dropped lo.lo term is 2^-22 |x'||y'|)
// issued as three K-passes over the same accumulator.  Each epilogue thread owns one image (= one TMEM lane) and
// 16 labels of the chunk, pulls its 3 x 16 columns with tcgen05.ld, releases the accumulator at once (so the
// MMAs of the next chunk overlap the arithmetic even with a single accumulator buffer) and runs the epilogue on
// packed label PAIRS (fma.rn.f32x2), then either stores the label-major score matrix (32 consecutive images per
// warp store: coalesced) or feeds the per-level top-k (register-resident k-best list per thread, deferred-angle
// filter, shared-memory candidate ring; see TopList and the epilogue).
//
// Data movement:
//   labels  -> lec_score_mma_prep (one small launch): per chunk of 32 labels a "blob" in the caller's
//              workspace = B_hi tile | B_lo tile (96 rows, K-major, no-swizzle UMMA canonical layout) | per-label-pair
//              constants {pi/2 - psi, cos psi, sin psi} (fp64-computed, same terms as lec_rows_fwd's aux) | header;
//              plus one (pi/2 - psi)[L] table for the top-k merge.  The main kernel pulls a blob with two cp.async.bulk copies
//              (TMA, mbarrier complete_tx): the tiles into a tile stage that the MMAs' completion frees, the constants
//              + header into a constant stage that the epilogue frees.
//   images  -> each CTA reads its 128 rows once, splits [y, |y|^2, 1] into hi/lo and writes them to tensor memory
//              as the A operand (tcgen05.st, TS-form MMA).
//   accumulators: TMEM, 1 or 2 buffers of 96 columns so that a CTA stays within 256 columns and two CTAs share an SM.
//
// UMMA canonical layout used for the B operand (Major-K, SWIZZLE_NONE; cute/atom/mma_traits_sm100.hpp
// "((8,n),2):((1,SBO),LBO)" in 16-byte units): a core matrix is 8 rows x 16 bytes stored contiguously
// (128 B); element (row r, k) of a tile with R rows lives at byte (k/4)*(16 R) + 16 r + 4 (k%4), i.e.
// LBO = 16 R (next 16-byte K group), SBO = 128 (next 8 rows).  One MMA consumes K = 8 tf32 = two K groups.
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "lec_common.cuh"
#include "lec_packed.cuh"
#include "lec_async.cuh"

namespace lec {

constexpr int kMmaM = 128;       // images per CTA (TMEM lanes)
constexpr int kMmaN = 96;        // B rows per chunk = TMEM columns per accumulator buffer
// FORMS = 3: the rows of a chunk are num | w2 | as2 of 32 labels (all pair algebra on the tensor pipe: 9 K-passes per
// score); FORMS = 1: plain label rows of 96 labels, p = <x, y> only, the pair algebra stays on the FMA pipe.  Three
// forms triple the tensor work (3 forms x 3 TF32 passes x Kp MACs per score), which the tensor pipe hides behind the
// epilogue only while Kp <= 32; wider rows keep one form.
constexpr int kMmaMaxChunks = 224;
constexpr int kMmaRing = 24;      // candidate ring entries per epilogue thread (top-k launches)
constexpr int kMmaRingRoom = 16;  // room a thread needs between two merge checks: one group of 16 labels

struct MmaChunk { int label0; short count; signed char level; unsigned char flags; };  // flags: 1 first, 2 last chunk of its level
struct MmaChunkTable { int n; MmaChunk c[kMmaMaxChunks]; };

struct MmaHdr { int label0, count, level, flags; float psi_max; int pad[3]; };  // 32 bytes, tail of a blob

// Forms per launch.  Rows up to D = 30 (D + 2 padded to <= 32): three forms in every mode.  Wider rows keep one form --
// three would triple a tensor time that is no longer hidden (r2 sweep at D = 50, Kp = 56: matrix 1.12 -> 1.34 ms, top-k
// 1.67 -> 1.91 ms) -- except in the matrix + top-k mode, whose epilogue is long enough to hide it and short of issue
// slots for the pair algebra (2.51 -> 2.16 ms), up to Kp = 56 (D <= 54).
inline int mma_forms(int D, bool matrix_and_topk = false) {
    const int kp3 = (D + 2 + 7) / 8 * 8;
    return kp3 <= 32 || (matrix_and_topk && kp3 <= 56) ? 3 : 1;
}
__host__ __device__ inline int mma_labels(int forms) { return kMmaN / forms; }                   // labels per chunk
__host__ __device__ inline int mma_kp(int D, int forms) { return ((forms == 3 ? D + 2 : D) + 7) / 8 * 8; }  // forms 3: [row, |row|^2-slot, 1-slot]
__host__ __device__ inline int mma_tile_bytes(int Kp) { return kMmaN * Kp * 4; }                 // one B tile (hi or lo)
__host__ __device__ inline int mma_const_bytes(int forms) { return (mma_labels(forms) / 2) * 12 * 4; }   // 12 floats per label pair
__host__ __device__ inline int mma_blob_bytes(int Kp, int forms) { return 2 * mma_tile_bytes(Kp) + mma_const_bytes(forms) + (int)sizeof(MmaHdr); }

__device__ __forceinline__ float to_tf32(float v) {
    unsigned r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

// ------------------------------------------------------------------------------------------------
// prep: labels -> chunk blobs
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMmaN) score_mma_prep_kernel(const float* __restrict__ labels, int D, int Kp, int forms, float K,
                                                                const MmaChunkTable tab, unsigned char* __restrict__ ws,
                                                                float* __restrict__ npsi) {
    const int c = blockIdx.x, j = threadIdx.x;   // thread j writes B row j: form j / NL of label j % NL
    const int NL = mma_labels(forms);
    const int form = j / NL, jl = j % NL;
    const MmaChunk ch = tab.c[c];
    unsigned char* blob = ws + (size_t)c * mma_blob_bytes(Kp, forms);
    float* hi = reinterpret_cast<float*>(blob);
    float* lo = reinterpret_cast<float*>(blob + mma_tile_bytes(Kp));
    float* cst = reinterpret_cast<float*>(blob + 2 * mma_tile_bytes(Kp));
    const bool live = jl < ch.count;
    const float* src = labels + (int64_t)(ch.label0 + (live ? jl : 0)) * D;
    double A = 0.0;
    for (int k = 0; k < D; ++k) {
        const double v = live ? (double)__ldg(src + k) : 0.0;
        A += v * v;
    }
    // forms == 3:  x'_num = [(1+A) x, -A, -A]   x'_w2 = [-2 x, A, 1]   x'_as2 = [-2A x, A, A^2]   (against y' = [y, B, 1])
    // forms == 1:  x' = x
    double coef = 1.0, tailB = 0.0, tail1 = 0.0;
    if (forms == 3) {
        coef = form == 0 ? 1.0 + A : (form == 1 ? -2.0 : -2.0 * A);
        tailB = form == 0 ? -A : A;
        tail1 = form == 0 ? -A : (form == 1 ? 1.0 : A * A);
    }
    for (int k0 = 0; k0 < Kp; k0 += 4) {
        float h[4], l[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int k = k0 + e;
            double dv = 0.0;
            if (live) {
                if (k < D) dv = coef * (double)__ldg(src + k);
                else if (k == D) dv = tailB;
                else if (k == D + 1) dv = tail1;
            }
            const float v = (float)dv;
            h[e] = to_tf32(v);
            l[e] = to_tf32(v - h[e]);
        }
        const int off = (k0 >> 2) * (kMmaN * 4) + j * 4;  // floats: K group * (16 B * 96 rows) + row * 16 B
        *reinterpret_cast<float4*>(hi + off) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(lo + off) = make_float4(l[0], l[1], l[2], l[3]);
    }
    const double Av = live ? A : 0.25;
    const Aux<double> x = row_aux<double>(LEC_GEOM_HYP, Av, K);
    if (form == 0) {
        const double sp = sin(x.t0), cp = sqrt(fmax(0.0, 1.0 - sp * sp));
        float* q = cst + (jl >> 1) * 12 + (jl & 1);
        const float hpsi = (float)(1.5707963267948966 - x.t0);   // pi/2 - psi: the constant acos_clamped_plus2 adds (fp64-computed)
        if (live) npsi[ch.label0 + jl] = hpsi;   // per-label copy for the top-k merge (candidates outlive their blob)
        if (forms == 3) {   // {pi/2-psi, pi/2-psi', cos psi, cos psi'} {sin psi, sin psi', 0, 0} {0, 0, 0, 0}
            q[0] = hpsi; q[2] = (float)cp; q[4] = (float)sp; q[6] = 0.f; q[8] = 0.f; q[10] = 0.f;
        } else {            // {A, A', 1+A, 1+A'} {A^2, A'^2, pi/2-psi, pi/2-psi'} {cos psi, cos psi', sin psi, sin psi'}
            q[0] = (float)Av; q[2] = (float)(1.0 + Av); q[4] = (float)(Av * Av); q[6] = hpsi;
            q[8] = (float)cp; q[10] = (float)sp;
        }
    }
    // largest half-aperture of the chunk (for the deferred-angle filter's validity test thr + psi <= pi)
    float pm = live ? (float)x.t0 : -INFINITY;
    __shared__ float wmax[kMmaN / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) pm = fmaxf(pm, __shfl_xor_sync(0xffffffffu, pm, o));
    if ((j & 31) == 0) wmax[j >> 5] = pm;
    __syncthreads();
    if (j == 0) {
        MmaHdr* h = reinterpret_cast<MmaHdr*>(blob + 2 * mma_tile_bytes(Kp) + mma_const_bytes(forms));
        h->label0 = ch.label0; h->count = ch.count; h->level = ch.level; h->flags = ch.flags;
        h->psi_max = fmaxf(wmax[0], fmaxf(wmax[1], wmax[2]));
        h->pad[0] = h->pad[1] = h->pad[2] = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// PTX wrappers (tcgen05 / mbarrier / bulk copy)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(unsigned dst_smem, unsigned cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(unsigned taddr, unsigned cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(unsigned bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, kind::tf32, issued by one thread
__device__ __forceinline__ void tc_mma_tf32(unsigned d_tmem, uint64_t a_desc, uint64_t b_desc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// same with the A operand read from tensor memory (lane = row, one 32-bit column per K element)
__device__ __forceinline__ void tc_mma_tf32_ts(unsigned d_tmem, unsigned a_tmem, uint64_t b_desc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// this thread's lane, 8 consecutive columns
__device__ __forceinline__ void tmem_st8(unsigned taddr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                   "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                   "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])) : "memory");
}
__device__ __forceinline__ void tmem_ld16(unsigned taddr, float (&v)[16]) {
    unsigned r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// three 16-column loads of this thread's lane in flight together, one wait
__device__ __forceinline__ void tmem_ld16x3(unsigned t0, unsigned t1, unsigned t2, float (&a)[16], float (&b)[16], float (&c)[16]) {
    unsigned r[48];
#define LEC_LD16(OFF, ADDR)                                                                                                   \
    asm volatile(                                                                                                             \
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];" \
        : "=r"(r[OFF + 0]), "=r"(r[OFF + 1]), "=r"(r[OFF + 2]), "=r"(r[OFF + 3]), "=r"(r[OFF + 4]), "=r"(r[OFF + 5]),          \
          "=r"(r[OFF + 6]), "=r"(r[OFF + 7]), "=r"(r[OFF + 8]), "=r"(r[OFF + 9]), "=r"(r[OFF + 10]), "=r"(r[OFF + 11]),       \
          "=r"(r[OFF + 12]), "=r"(r[OFF + 13]), "=r"(r[OFF + 14]), "=r"(r[OFF + 15])                                          \
        : "r"(ADDR) : "memory")
    LEC_LD16(0, t0);
    LEC_LD16(16, t1);
    LEC_LD16(32, t2);
#undef LEC_LD16
    // the wait names every destination register as read-write, so no use of a loaded value can be scheduled above it
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 48; ++i) asm volatile("" : "+r"(r[i]));
#pragma unroll
    for (int i = 0; i < 16; ++i) { a[i] = __uint_as_float(r[i]); b[i] = __uint_as_float(r[16 + i]); c[i] = __uint_as_float(r[32 + i]); }
}
// shared-memory matrix descriptor: Major-K, SWIZZLE_NONE, version 1 (cute/arch/mma_sm100_desc.hpp SmemDescriptor)
__device__ __forceinline__ uint64_t umma_desc(unsigned saddr, unsigned lbo_bytes, unsigned sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32) | (1ull << 46);
}
// instruction descriptor (InstrDescriptor): D fp32, A/B tf32, both K-major, N = 64, M = 128
__host__ __device__ constexpr unsigned umma_idesc_tf32(int M, int Nn) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(Nn >> 3) << 17) | ((unsigned)(M >> 4) << 24);
}

struct MmaArgs {
    const float* images; int64_t N; int D; int Kp;
    const unsigned char* ws; int n_chunks;
    float* scores;           // label-major [L, N] or NULL
    int32_t* topk_idx; float* topk_val; int k, n_levels;
    const float* npsi;       // [L] pi/2 - psi(label), written by the prep launch (top-k merge of deferred candidates)
    int ring;                // candidate ring entries per thread
    int stages;              // label-tile stages in shared memory (1..4), released by the MMAs that read them
    int cstages;             // constant + header stages (1..4), released by the epilogue threads
    int acc_stages;          // accumulator buffers in TMEM (1 or 2)
    int tmem_cols;           // power of two >= acc_stages * 96 + 2 Kp
};

constexpr int kMmaMaxStages = 4;

// Optional cycle trace of the pipeline (build with -DLEC_TC_TRACE; LEC_TC_TRACE=0 silences it): sums of clock64 deltas over
// all CTAs, printed by the launcher.  [0] MMA warp waits for tiles  [1] MMA warp waits for a free accumulator  [2] MMA
// issue  [3] chunks issued  [4] epilogue (first thread of each 4-warp group) waits for constants  [5] ... for the
// accumulator  [6] TMEM loads  [7] whole chunk loop  [8] chunk visits  [9] MMA issue -> accumulator seen by the epilogue
// [10] CTA prologue (start -> first MMA may issue)  [11] CTAs
#ifdef LEC_TC_TRACE
__device__ unsigned long long g_tc_trace[16];
#define TC_T0(var) const long long var = clock64()
#define TC_ADD(slot, var) trace_acc[slot] += clock64() - (var)
#else
#define TC_T0(var)
#define TC_ADD(slot, var)
#endif
constexpr int kEpiThreads = 2 * kMmaM;          // 8 epilogue warps: two threads per image, 16 labels (3 x 16 columns) each
constexpr int kMmaThreads = kEpiThreads + 64;   // + warp 8 (tcgen05.mma issue) + warp 9 (TMA bulk copies)

__device__ __forceinline__ void tmem_ld32(unsigned taddr, float (&v)[32]) {
    unsigned r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}


// Sorted k-best list of one epilogue thread, register resident for the whole level (r1f profile: with the list in
// shared memory and a runtime k, one merged candidate cost ~135 issue slots and merges were 37 % of the top-k kernel).
// KK = 5 serves the reference's k = 5; KK = LEC_MAX_TOPK keeps the 8 best and reports the first k.
template <int KK>
struct TopList {
    float v[KK];
    int l[KK];
    __device__ __forceinline__ void reset() {
#pragma unroll
        for (int q = 0; q < KK; ++q) { v[q] = INFINITY; l[q] = -1; }
    }
    __device__ __forceinline__ void shift_in(const bool (&b)[KK], float E, int lab) {
#pragma unroll
        for (int q = KK - 1; q > 0; --q) {
            v[q] = b[q - 1] ? v[q - 1] : (b[q] ? E : v[q]);
            l[q] = b[q - 1] ? l[q - 1] : (b[q] ? lab : l[q]);
        }
        v[0] = b[0] ? E : v[0];
        l[0] = b[0] ? lab : l[0];
    }
    // A thread meets its labels in ascending order, so an entry of its own stream carries a higher label than anything
    // already listed: a strict compare keeps ties in label order.  NaN never enters (torch.topk ranks it last).
    __device__ __forceinline__ void insert_ascending(float E, int lab) {
        bool b[KK];
#pragma unroll
        for (int q = 0; q < KK; ++q) b[q] = E < v[q];
        shift_in(b, E, lab);
    }
    // entry of another stream (the peer thread's list): ties go to the lower label; empty slots carry label -1
    __device__ __forceinline__ void insert_any(float E, int lab) {
        bool b[KK];
#pragma unroll
        for (int q = 0; q < KK; ++q) b[q] = E < v[q] || (E == v[q] && (unsigned)lab < (unsigned)l[q]);
        shift_in(b, E, lab);
    }
    __device__ __forceinline__ float kth(int k) const {
        if (KK == 5) return v[4];
        float r = v[0];
#pragma unroll
        for (int q = 1; q < KK; ++q) r = (q < k) ? v[q] : r;
        return r;
    }
};

// Warp roles: warps 0..7 = epilogue (warp w reads TMEM lanes 32 (w % 4) .., labels 16 (w / 4) .. of every chunk),
// warp 8 = MMA issuer (warp-uniform code so descriptors live in uniform registers; one lane issues), warp 9 =
// loader (one lane issues the bulk copies).  Pipelines: full[s] (blob landed in stage s), done[t] (accumulator t
// complete), accfree[t] (all 256 epilogue threads hold accumulator t's values in registers), empty[s] (all 256
// epilogue threads are finished with the constants of blob stage s, whose MMAs have completed).
// MODE 0: top-k only (deferred angle), 1: matrix only, 2: matrix + top-k.  KK: slots of the per-thread k-best list.
template <int MODE, int FORMS, int KK>
__global__ void __launch_bounds__(kMmaThreads, 2) score_mma_kernel(const MmaArgs a) {
    constexpr int NL = kMmaN / FORMS;        // labels per chunk
    constexpr int LT = NL / 2;               // labels per epilogue thread and chunk
    constexpr int GROUPS = LT / 16;          // groups of 16 labels (8 packed pairs) per thread and chunk
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int Kp = a.Kp, KS = Kp >> 3;
    const int b_tile = mma_tile_bytes(Kp);
    const int blob = mma_blob_bytes(Kp, FORMS);
    const int NS = a.stages, NC = a.cstages;
    // A blob travels in two bulk copies: its B_hi | B_lo tiles into a tile stage, which the MMAs' own completion frees
    // (tcgen05.commit on tfree[s]), and its constants + header into a small constant stage that the epilogue threads
    // hold for the whole chunk.  Wide rows (D = 50: 43 KB of tiles per chunk) then need a single tile stage and two
    // CTAs fit an SM in every mode (r1f profile: the top-k launches ran one CTA per SM at 37 % issue utilisation).
    const int tiles = 2 * b_tile, cbytes = blob - tiles, cstride = (cbytes + 127) & ~127;
    unsigned char* sB = smem_raw;                // NS tile stages
    unsigned char* sC = sB + (size_t)NS * tiles; // NC constant stages
    // top-k launches: final lists of the second thread of every image [2 buffers][KK][128] {E, label}, the k-th best
    // every thread publishes for its peer [256] {E, level}, candidate ring [ring][256] {E or g, label}
    float2* top = reinterpret_cast<float2*>(sC + (size_t)NC * cstride);
    float2* thr_pub = top + (MODE == 1 ? 0 : 2 * KK * kMmaM);
    float2* ring = thr_pub + (MODE == 1 ? 0 : kEpiThreads);
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)a.ring * kEpiThreads);  // full[4], done[4], empty[4], accfree[4], tfull[4], tfree[4]
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 6 * kMmaMaxStages);

    const int tid = threadIdx.x, warp = tid >> 5;
#ifdef LEC_TC_TRACE
    const long long cta_t0 = clock64();
    __shared__ long long trace_issue[256];
#endif
    const int NA = a.acc_stages;
    const unsigned bar_full0 = smem_u32(bars), bar_done0 = smem_u32(bars + kMmaMaxStages), bar_empty0 = smem_u32(bars + 2 * kMmaMaxStages);
    const unsigned bar_accfree0 = smem_u32(bars + 3 * kMmaMaxStages);
    const unsigned bar_tfull0 = smem_u32(bars + 4 * kMmaMaxStages), bar_tfree0 = smem_u32(bars + 5 * kMmaMaxStages);
    // tensor memory: NA accumulator buffers of 96 columns, then the image tile as the A operand: A_hi | A_lo, Kp
    // columns each (lane = image row); the host rounded the total up to a power of two
    const unsigned col_ahi = (unsigned)(NA * kMmaN), col_alo = col_ahi + (unsigned)Kp;
    const unsigned tmem_cols = (unsigned)a.tmem_cols;

    if (warp == 8) tmem_alloc(smem_u32(tmem_slot), tmem_cols);   // the allocating warp also frees
    if (tid == 0) {
        for (int s = 0; s < kMmaMaxStages; ++s) {
            mbar_init(bar_full0 + 8 * s, 1);
            mbar_init(bar_done0 + 8 * s, 1);
            mbar_init(bar_tfull0 + 8 * s, 1);
            mbar_init(bar_tfree0 + 8 * s, 1);
            // matrix-only launches with two accumulators split the chunks between the two 4-warp groups (see the
            // epilogue): a stage is then released by the 128 threads of its owner group only
            const unsigned owners = (MODE == 1 && NA == 2) ? kEpiThreads / 2 : kEpiThreads;
            mbar_init(bar_empty0 + 8 * s, owners);
            mbar_init(bar_accfree0 + 8 * s, owners);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // no level is published yet (shared memory arrives with whatever the previous CTA left there)
    if (MODE != 1 && tid < kEpiThreads) thr_pub[tid] = make_float2(INFINITY, __int_as_float(-1));

    // ---- image rows -> the A operand in tensor memory.  Two threads per row: warps 0-3 write the tf32 hi parts,
    //      warps 4-7 the lo parts (a warp can only touch TMEM lanes 32 (warp % 4) ..); both keep |y|^2.
    tc_fence_before();
    __syncthreads();           // TMEM base address + mbarrier inits visible
    tc_fence_after();
    const unsigned tmem_base = *tmem_slot;
    const int row = tid & (kMmaM - 1), half = (tid >> 7) & 1;
    const int64_t img = (int64_t)blockIdx.x * kMmaM + row;
    const bool img_ok = img < a.N;
    float Bn = 0.f;
    if (tid < kEpiThreads) {
        const float* src = a.images + (img_ok ? img : 0) * (int64_t)a.D;
        const unsigned dst = tmem_base + ((unsigned)((warp & 3) * 32) << 16) + (half ? col_alo : col_ahi);
        if (img_ok)
            for (int k = 0; k < a.D; ++k) { const float v = __ldg(src + k); Bn = fmaf(v, v, Bn); }
        // FORMS == 3: y' = [y, |y|^2, 1, 0 ...];  FORMS == 1: y' = [y, 0 ...]
        for (int k0 = 0; k0 < Kp; k0 += 8) {
            float o[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int k = k0 + e;
                float v = 0.f;
                if (img_ok) v = (k < a.D) ? __ldg(src + k) : ((FORMS == 3 && k == a.D) ? Bn : ((FORMS == 3 && k == a.D + 1) ? 1.f : 0.f));
                const float h = to_tf32(v);
                o[e] = half ? to_tf32(v - h) : h;
            }
            tmem_st8(dst + (unsigned)k0, o);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    } else if (warp == 9 && elect_one()) {
        // the first label blobs stream in while the image tile is being converted
        const unsigned sB_u = smem_u32(sB), sC_u = smem_u32(sC);
        for (int c = 0; c < NS && c < a.n_chunks; ++c) {
            mbar_expect_tx(bar_tfull0 + 8 * c, (unsigned)tiles);
            bulk_g2s(sB_u + c * tiles, a.ws + (size_t)c * blob, (unsigned)tiles, bar_tfull0 + 8 * c);
        }
        for (int c = 0; c < NC && c < a.n_chunks; ++c) {
            mbar_expect_tx(bar_full0 + 8 * c, (unsigned)cbytes);
            bulk_g2s(sC_u + c * cstride, a.ws + (size_t)c * blob + tiles, (unsigned)cbytes, bar_full0 + 8 * c);
        }
    }
    tc_fence_before();
    __syncthreads();           // A operand complete before the first MMA
    tc_fence_after();

    // ================================ producer warps ================================
    if (warp == 9) {
        // loader: the tiles of chunk ct go into tile stage ct % NS as soon as the MMAs of chunk ct - NS have completed,
        // the constants of chunk cc into constant stage cc % NC once the epilogue of chunk cc - NC has released it.
        // One thread serves both streams and never blocks on one while the other could move.
        if (elect_one()) {
            const unsigned sB_u = smem_u32(sB), sC_u = smem_u32(sC);
            int ct = NS, st = 0, cc = NC, sc = 0;
            unsigned part = 0, parc = 0, idle = 0;
            while (ct < a.n_chunks || cc < a.n_chunks) {
                bool moved = false;
                if (ct < a.n_chunks && mbar_test(bar_tfree0 + 8 * st, part)) {
                    mbar_expect_tx(bar_tfull0 + 8 * st, (unsigned)tiles);
                    bulk_g2s(sB_u + st * tiles, a.ws + (size_t)ct * blob, (unsigned)tiles, bar_tfull0 + 8 * st);
                    ++ct;
                    if (++st == NS) { st = 0; part ^= 1u; }
                    moved = true;
                }
                if (cc < a.n_chunks && mbar_test(bar_empty0 + 8 * sc, parc)) {
                    mbar_expect_tx(bar_full0 + 8 * sc, (unsigned)cbytes);
                    bulk_g2s(sC_u + sc * cstride, a.ws + (size_t)cc * blob + tiles, (unsigned)cbytes, bar_full0 + 8 * sc);
                    ++cc;
                    if (++sc == NC) { sc = 0; parc ^= 1u; }
                    moved = true;
                }
                if (moved) idle = 0;
                else {
                    __nanosleep(kMbarSleepNs);
                    if (++idle > (1u << 24)) __trap();   // a lost arrival traps instead of hanging the GPU
                }
            }
        }
        __syncwarp();
    } else if (warp == 8) {
        // MMA issuer: chunk c needs its tiles (tfull[c % NS]) and an accumulator buffer, which is free as soon as every
        // epilogue thread that reads it has pulled the previous chunk out of it (accfree), i.e. before that chunk's
        // arithmetic.  The whole issue sequence runs on one elected lane with warp-uniform operands, so it compiles to
        // uniform-datapath code (UTCHMMA back to back); r2 trace: with `if (lane == 0)` around each tcgen05.mma the
        // compiler serialised every operand through an ELECT / R2UR.BROADCAST loop and one chunk took ~1500 cycles to
        // issue -- the epilogue warps spent a third of their time waiting for accumulators.
        const unsigned sB_u = smem_u32(sB);
        const unsigned idesc = umma_idesc_tf32(kMmaM, kMmaN);
#ifdef LEC_TC_TRACE
        long long trace_acc[4] = {0, 0, 0, 0};
        trace_acc[3] = a.n_chunks;
        if ((tid & 31) == 0) { atomicAdd(&g_tc_trace[10], (unsigned long long)(clock64() - cta_t0)); atomicAdd(&g_tc_trace[11], 1ull); }
#endif
        auto issue = [&](int c, int s, int t) {
            (void)c;
            tc_fence_after();
            const unsigned d = tmem_base + (unsigned)(t * kMmaN);
            const unsigned bh = sB_u + s * tiles, bl = bh + b_tile;
            if (elect_one()) {
                // the descriptors of a stage differ in the 14-bit start-address field only: one add per MMA
                const uint64_t dh = umma_desc(bh, kMmaN * 16, 128), dl = umma_desc(bl, kMmaN * 16, 128);
                unsigned acc = 0;
#pragma unroll 1
                for (int pass = 0; pass < 3; ++pass) {
                    const unsigned pa = tmem_base + ((pass == 2) ? col_alo : col_ahi);   // hi.hi, hi.lo, lo.hi
                    const uint64_t pb = (pass == 1) ? dl : dh;
                    for (int ks = 0; ks < KS; ++ks) {
                        tc_mma_tf32_ts(d, pa + (unsigned)(ks * 8), pb + (uint64_t)(ks * ((2 * kMmaN * 16) >> 4)), idesc, acc);
                        acc = 1;
                    }
                }
                tc_commit(bar_done0 + 8 * t);    // accumulator of chunk c complete -> epilogue
                tc_commit(bar_tfree0 + 8 * s);   // tile stage s read -> loader
            }
            __syncwarp();
#ifdef LEC_TC_TRACE
            if ((tid & 31) == 0) trace_issue[c & 255] = clock64();
#endif
        };
        if (MODE == 1 && NA == 2) {
            // Matrix-only launches: each 4-warp epilogue group owns one accumulator and every other chunk.  The two
            // chunk streams are served independently -- whichever group has released its accumulator (and has its tiles)
            // gets its next chunk; with in-order issue the faster group waited for the slower one's release.
            int cn[2] = {0, 1}, sg[2] = {0, 1 % NS};
            unsigned ps[2] = {0u, (unsigned)((1 / NS) & 1)}, pa_[2] = {0u, 0u};
            unsigned idle = 0;
            while (cn[0] < a.n_chunks || cn[1] < a.n_chunks) {
                bool any = false;
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    const int c = cn[g];
                    if (c >= a.n_chunks) continue;
                    if (!mbar_test(bar_tfull0 + 8 * sg[g], ps[g])) continue;
                    if (c >= 2) {
                        if (!mbar_test(bar_accfree0 + 8 * g, pa_[g])) continue;
                        pa_[g] ^= 1u;
                    }
                    issue(c, sg[g], g);
                    cn[g] = c + 2;
                    sg[g] += 2;
                    while (sg[g] >= NS) { sg[g] -= NS; ps[g] ^= 1u; }
                    any = true;
                }
                if (any) idle = 0;
                else {
                    __nanosleep(20);
                    if (++idle > (1u << 24)) __trap();   // a lost arrival traps instead of hanging the GPU
                }
            }
        } else {
            int s = 0, t = 0;
            unsigned par = 0, par_t = 1;   // accfree[t] is first waited on for chunk NA, i.e. after one wrap of t
            for (int c = 0; c < a.n_chunks; ++c) {
                TC_T0(w0);
                mbar_wait(bar_tfull0 + 8 * s, par);
                TC_ADD(0, w0);
                TC_T0(w1);
                if (c >= NA) mbar_wait(bar_accfree0 + 8 * t, par_t);
                TC_ADD(1, w1);
                TC_T0(w2);
                issue(c, s, t);
                TC_ADD(2, w2);
                if (++s == NS) { s = 0; par ^= 1u; }
                if (++t == NA) { t = 0; par_t ^= 1u; }
            }
        }
        __syncwarp();
#ifdef LEC_TC_TRACE
        if ((tid & 31) == 0) for (int q = 0; q < 4; ++q) atomicAdd(&g_tc_trace[q], (unsigned long long)trace_acc[q]);
#endif
    } else {
        // ================================ epilogue warps ================================
        const u64 B2 = pack2(Bn, Bn), C2 = pack2(-1.f - Bn, -1.f - Bn);   // FORMS == 1 only
        (void)B2; (void)C2;
        const int k = a.k;
        const int et = tid;  // 0..255: slot in the per-thread ring / published-threshold arrays
        const unsigned ring0 = smem_u32(ring + et);
        unsigned rp = ring0;
        const unsigned ring_trigger = ring0 + (unsigned)(a.ring - kMmaRingRoom) * kEpiThreads * 8;
        float thr = INFINITY;                  // MODE 2: k-th best energy so far
        float cT = 0.f, nsT = 0.f, off = -INFINITY;  // MODE 0: accept g >= cT cos(psi) - sT sin(psi) + off
        float psi_max = 0.f;
        int level = -1, lvl_buf = 0;
        TopList<KK> list;
        list.reset();

        auto refresh = [&]() {
            // both threads of an image feed one top-k: the tighter of the two k-th bests bounds either stream.  The peer's
            // published value counts only while it is working on the same level (it may be a chunk ahead or behind).
            // Deliberately unsynchronised (compute-sanitizer racecheck flags this read against publish()): value and
            // level tag travel in one aligned 8-byte store / load, and ANY value the peer published for this level is
            // a valid upper bound of the image's k-th best.
            const float2 pe = thr_pub[et ^ kMmaM];
            const float t = fminf(list.kth(k), __float_as_int(pe.y) == level ? pe.x : INFINITY);
            thr = t;
            if (t <= 0.f) { cT = 0.f; nsT = 0.f; off = INFINITY; }
            else if (!(t + psi_max <= 3.1415f)) { cT = 0.f; nsT = 0.f; off = -INFINITY; }
            else { float sn, cs; __sincosf(t, &sn, &cs); cT = cs; nsT = -sn; off = -4e-6f; }
        };
        auto publish = [&]() { thr_pub[et] = make_float2(list.kth(k), __int_as_float(level)); };
        auto merge = [&]() {
            // ring entries two at a time: one packed acos serves both (MODE 0: the ring holds g; the same instruction
            // sequence as the matrix path, so deferred and direct energies agree bit for bit)
            const int cnt = (int)((rp - ring0) / (kEpiThreads * 8));
            for (int j = 0; j < cnt; j += 2) {
                const bool two = j + 1 < cnt;
                const float2 e0 = ring[j * kEpiThreads + et];
                const float2 e1 = ring[(two ? j + 1 : j) * kEpiThreads + et];
                const int lab0 = __float_as_int(e0.y), lab1 = __float_as_int(e1.y);
                float E0 = e0.x, E1 = e1.x;
                if (MODE == 0) {
                    const float np0 = __ldg(a.npsi + lab0), np1 = __ldg(a.npsi + lab1);
                    float z0, z1;
                    unpack2(acos_clamped_plus2(pack2(e0.x, e1.x), pack2(np0, np1)), z0, z1);
                    E0 = max_nan(z0, 0.f);
                    E1 = max_nan(z1, 0.f);
                }
                list.insert_ascending(E0, lab0);
                if (two) list.insert_ascending(E1, lab1);
            }
            if (cnt > 0) publish();
            rp = ring0;
            refresh();
        };

        const int lane_base = (warp & 3) * 32;
        const unsigned row_bytes = (unsigned)a.N * 4u;   // bytes between two label rows of the score matrix (the host checks N < 2^30)
        // Chunk ownership.  Top-k launches: every epilogue thread visits every chunk and takes half of its labels (the two
        // threads of an image keep separate lists, merged at the end of a level).  Matrix-only launches with two
        // accumulator buffers (ALT): warps 0-3 take the even chunks and warps 4-7 the odd ones, all labels of the chunk in
        // two batches -- half as many barrier / header / TMEM-load prologues per warp, and the two groups run out of
        // phase, so their MUFU- and FMA-heavy stretches interleave on an SM sub-partition instead of colliding.
        const bool alt = (MODE == 1) && NA == 2;
        const int cstep = alt ? 2 : 1;
        // stage indices and phase parities advance by increments (no integer division in the chunk loop)
        int s = alt ? half : 0, t = alt ? half : 0;
        unsigned par = 0, par_t = 0;
        while (s >= NC) { s -= NC; par ^= 1u; }
#ifdef LEC_TC_TRACE
        long long trace_acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        const bool tracer = (tid & 127) == 0;
        const long long loop_t0 = clock64();
#endif
        for (int c = alt ? half : 0; c < a.n_chunks; c += cstep) {
            TC_T0(e0);
            mbar_wait(bar_full0 + 8 * s, par);   // constants + header of chunk c visible to this thread
            TC_ADD(4, e0);
            const unsigned char* bl = sC + (size_t)s * cstride;
            const float* cst = reinterpret_cast<const float*>(bl);
            const MmaHdr hdr = *reinterpret_cast<const MmaHdr*>(bl + mma_const_bytes(FORMS));
            const bool want_topk = (MODE != 1) && hdr.level >= 0;
            if (want_topk) {
                if (hdr.flags & 1) {
                    list.reset();
                    rp = ring0;
                    level = hdr.level;
                    publish();
                }
                psi_max = hdr.psi_max;
                refresh();
            }
            TC_T0(e1);
            mbar_wait(bar_done0 + 8 * t, par_t);   // accumulator of chunk c complete
            TC_ADD(5, e1);
#ifdef LEC_TC_TRACE
            trace_acc[9] += clock64() - trace_issue[c & 255];
            trace_acc[8] += 1;
#endif
            tc_fence_after();

            const bool store = (MODE != 0) && a.scores != nullptr && img_ok;
            for (int hb = 0; hb < cstep; ++hb) {
            const int lbase = (alt ? hb : half) * LT;        // first label of this batch within the chunk
            // 48 accumulator columns -> registers; the accumulator buffer is released right after the last batch's load.
            // FORMS == 3: v[0] = num, v[1] = w2, v[2] = A s^2 of 16 labels;  FORMS == 1: v[gi] = p of labels 16 gi ..
            float v[3][16];
            {
                const unsigned tcol = tmem_base + ((unsigned)lane_base << 16) + (unsigned)(t * kMmaN);
                TC_T0(e2);
                tmem_ld16x3(tcol + (unsigned)lbase, tcol + (unsigned)(FORMS == 3 ? NL + lbase : lbase + 16),
                            tcol + (unsigned)(FORMS == 3 ? 2 * NL + lbase : lbase + 32), v[0], v[1], v[2]);
                TC_ADD(6, e2);
            }
            if (hb == cstep - 1) {
                tc_fence_before();
                mbar_arrive(bar_accfree0 + 8 * t);
            }
#pragma unroll
            for (int gi = 0; gi < GROUPS; ++gi) {
                const int gbase = lbase + 16 * gi;               // first label of this group within the chunk
                const int g_count = hdr.count - gbase;           // labels of the group that exist
                if (g_count <= 0) break;                         // uniform over the CTA half
                const float* cp = cst + (gbase >> 1) * 12;
                // ---- cos of the cone angle for 8 label pairs, branch-free so that the 8 dependent chains interleave
                u64 g[8], NPSI[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    u64 num, d2;
                    if (FORMS == 3) {
                        const float2 k1 = *reinterpret_cast<const float2*>(cp + q * 12);        // pi/2 - psi, pi/2 - psi'
                        NPSI[q] = pack2(k1.x, k1.y);
                        num = pack2(v[0][2 * q], v[0][2 * q + 1]);
                        d2 = fmul2(pack2(v[2][2 * q], v[2][2 * q + 1]), pack2(v[1][2 * q], v[1][2 * q + 1]));   // A s^2 w^2
                    } else {
                        const float4 k0 = *reinterpret_cast<const float4*>(cp + q * 12);       // A, A', 1+A, 1+A'
                        const float4 k1 = *reinterpret_cast<const float4*>(cp + q * 12 + 4);   // A^2, A'^2, pi/2 - psi, pi/2 - psi'
                        const u64 A2 = pack2(k0.x, k0.y), A12 = pack2(k0.z, k0.w), ASQ = pack2(k1.x, k1.y);
                        NPSI[q] = pack2(k1.z, k1.w);
                        const u64 P = pack2(v[gi][2 * q], v[gi][2 * q + 1]);
                        const u64 qq = fmul2(P, pack2(-2.f, -2.f));
                        num = ffma2(P, A12, fmul2(A2, C2));                                      // p(1+A) - A(1+B)
                        const u64 w2 = fadd2(qq, ffma2(A2, B2, pack2(1.f, 1.f)));               // 1 + AB - 2p
                        const u64 as2 = ffma2(A2, qq, ffma2(A2, B2, ASQ));                      // A (A + B - 2p)
                        d2 = fmul2(as2, w2);
                    }
                    float d0, d1;
                    unpack2(d2, d0, d1);
                    g[q] = fmul2(num, pack2(rsqrt_approx(d0), rsqrt_approx(d1)));
                }
                const int lab0 = hdr.label0 + gbase;
                if (MODE == 0) {
                    if (FORMS == 3 && want_topk && (hdr.flags & 1) && gi == 0) {
                        // first group of a level: the list is empty, so every label is a candidate -- skip the ring and
                        // insert the 16 energies directly (same packed acos as the matrix path; uniform over the warp).
                        // Short rows only: in the FORMS == 1 kernel the extra code spills (D=50 top-k 1.81 -> 2.23 ms).
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            float z0, z1;
                            unpack2(acos_clamped_plus2(g[q], NPSI[q]), z0, z1);
                            if (2 * q < g_count) list.insert_ascending(max_nan(z0, 0.f), lab0 + 2 * q);
                            if (2 * q + 1 < g_count) list.insert_ascending(max_nan(z1, 0.f), lab0 + 2 * q + 1);
                        }
                        publish();
                        refresh();
                    } else if (want_topk) {
                        // deferred angle: E < thr  <=>  g > cos(thr + psi); candidates go to the ring as {g, label}
                        u64 cb[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float4 kc = *reinterpret_cast<const float4*>(cp + q * 12 + (FORMS == 3 ? 0 : 8));
                            const float2 ks = *reinterpret_cast<const float2*>(cp + q * 12 + (FORMS == 3 ? 4 : 10));
                            const u64 COS = FORMS == 3 ? pack2(kc.z, kc.w) : pack2(kc.x, kc.y);
                            cb[q] = ffma2(pack2(cT, cT), COS, ffma2(pack2(nsT, nsT), pack2(ks.x, ks.y), pack2(off, off)));
                        }
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            float g0, g1, b0, b1;
                            unpack2(g[q], g0, g1);
                            unpack2(cb[q], b0, b1);
                            if (2 * q < g_count && g0 >= b0) {
                                asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(rp), "f"(g0), "r"(lab0 + 2 * q) : "memory");
                                rp += kEpiThreads * 8;
                            }
                            if (2 * q + 1 < g_count && g1 >= b1) {
                                asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(rp), "f"(g1), "r"(lab0 + 2 * q + 1) : "memory");
                                rp += kEpiThreads * 8;
                            }
                        }
                        if (__any_sync(0xffffffffu, rp > ring_trigger)) merge();
                    }
                } else {
                    float E[16];
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        float z0, z1;
                        unpack2(acos_clamped_plus2(g[q], NPSI[q]), z0, z1);
                        E[2 * q] = max_nan(z0, 0.f);
                        E[2 * q + 1] = max_nan(z1, 0.f);
                    }
                    if (store) {
                        // row j of the group lives j * 4N bytes further on: a 32 x 32 -> 64 bit multiply-add per store
                        // (IMAD.WIDE.U32) instead of a carried 64-bit add chain
                        char* out = reinterpret_cast<char*>(a.scores + (int64_t)lab0 * a.N + img);
                        if (g_count >= 16) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) *reinterpret_cast<float*>(out + (unsigned long long)row_bytes * (unsigned)j) = E[j];
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (j < g_count) *reinterpret_cast<float*>(out + (unsigned long long)row_bytes * (unsigned)j) = E[j];
                        }
                    }
                    if (MODE == 2 && want_topk) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            if (j < g_count && E[j] < thr) {
                                asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(rp), "f"(E[j]), "r"(lab0 + j) : "memory");
                                rp += kEpiThreads * 8;
                            }
                        }
                        if (__any_sync(0xffffffffu, rp > ring_trigger)) merge();
                    }
                }
            }
            }   // batches
            if (want_topk && (hdr.flags & 2)) {
                merge();
                // The second thread of every image hands its list over (double buffered by level, so its next hand-over
                // cannot overtake the fold) and a barrier of just the two warps that share the 32 images orders it.
                float2* hand = top + (size_t)lvl_buf * (KK * kMmaM) + row;
                if (half) {
#pragma unroll
                    for (int j = 0; j < KK; ++j) hand[j * kMmaM] = make_float2(list.v[j], __int_as_float(list.l[j]));
                }
                switch (warp & 3) {   // immediate barrier ids, so that the kernel reserves five barriers and not all sixteen
                    case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
                    case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
                    case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
                    default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
                }
                if (!half) {
#pragma unroll
                    for (int j = 0; j < KK; ++j) {
                        const float2 e = hand[j * kMmaM];
                        if (__float_as_int(e.y) >= 0) list.insert_any(e.x, __float_as_int(e.y));
                    }
                    if (img_ok) {
                        const int64_t o = (img * a.n_levels + hdr.level) * k;
#pragma unroll
                        for (int j = 0; j < KK; ++j) {
                            if (j < k) {
                                a.topk_idx[o + j] = list.l[j];
                                if (a.topk_val) a.topk_val[o + j] = list.v[j];
                            }
                        }
                    }
                }
                lvl_buf ^= 1;
                level = -1;
            }
            // this thread is done with the constants of stage s
            mbar_arrive(bar_empty0 + 8 * s);
            s += cstep;
            while (s >= NC) { s -= NC; par ^= 1u; }
            if (alt) par_t ^= 1u;
            else if (++t == NA) { t = 0; par_t ^= 1u; }
        }
#ifdef LEC_TC_TRACE
        trace_acc[7] = clock64() - loop_t0;
        if (tracer) for (int q = 4; q < 10; ++q) atomicAdd(&g_tc_trace[q], (unsigned long long)trace_acc[q]);
#endif
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int build_chunks(int64_t L, const int32_t* level_start, const int32_t* level_stop, int n_levels, bool gaps, int NL,
                        MmaChunkTable& t) {
    t.n = 0;
    auto add_segment = [&](int64_t s, int64_t e, int level) -> bool {
        for (int64_t l0 = s; l0 < e || (l0 == s && level >= 0); l0 += NL) {
            if (t.n >= kMmaMaxChunks) return false;
            MmaChunk& c = t.c[t.n++];
            const int64_t cnt = e - l0 < NL ? e - l0 : NL;
            c.label0 = (int)l0; c.count = (short)(cnt < 0 ? 0 : cnt); c.level = (signed char)level;
            c.flags = (unsigned char)((l0 == s ? 1 : 0) | (l0 + NL >= e ? 2 : 0));
            if (e <= s) break;  // empty level: one empty chunk so that its top-k rows are still written
        }
        return true;
    };
    int64_t cursor = 0;
    for (int i = 0; i < n_levels; ++i) {
        int64_t s = level_start[i], e = level_stop[i];
        if (s < cursor || e < s) return LEC_E_K;
        if (e > L) e = L;
        if (s > L) s = L;
        if (gaps && s > cursor && !add_segment(cursor, s, -1)) return LEC_E_SIZE;
        if (!add_segment(s, e, i)) return LEC_E_SIZE;
        cursor = e;
    }
    if (gaps && cursor < L && !add_segment(cursor, L, -1)) return LEC_E_SIZE;
    return 0;
}

static int64_t mma_max_chunks(int64_t L, int n_levels, int NL) { return (L + NL - 1) / NL + 2 * (int64_t)n_levels + 2; }

int64_t score_mma_workspace_bytes(int64_t L, int D, int n_levels) {
    // chunk blobs + the per-label (pi/2 - psi) table the top-k merge reads; the larger of the two layouts a launch may pick
    int64_t best = 0;
    for (int both = 0; both < 2; ++both) {
        const int forms = mma_forms(D, both != 0);
        const int64_t b = mma_max_chunks(L, n_levels, mma_labels(forms)) * mma_blob_bytes(mma_kp(D, forms), forms);
        if (b > best) best = b;
    }
    return best + (L + 32) * 4;
}

// TMEM budget of one CTA: acc_stages accumulator buffers of 96 columns + the image tile (2 Kp columns).  Two buffers
// inside 256 columns when the rows are short (two CTAs per SM), else one buffer inside 256, else two inside 512.
static bool mma_plan(int Kp, int& acc_stages, int& tmem_cols) {
    if (2 * kMmaN + 2 * Kp <= 256) { acc_stages = 2; tmem_cols = 256; return true; }
    if (kMmaN + 2 * Kp <= 256) { acc_stages = 1; tmem_cols = 256; return true; }
    if (2 * kMmaN + 2 * Kp <= 512) { acc_stages = 2; tmem_cols = 512; return true; }
    return false;
}

bool score_mma_supported(int geom, int precision, int D, int64_t L, int n_levels) {
    int na, tc;
    if (!(geom == LEC_GEOM_HYP && precision == LEC_PREC_F32 && D >= 1 && D <= 128)) return false;
    for (int both = 0; both < 2; ++both) {
        const int forms = mma_forms(D, both != 0);
        if (!mma_plan(mma_kp(D, forms), na, tc) || mma_max_chunks(L, n_levels, mma_labels(forms)) > kMmaMaxChunks) return false;
    }
    return true;
}

int score_mma_launch(const float* labels, int64_t L, const float* images, int64_t N, int D, float K, const int32_t* level_start,
                     const int32_t* level_stop, int n_levels, int k, float* scores, int32_t* topk_idx, float* topk_val,
                     void* workspace, int64_t workspace_bytes, cudaStream_t st) {
    if (N == 0 || L == 0) return 0;
    const int forms = mma_forms(D, scores != nullptr && topk_idx != nullptr);
    MmaChunkTable tab;
    if (int e = build_chunks(L, level_start, level_stop, topk_idx ? n_levels : 0, scores != nullptr, mma_labels(forms), tab)) return e;
    if (tab.n == 0) return 0;
    const int Kp = mma_kp(D, forms);
    const int blob = mma_blob_bytes(Kp, forms);
    if ((int64_t)tab.n * blob + L * 4 > workspace_bytes) return LEC_E_SIZE;
    if (reinterpret_cast<uintptr_t>(workspace) & 127) return LEC_E_ALIGN;
    if (topk_idx && (k < 1 || k > LEC_MAX_TOPK)) return LEC_E_K;
    if (scores && N >= (1LL << 30)) return LEC_E_SIZE;   // the kernel keeps the row stride in bytes in 32 bits
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* npsi = reinterpret_cast<float*>(ws + (size_t)tab.n * blob);   // blob sizes are multiples of 32 bytes
    score_mma_prep_kernel<<<tab.n, kMmaN, 0, st>>>(labels, D, Kp, forms, K, tab, ws, npsi);
    ++g_launches;
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return (int)ce;

    MmaArgs a{};
    a.images = images; a.N = N; a.D = D; a.Kp = Kp; a.ws = ws; a.n_chunks = tab.n; a.scores = scores;
    a.topk_idx = topk_idx; a.topk_val = topk_val; a.k = topk_idx ? k : 1; a.n_levels = n_levels;
    a.npsi = npsi;
    a.ring = topk_idx ? kMmaRing : 0;   // matrix-only launches need no candidate ring
    const int kk = (a.k == 5) ? 5 : LEC_MAX_TOPK;
    const size_t fixed = (topk_idx ? (size_t)(2 * kk * kMmaM + kEpiThreads) * 8 : 0) + (size_t)a.ring * kEpiThreads * 8 + 256;
    // Stages.  Constants + header: four small stages (the epilogue holds one per chunk in flight).  Tiles: a stage is
    // free again as soon as the MMAs that read it complete, so one stage already overlaps the copy of chunk c + 1 with
    // the epilogue of chunk c; more only help short rows whose epilogue is as short as a bulk copy.  Within 256 TMEM
    // columns the budget is half an SM's shared memory so that two CTAs (20 warps) stay resident; otherwise the whole SM.
    if (!mma_plan(Kp, a.acc_stages, a.tmem_cols)) return LEC_E_DIM;
    const size_t tiles = 2 * (size_t)mma_tile_bytes(Kp), cstride = ((size_t)blob - tiles + 127) & ~(size_t)127;
    a.cstages = kMmaMaxStages;
    const size_t fixed_c = fixed + (size_t)a.cstages * cstride;
    const size_t half_sm = 113 * 1024, whole_sm = 226 * 1024;
    auto stages_for = [&](size_t budget) { return budget > fixed_c ? (int)((budget - fixed_c) / tiles) : 0; };
    int stages = a.tmem_cols <= 256 ? stages_for(half_sm) : 0;
    if (stages < 1) stages = stages_for(whole_sm);
    if (stages < 1) return LEC_E_DIM;
    a.stages = stages > kMmaMaxStages ? kMmaMaxStages : stages;
    const size_t smem = fixed_c + (size_t)a.stages * tiles;
    const int mode = topk_idx ? (scores ? 2 : 0) : 1;
    const int64_t grid = (N + kMmaM - 1) / kMmaM;
    if (grid > 0x7fffffffLL) return LEC_E_SIZE;
    auto launch = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
#ifdef LEC_TC_TRACE
        static const bool trace_on = [] { const char* e = getenv("LEC_TC_TRACE"); return e == nullptr || atoi(e) != 0; }();
        unsigned long long z[16] = {0};
        if (trace_on) cudaMemcpyToSymbol(g_tc_trace, z, sizeof(z));
#endif
        kern<<<(unsigned)grid, kMmaThreads, smem, st>>>(a);
        ++g_launches;
#ifdef LEC_TC_TRACE
        if (trace_on) {
            cudaStreamSynchronize(st);
            cudaMemcpyFromSymbol(z, g_tc_trace, sizeof(z));
            const double ctas = (double)z[11], ch = (double)z[3], vis = (double)z[8];
            fprintf(stderr, "tc trace mode %d forms %d: CTAs %.0f chunks/CTA %.1f | MMA warp per chunk: wait tiles %.0f, wait acc %.0f, issue %.0f"
                            " | epilogue per visit: wait const %.0f, wait acc %.0f, tmem ld %.0f, issue->seen %.0f | loop per CTA-group %.0f,"
                            " visits %.0f, prologue %.0f cycles\n", mode, forms, ctas, ch / ctas, z[0] / ch, z[1] / ch, z[2] / ch,
                    z[4] / vis, z[5] / vis, z[6] / vis, z[9] / vis, z[7] / (2 * ctas), vis, z[10] / ctas);
        }
#endif
        return (int)cudaGetLastError();
    };
    if (forms == 3) {
        if (mode == 1) return launch(score_mma_kernel<1, 3, 5>);
        if (mode == 0) return kk == 5 ? launch(score_mma_kernel<0, 3, 5>) : launch(score_mma_kernel<0, 3, LEC_MAX_TOPK>);
        return kk == 5 ? launch(score_mma_kernel<2, 3, 5>) : launch(score_mma_kernel<2, 3, LEC_MAX_TOPK>);
    }
    if (mode == 1) return launch(score_mma_kernel<1, 1, 5>);
    if (mode == 0) return kk == 5 ? launch(score_mma_kernel<0, 1, 5>) : launch(score_mma_kernel<0, 1, LEC_MAX_TOPK>);
    return kk == 5 ? launch(score_mma_kernel<2, 1, 5>) : launch(score_mma_kernel<2, 1, LEC_MAX_TOPK>);
}

}  // namespace lec
