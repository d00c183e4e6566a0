// extern "C" surface of liblec_b200.so: argument validation + dispatch.  See include/lec_b200.h.
#include "lec_pairs_impl.cuh"
#include "lec_featnet.cuh"

namespace lec {
std::atomic<unsigned long long> g_launches{0};
thread_local int t_pdl = 0;
#ifdef LEC_STEP_TRACE
unsigned long long* g_step_trace = nullptr;
#endif

// pairs whose endpoint id fell outside the table since the last lec_index_errors(reset) (per device)
__device__ unsigned g_index_errors = 0;
static unsigned* index_errors_ptr() {
    void* p = nullptr;
    return cudaGetSymbolAddress(&p, g_index_errors) == cudaSuccess ? static_cast<unsigned*>(p) : nullptr;
}

int launch_flat_euc32(const FlatArgs&, cudaStream_t);
int launch_flat_hyp32(const FlatArgs&, cudaStream_t);
int launch_flat_hyp64(const FlatArgs&, cudaStream_t);
int launch_flat_oe32(const FlatArgs&, cudaStream_t);
int launch_grouped_euc32(const GroupArgs&, cudaStream_t);
int launch_grouped_hyp32(const GroupArgs&, cudaStream_t);
int launch_grouped_hyp64(const GroupArgs&, cudaStream_t);
int launch_grouped_oe32(const GroupArgs&, cudaStream_t);
int launch_dense_euc32(const DenseArgs&, bool, cudaStream_t);
int launch_dense_hyp32(const DenseArgs&, bool, cudaStream_t);
int launch_dense_hyp64(const DenseArgs&, bool, cudaStream_t);
int launch_dense_oe32(const DenseArgs&, bool, cudaStream_t);

int rows_fwd_launch(const float*, int64_t, int, int, int, float, float*, int, double*, float*, int, int64_t, double*, cudaStream_t);
int rows_bwd_launch(const float*, const float*, int, int64_t, int64_t, int, int, int, float, float*, int, cudaStream_t);
int rsgd_launch(float*, const float*, int, int64_t, int, int, float, float, int, float*, cudaStream_t);
int reduce_replicas_launch(const float*, int, int64_t, float*, cudaStream_t);
int update_rows_launch(const lec_update_t&, const lec_exchange_t*, cudaStream_t);
int64_t two_shot_bytes(int64_t n, int ld, int world);
bool featnet_supported(int F, int D);
int featnet_fwd_launch(const FeatArgs&, cudaStream_t);
int featnet_wgrad_launch(const FeatArgs&, cudaStream_t);
int score_launch(int, int, const float*, int64_t, const float*, int64_t, int, float, const int32_t*, const int32_t*,
                 int, int, float*, int64_t, int64_t, int32_t*, float*, cudaStream_t);

bool score_mma_supported(int geom, int precision, int D, int64_t L, int n_levels);
int64_t score_mma_workspace_bytes(int64_t L, int D, int n_levels);
int score_mma_launch(const float*, int64_t, const float*, int64_t, int, float, const int32_t*, const int32_t*, int, int, float*,
                     int32_t*, float*, void*, int64_t, cudaStream_t);

static int pick_core(int geom, int precision) {
    if (precision != LEC_PREC_F32 && precision != LEC_PREC_F64CORE) return -1;
    switch (geom) {
        case LEC_GEOM_EUC: return CORE_EUC32;  // fp64 core is defined for the hyperbolic energy only
        case LEC_GEOM_HYP: return precision == LEC_PREC_F64CORE ? CORE_HYP64 : CORE_HYP32;
        case LEC_GEOM_OE: return CORE_OE32;
    }
    return -1;
}

static int check_rows(const float* rows, int D, int ld) {
    if (!rows) return LEC_E_NULL;
    if (D < 1 || D > LEC_MAX_DIM || ld < D || (ld & 3)) return LEC_E_DIM;
    if (reinterpret_cast<uintptr_t>(rows) & 15) return LEC_E_ALIGN;
    return 0;
}
}  // namespace lec

using namespace lec;

extern "C" {

int lec_abi_version(void) { return LEC_ABI_VERSION; }

int64_t lec_launch_count(void) { return (int64_t)g_launches.load(); }

int lec_set_pdl(int on) {
    const int prev = t_pdl;
    t_pdl = on ? 1 : 0;
    return prev;
}

int lec_index_errors(int64_t* count_out, int reset, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* dev = index_errors_ptr();
    if (!dev) return (int)cudaGetLastError();
    unsigned host = 0;
    cudaError_t e = cudaMemcpyAsync(&host, dev, sizeof(host), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && reset) e = cudaMemsetAsync(dev, 0, sizeof(unsigned), st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (count_out) *count_out = (int64_t)host;
    return (int)e;
}

const char* lec_error_string(int code) {
    switch (code) {
        case 0: return "ok";
        case LEC_E_NULL: return "required pointer is NULL";
        case LEC_E_DIM: return "bad dimension: need 1 <= D <= 1024, ld >= D, ld % 4 == 0";
        case LEC_E_ENUM: return "unknown geometry / mode / precision / idx_bytes";
        case LEC_E_SIZE: return "negative element count";
        case LEC_E_ALIGN: return "rows / grad_rows must be 16-byte aligned";
        case LEC_E_K: return "top-k: need 1 <= k <= 8 and 1 <= n_levels <= 8";
        case LEC_E_REPLICAS: return "grad_replicas must be >= 1";
        case LEC_E_EMPTY: return "negative sampler: a draw has no candidate (the reference's random.choice raises IndexError)";
        case LEC_E_INDEX: return "node index outside [0, n_nodes)";
        case LEC_E_PEERS: return "peer exchange: need 2 <= world <= 16, 0 <= rank < world, slot in {0,1}, slot_packets >= n*ld/2+1, non-NULL peer buffers";
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "unknown lec error";
}

int lec_rows_fwd(const float* in, int64_t n, int D, int mode, int geom, float K, float* rows_out, int ld,
                 double* aux_out, float* zero_out, int zero_replicas, int64_t zero_stride, double* zero_scalar, void* stream) {
    if (zero_out && zero_replicas < 1) return LEC_E_REPLICAS;
    if (zero_stride < 0 || (zero_stride & 3) || (zero_stride > 0 && zero_stride < n * (int64_t)ld)) return LEC_E_SIZE;
    if (aux_out && (geom < LEC_GEOM_EUC || geom > LEC_GEOM_OE)) return LEC_E_ENUM;
    if (aux_out && (reinterpret_cast<uintptr_t>(aux_out) & 15)) return LEC_E_ALIGN;
    if (!in || !rows_out) return LEC_E_NULL;
    if (n < 0) return LEC_E_SIZE;
    if (mode < LEC_ROWS_NONE || mode > LEC_ROWS_HYP_TANH_FEAT) return LEC_E_ENUM;
    if (int e = check_rows(rows_out, D, ld)) return e;
    return rows_fwd_launch(in, n, D, mode, geom, K, rows_out, ld, aux_out, zero_out, zero_replicas, zero_stride, zero_scalar,
                           (cudaStream_t)stream);
}

int lec_rows_bwd(const float* in, const float* grad_rows, int grad_replicas, int64_t grad_stride, int64_t n, int D, int ld,
                 int mode, float K, float* grad_in, int accumulate, void* stream) {
    if (grad_replicas < 1) return LEC_E_REPLICAS;
    if (grad_stride < 0 || (grad_stride & 3) || (grad_stride > 0 && grad_stride < n * (int64_t)ld)) return LEC_E_SIZE;
    if (!in || !grad_rows || !grad_in) return LEC_E_NULL;
    if (n < 0) return LEC_E_SIZE;
    if (mode < LEC_ROWS_NONE || mode > LEC_ROWS_HYP_TANH_FEAT) return LEC_E_ENUM;
    if (int e = check_rows(grad_rows, D, ld)) return e;
    return rows_bwd_launch(in, grad_rows, grad_replicas, grad_stride, n, D, ld, mode, K, grad_in, accumulate, (cudaStream_t)stream);
}

int lec_reduce_replicas(const float* in, int replicas, int64_t count, float* out, void* stream) {
    if (!in || !out) return LEC_E_NULL;
    if (count < 0) return LEC_E_SIZE;
    if (replicas < 1) return LEC_E_REPLICAS;
    return reduce_replicas_launch(in, replicas, count, out, (cudaStream_t)stream);
}

int lec_pairs_flat(int geom, int precision, const float* rows, const double* aux, int64_t n_rows, int D, int ld, const void* from_idx,
                   const void* to_idx, int idx_bytes, const float* w, const uint8_t* is_pos, int64_t P, float K,
                   float alpha, float* E_out, double* loss_out, float* grad_rows, int grad_replicas, void* stream) {
    const int core = pick_core(geom, precision);
    if (core < 0 || (idx_bytes != 2 && idx_bytes != 4 && idx_bytes != 8)) return LEC_E_ENUM;
    if (P < 0 || n_rows < 0) return LEC_E_SIZE;
    if (int e = check_rows(rows, D, ld)) return e;
    if (grad_rows && (reinterpret_cast<uintptr_t>(grad_rows) & 15)) return LEC_E_ALIGN;
    if (grad_rows && grad_replicas < 1) return LEC_E_REPLICAS;
    if (P == 0) return 0;
    if (!from_idx || !to_idx || !E_out) return LEC_E_NULL;
    if (geom != LEC_GEOM_OE && !aux) return LEC_E_NULL;
    if (aux && (reinterpret_cast<uintptr_t>(aux) & 15)) return LEC_E_ALIGN;
    FlatArgs a{rows, aux, ld, from_idx, to_idx, idx_bytes, w, is_pos, P, K, alpha, E_out, loss_out, grad_rows,
               grad_replicas, n_rows * (int64_t)ld, n_rows, index_errors_ptr()};
    cudaStream_t st = (cudaStream_t)stream;
    switch (core) {
        case CORE_EUC32: return launch_flat_euc32(a, st);
        case CORE_HYP32: return launch_flat_hyp32(a, st);
        case CORE_HYP64: return launch_flat_hyp64(a, st);
        default: return launch_flat_oe32(a, st);
    }
}

// lec_pairs_poincare and lec_pairs_lorentz: the same checks, the same kernel with the distance as a policy
static int pairs_softmax(int geom, int precision, const float* rows, int64_t n_rows, int D, int ld, const void* pos_from,
                         const void* pos_to, const void* neg_to, int idx_bytes, int64_t B, int N, float* E_pos, float* E_neg,
                         double* loss_out, float* grad_rows, int grad_replicas, void* stream) {
    if (precision != LEC_PREC_F64CORE || (idx_bytes != 2 && idx_bytes != 4 && idx_bytes != 8)) return LEC_E_ENUM;
    if (B < 0 || N < 0 || n_rows < 0) return LEC_E_SIZE;
    if (int e = check_rows(rows, D, ld)) return e;
    if (grad_rows && (reinterpret_cast<uintptr_t>(grad_rows) & 15)) return LEC_E_ALIGN;
    if (grad_rows && grad_replicas < 1) return LEC_E_REPLICAS;
    if (B == 0) return 0;
    if (!pos_from || !pos_to || !E_pos) return LEC_E_NULL;
    if (N > 0 && (!neg_to || !E_neg)) return LEC_E_NULL;
    SoftmaxArgs a{rows, ld, pos_from, pos_to, neg_to, idx_bytes, B, N, E_pos, E_neg, loss_out, grad_rows, grad_replicas,
                  n_rows * (int64_t)ld, n_rows, index_errors_ptr(), (D - (ld / 4 - 1) * 4) <= 2 ? 1 : 0};
    return geom == LEC_GEOM_LORENTZ ? launch_pairs_lorentz(a, (cudaStream_t)stream)
                                    : launch_pairs_poincare(a, (cudaStream_t)stream);
}

int lec_pairs_poincare(int precision, const float* rows, int64_t n_rows, int D, int ld, const void* pos_from, const void* pos_to,
                       const void* neg_to, int idx_bytes, int64_t B, int N, float* E_pos, float* E_neg, double* loss_out,
                       float* grad_rows, int grad_replicas, void* stream) {
    return pairs_softmax(LEC_GEOM_POINCARE, precision, rows, n_rows, D, ld, pos_from, pos_to, neg_to, idx_bytes, B, N, E_pos,
                         E_neg, loss_out, grad_rows, grad_replicas, stream);
}

int lec_pairs_lorentz(int precision, const float* rows, int64_t n_rows, int D, int ld, const void* pos_from, const void* pos_to,
                      const void* neg_to, int idx_bytes, int64_t B, int N, float* E_pos, float* E_neg, double* loss_out,
                      float* grad_rows, int grad_replicas, void* stream) {
    return pairs_softmax(LEC_GEOM_LORENTZ, precision, rows, n_rows, D, ld, pos_from, pos_to, neg_to, idx_bytes, B, N, E_pos,
                         E_neg, loss_out, grad_rows, grad_replicas, stream);
}

int lec_pairs_grouped(int geom, int precision, const float* rows, const double* aux, int64_t n_rows, int D, int ld, const void* pos_from,
                      const void* pos_to, const void* neg_to, const void* neg_from, int idx_bytes, int64_t B, int N,
                      const float* w_pos, const float* w_neg, float K, float alpha, float* E_pos, float* E_neg,
                      double* loss_out, float* grad_rows, int grad_replicas, void* stream) {
    const int core = pick_core(geom, precision);
    if (core < 0 || (idx_bytes != 2 && idx_bytes != 4 && idx_bytes != 8)) return LEC_E_ENUM;
    if (B < 0 || N < 0 || n_rows < 0) return LEC_E_SIZE;
    if (int e = check_rows(rows, D, ld)) return e;
    if (grad_rows && (reinterpret_cast<uintptr_t>(grad_rows) & 15)) return LEC_E_ALIGN;
    if (grad_rows && grad_replicas < 1) return LEC_E_REPLICAS;
    if (B == 0) return 0;
    if (!pos_from || !pos_to || !E_pos) return LEC_E_NULL;
    if (N > 0 && (!neg_to || !neg_from || !E_neg)) return LEC_E_NULL;
    if (geom != LEC_GEOM_OE && !aux) return LEC_E_NULL;
    if (aux && (reinterpret_cast<uintptr_t>(aux) & 15)) return LEC_E_ALIGN;
    GroupArgs a{rows, aux, ld, pos_from, pos_to, neg_to, neg_from, idx_bytes, B, N, w_pos, w_neg, K, alpha,
                E_pos, E_neg, loss_out, grad_rows, grad_replicas, n_rows * (int64_t)ld, n_rows, index_errors_ptr(), 0};
    a.narrow_tail = (D - (ld / 4 - 1) * 4) <= 2 ? 1 : 0;
    cudaStream_t st = (cudaStream_t)stream;
    switch (core) {
        case CORE_EUC32: return launch_grouped_euc32(a, st);
        case CORE_HYP32: return launch_grouped_hyp32(a, st);
        case CORE_HYP64: return launch_grouped_hyp64(a, st);
        default: return launch_grouped_oe32(a, st);
    }
}

static int dense_common(int geom, int precision, const DenseArgs& a, bool bwd, void* stream) {
    const int core = pick_core(geom, precision);
    if (core < 0) return LEC_E_ENUM;
    if (a.P < 0) return LEC_E_SIZE;
    if (a.D < 1 || a.D > LEC_MAX_DIM) return LEC_E_DIM;
    if (a.P == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    switch (core) {
        case CORE_EUC32: return launch_dense_euc32(a, bwd, st);
        case CORE_HYP32: return launch_dense_hyp32(a, bwd, st);
        case CORE_HYP64: return launch_dense_hyp64(a, bwd, st);
        default: return launch_dense_oe32(a, bwd, st);
    }
}

int lec_energy_dense(int geom, int precision, const float* x, const float* y, int64_t P, int D, float K, float* E_out,
                     void* stream) {
    if (P > 0 && (!x || !y || !E_out)) return LEC_E_NULL;
    DenseArgs a{x, y, nullptr, P, D, K, E_out, nullptr, nullptr};
    return dense_common(geom, precision, a, false, stream);
}

int lec_energy_dense_bwd(int geom, int precision, const float* x, const float* y, const float* gE, int64_t P, int D,
                         float K, float* gx, float* gy, void* stream) {
    if (P > 0 && (!x || !y || !gE || !gx || !gy)) return LEC_E_NULL;
    DenseArgs a{x, y, gE, P, D, K, nullptr, gx, gy};
    return dense_common(geom, precision, a, true, stream);
}

int lec_rsgd_update(float* table, const float* grad, int grad_replicas, int64_t n, int D, int ld_g, float lr, float r_in,
                    int lambda_mode, float* grad_out, void* stream) {
    if (!table || !grad) return LEC_E_NULL;
    if (grad_replicas < 1) return LEC_E_REPLICAS;
    if (n < 0) return LEC_E_SIZE;
    if (D < 1 || D > LEC_MAX_DIM || ld_g < D) return LEC_E_DIM;
    if (lambda_mode != 0 && lambda_mode != 1) return LEC_E_ENUM;
    return rsgd_launch(table, grad, grad_replicas, n, D, ld_g, lr, r_in, lambda_mode, grad_out, (cudaStream_t)stream);
}

static int check_update(const lec_update_t* u) {
    if (!u) return LEC_E_NULL;
    if (u->rule < LEC_UPD_NONE || u->rule > LEC_UPD_RSGD_LORENTZ) return LEC_E_ENUM;
    if (u->row_mode < LEC_ROWS_NONE || u->row_mode > LEC_ROWS_HYP_TANH) return LEC_E_ENUM;   // table modes only
    if (u->rule == LEC_UPD_RSGD_RETRACT && u->row_mode != LEC_ROWS_NONE) return LEC_E_ENUM;
    if (u->rule == LEC_UPD_RSGD_LORENTZ && (u->geom != LEC_GEOM_LORENTZ || u->row_mode != LEC_ROWS_NONE || u->aux_out))
        return LEC_E_ENUM;
    if (u->lambda_mode != 0 && u->lambda_mode != 1) return LEC_E_ENUM;
    if (u->aux_out && (u->geom < LEC_GEOM_EUC || u->geom > LEC_GEOM_OE)) return LEC_E_ENUM;
    if (!u->table || !u->grad_rows) return LEC_E_NULL;
    if (u->grad_replicas < 1) return LEC_E_REPLICAS;
    if (u->n < 0) return LEC_E_SIZE;
    if (u->grad_stride < 0 || (u->grad_stride & 3) || (u->grad_stride > 0 && u->grad_stride < u->n * (int64_t)u->ld)) return LEC_E_SIZE;
    if (u->D < 1 || u->D > LEC_MAX_DIM || u->ld < u->D || (u->ld & 3)) return LEC_E_DIM;
    if (reinterpret_cast<uintptr_t>(u->grad_rows) & 15) return LEC_E_ALIGN;
    if (u->rows_out && (reinterpret_cast<uintptr_t>(u->rows_out) & 15)) return LEC_E_ALIGN;
    if (u->aux_out && (reinterpret_cast<uintptr_t>(u->aux_out) & 15)) return LEC_E_ALIGN;
    if (u->rule == LEC_UPD_ADAM && (!u->state_m || !u->state_v)) return LEC_E_NULL;
    if (u->rule == LEC_UPD_SGD && u->momentum != 0.f && !u->state_m) return LEC_E_NULL;
    if ((u->state_m && (reinterpret_cast<uintptr_t>(u->state_m) & 15)) || (u->state_v && (reinterpret_cast<uintptr_t>(u->state_v) & 15)))
        return LEC_E_ALIGN;
    return 0;
}

static int check_exchange(const lec_exchange_t* x, int64_t n, int ld) {
    if (!x || x->world <= 1) return 0;
    if (!x->peer_bufs) return LEC_E_NULL;
    if (x->world > LEC_MAX_PEERS || x->rank < 0 || x->rank >= x->world || (x->slot != 0 && x->slot != 1) || x->tag == 0)
        return LEC_E_PEERS;
    if (x->mode != LEC_XCHG_ONE_SHOT && x->mode != LEC_XCHG_TWO_SHOT) return LEC_E_ENUM;
    if (x->mode == LEC_XCHG_ONE_SHOT && x->slot_packets < lec_exchange_packets(n, ld)) return LEC_E_PEERS;
    for (int p = 0; p < x->world; ++p) {
        if (!x->peer_bufs[p]) return LEC_E_NULL;
        if (reinterpret_cast<uintptr_t>(x->peer_bufs[p]) & 15) return LEC_E_ALIGN;
    }
    return 0;
}

int64_t lec_exchange_packets(int64_t n, int ld) { return (n < 0 || ld < 0) ? 0 : n * (int64_t)ld / 2 + 1; }

int64_t lec_exchange_bytes(int64_t n, int ld, int world, int mode) {
    if (n < 0 || ld < 4 || (ld & 3) || world < 1 || world > LEC_MAX_PEERS) return 0;
    if (mode == LEC_XCHG_TWO_SHOT) return two_shot_bytes(n, ld, world);
    return 2 * (int64_t)world * lec_exchange_packets(n, ld) * 16;
}

int lec_update_rows(const lec_update_t* u, const lec_exchange_t* x, void* stream) {
    if (int e = check_update(u)) return e;
    if (int e = check_exchange(x, u->n, u->ld)) return e;
    return update_rows_launch(*u, x, (cudaStream_t)stream);
}

int lec_cone_step(const lec_step_t* s, void* stream) {
    if (!s) return LEC_E_NULL;
    const lec_update_t& u = s->upd;
    if (int e = check_update(&u)) return e;
    if (int e = check_exchange(&s->xchg, u.n, u.ld)) return e;
    if (!u.rows_out || !u.loss_acc) return LEC_E_NULL;
    // Nickel & Kiela's embeddings (Poincare ball or Lorentz model): the softmax pair kernel on untransformed rows
    const bool poincare = s->geom == LEC_GEOM_POINCARE || s->geom == LEC_GEOM_LORENTZ;
    if (poincare && (s->precision != LEC_PREC_F64CORE || u.row_mode != LEC_ROWS_NONE || s->w_pos || s->w_neg))
        return LEC_E_ENUM;
    struct PdlScope {   // the kernels of this step are launched as programmatic dependents of one another
        int prev;
        PdlScope() : prev(t_pdl) { t_pdl = 1; }
        ~PdlScope() { t_pdl = prev; }
    } pdl_scope;
    cudaStream_t st = (cudaStream_t)stream;
    if (!s->fused) {
        const int e = lec_rows_fwd(u.table, u.n, u.D, u.row_mode, s->geom, u.K, u.rows_out, u.ld, u.aux_out, u.grad_rows,
                                   u.grad_replicas, u.grad_stride, u.loss_acc, stream);
        if (e) return e;
    }
    if (s->ev_pairs_start) cudaEventRecord((cudaEvent_t)s->ev_pairs_start, st);
    const int e = poincare
        ? pairs_softmax(s->geom, s->precision, u.rows_out, u.n, u.D, u.ld, s->pos_from, s->pos_to, s->neg_to, s->idx_bytes,
                        s->B, s->N, s->E_pos, s->E_neg, u.loss_acc, u.grad_rows, u.grad_replicas, stream)
        : lec_pairs_grouped(s->geom, s->precision, u.rows_out, u.aux_out, u.n, u.D, u.ld, s->pos_from, s->pos_to,
                            s->neg_to, s->neg_from, s->idx_bytes, s->B, s->N, s->w_pos, s->w_neg, u.K, s->alpha,
                            s->E_pos, s->E_neg, u.loss_acc, u.grad_rows, u.grad_replicas, stream);
    if (s->ev_pairs_stop) cudaEventRecord((cudaEvent_t)s->ev_pairs_stop, st);
    if (e) return e;
    return update_rows_launch(u, &s->xchg, st);
}

int lec_featnet_supported(int F, int D) { return featnet_supported(F, D) ? 1 : 0; }

static int check_featnet(const float* features, int64_t n_pool, int F, const void* sel, int sel_bytes, int64_t m, int D) {
    if (m < 0 || n_pool < 0) return LEC_E_SIZE;
    if (!featnet_supported(F, D)) return LEC_E_DIM;
    if (sel && sel_bytes != 4 && sel_bytes != 8) return LEC_E_ENUM;
    if (m > 0 && !features) return LEC_E_NULL;
    if (reinterpret_cast<uintptr_t>(features) & 15) return LEC_E_ALIGN;
    if (!sel && m > n_pool) return LEC_E_SIZE;
    return 0;
}

int lec_featnet_fwd(const float* features, int64_t n_pool, int F, const void* sel, int sel_bytes, int64_t m,
                    const float* weight, const float* bias, int D, float* Y, void* stream) {
    if (int e = check_featnet(features, n_pool, F, sel, sel_bytes, m, D)) return e;
    if (m > 0 && (!weight || !Y)) return LEC_E_NULL;
    if (reinterpret_cast<uintptr_t>(weight) & 15) return LEC_E_ALIGN;
    FeatArgs a{features, n_pool, F, sel, sel_bytes, m, weight, bias, D, Y, nullptr, nullptr, 1, 0, index_errors_ptr()};
    return featnet_fwd_launch(a, (cudaStream_t)stream);
}

int lec_featnet_wgrad(const float* features, int64_t n_pool, int F, const void* sel, int sel_bytes, int64_t m,
                      const float* gY, int D, float* grad_flat, int grad_replicas, int64_t grad_stride, void* stream) {
    if (int e = check_featnet(features, n_pool, F, sel, sel_bytes, m, D)) return e;
    if (grad_replicas < 1) return LEC_E_REPLICAS;
    if (m > 0 && (!gY || !grad_flat)) return LEC_E_NULL;
    if ((reinterpret_cast<uintptr_t>(grad_flat) & 15) || (grad_stride & 3)) return LEC_E_ALIGN;
    if (grad_replicas > 1 && grad_stride < (int64_t)D * F + D) return LEC_E_SIZE;
    FeatArgs a{features, n_pool, F, sel, sel_bytes, m, nullptr, nullptr, D, nullptr, gY, grad_flat, grad_replicas, grad_stride,
               index_errors_ptr()};
    return featnet_wgrad_launch(a, (cudaStream_t)stream);
}

int lec_score_topk_ex(int geom, int precision, const float* labels, int64_t L, const float* images, int64_t N, int D,
                      float K, const int32_t* level_start, const int32_t* level_stop, int n_levels, int k, float* scores,
                      int scores_layout, int32_t* topk_idx, float* topk_val, void* stream) {
    // the Poincare and Lorentz distances have the fp32 SIMT kernel only (D <= 64)
    const bool poincare = geom == LEC_GEOM_POINCARE || geom == LEC_GEOM_LORENTZ;
    if (poincare ? precision != LEC_PREC_F32 : pick_core(geom, precision) < 0) return LEC_E_ENUM;
    if (poincare && (D < 1 || D > 64)) return LEC_E_DIM;
    if (scores_layout != LEC_SCORES_IMAGE_MAJOR && scores_layout != LEC_SCORES_LABEL_MAJOR) return LEC_E_ENUM;
    if (L < 0 || N < 0) return LEC_E_SIZE;
    if (D < 1 || D > 128) return LEC_E_DIM;
    if (n_levels < 0 || n_levels > LEC_MAX_LEVELS) return LEC_E_K;
    if (topk_idx && (k < 1 || k > LEC_MAX_TOPK || n_levels < 1)) return LEC_E_K;
    if (!topk_idx) { n_levels = 0; k = 1; }
    if (n_levels > 0 && (!level_start || !level_stop)) return LEC_E_NULL;
    if (N > 0 && L > 0 && (!labels || !images)) return LEC_E_NULL;
    const int64_t s_img = scores_layout == LEC_SCORES_IMAGE_MAJOR ? L : 1;
    const int64_t s_lab = scores_layout == LEC_SCORES_IMAGE_MAJOR ? 1 : N;
    return score_launch(geom, precision, labels, L, images, N, D, K, level_start, level_stop, n_levels, k, scores,
                        s_img, s_lab, topk_idx, topk_val, (cudaStream_t)stream);
}

int lec_score_tc_supported(int geom, int precision, int D, int64_t L, int n_levels) {
    return (n_levels >= 0 && n_levels <= LEC_MAX_LEVELS && L >= 0 && score_mma_supported(geom, precision, D, L, n_levels)) ? 1 : 0;
}

int64_t lec_score_workspace_bytes(int64_t L, int D, int n_levels) {
    if (L < 0 || D < 1 || n_levels < 0) return 0;
    return score_mma_workspace_bytes(L, D, n_levels);
}

int lec_score_topk_tc(int geom, int precision, const float* labels, int64_t L, const float* images, int64_t N, int D,
                      float K, const int32_t* level_start, const int32_t* level_stop, int n_levels, int k, float* scores,
                      int32_t* topk_idx, float* topk_val, void* workspace, int64_t workspace_bytes, void* stream) {
    if (pick_core(geom, precision) < 0) return LEC_E_ENUM;
    if (L < 0 || N < 0) return LEC_E_SIZE;
    if (D < 1 || D > 128) return LEC_E_DIM;
    if (n_levels < 0 || n_levels > LEC_MAX_LEVELS) return LEC_E_K;
    if (topk_idx && (k < 1 || k > LEC_MAX_TOPK || n_levels < 1)) return LEC_E_K;
    if (!topk_idx) { n_levels = 0; k = 1; }
    if (!score_mma_supported(geom, precision, D, L, n_levels)) return LEC_E_ENUM;
    if (n_levels > 0 && (!level_start || !level_stop)) return LEC_E_NULL;
    if (N > 0 && L > 0 && (!labels || !images || !workspace)) return LEC_E_NULL;
    return score_mma_launch(labels, L, images, N, D, K, level_start, level_stop, n_levels, k, scores, topk_idx, topk_val,
                            workspace, workspace_bytes, (cudaStream_t)stream);
}

int lec_score_topk(int geom, int precision, const float* labels, int64_t L, const float* images, int64_t N, int D,
                   float K, const int32_t* level_start, const int32_t* level_stop, int n_levels, int k, float* scores,
                   int32_t* topk_idx, float* topk_val, void* stream) {
    return lec_score_topk_ex(geom, precision, labels, L, images, N, D, K, level_start, level_stop, n_levels, k, scores,
                             LEC_SCORES_IMAGE_MAJOR, topk_idx, topk_val, stream);
}

}  // extern "C"

#ifdef LEC_STEP_TRACE
// debug builds only (not part of the ABI): out7 <- the step trace, which is then reset; synchronises the device
extern "C" int lec_debug_step_trace(unsigned long long* out7) {
    const unsigned long long init[7] = {~0ull, 0, ~0ull, 0, 0, 0, 0};
    if (!lec::g_step_trace) {
        if (cudaMalloc(&lec::g_step_trace, sizeof(init)) != cudaSuccess) return -1;
    } else {
        cudaDeviceSynchronize();
        if (out7) cudaMemcpy(out7, lec::g_step_trace, sizeof(init), cudaMemcpyDeviceToHost);
    }
    cudaMemcpy(lec::g_step_trace, init, sizeof(init), cudaMemcpyHostToDevice);
    return 0;
}
#endif
