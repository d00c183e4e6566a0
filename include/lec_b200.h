/*
 * lec_b200.h -- C ABI of the B200 (sm_100a) entailment-cone kernels.
 *
 * The reference (ankitdhall/learning_embeddings) is pure Python/PyTorch and has no FFI of its own
 * (SURVEY.md 8b); its "operator interface" for this path is the Python class protocol of
 * network/order_embeddings*.py and network/oe*.py.  Each entry point below names the reference
 * code it replaces.  The Python host (learning_embeddings_b200/) binds these with ctypes; a
 * maintainer of the reference would bind them the same way (INTEGRATION.md).
 *
 * Conventions
 *   - plain C, raw DEVICE pointers, explicit sizes, explicit stream (a cudaStream_t passed as void*)
 *   - returns 0 on success, a positive cudaError_t, or a negative LEC_E_* argument error
 *   - never allocates, frees or synchronises; all buffers are owned by the caller.  Exceptions, each documented at its
 *     declaration: lec_index_errors reads a counter back (synchronises the stream); lec_host_pipe_create / _destroy own
 *     a small host object (one stream, 3 events per slot) and lec_host_pipe_wait blocks on an event by design
 *   - all floating point is IEEE fp32 storage; `precision` selects the arithmetic of the per-pair
 *     scalar core: LEC_PREC_F32 (fp32 throughout) or LEC_PREC_F64CORE (dot products and the
 *     angle/aperture algebra in fp64, vectors and outputs fp32)
 *   - "rows" is the TRANSFORMED embedding table the energies are evaluated on: [n_rows, ld] fp32,
 *     ld a multiple of 4 (>= D), pad columns zero, base 16-byte aligned.  It is produced from the
 *     raw parameter table by lec_rows_fwd (together with the per-row "aux" terms) and its gradient is
 *     mapped back by lec_rows_bwd.
 *   - index arrays are uint16, int32 or int64 (idx_bytes = 2, 4 or 8; uint16 needs n_rows <= 65536 and
 *     halves the host->device bytes of a step's index block)
 */
#ifndef LEC_B200_H
#define LEC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LEC_ABI_VERSION 14

/* geometry of the energy */
#define LEC_GEOM_EUC 0 /* EucConesLoss.E_operator, order_embeddings.py:954-969 = oe.py:721-739 (cos-space) */
#define LEC_GEOM_HYP 1 /* hyperbolic EucConesLoss.E_operator, order_embeddings_h.py:1097-1120 = oe_h.py:811-833 */
#define LEC_GEOM_OE  2 /* OrderEmbeddingLoss.E_operator, order_embeddings.py:818-824 */

/* per-row transform applied to the raw parameter rows (Embedder.forward / FeatNet tail) */
#define LEC_ROWS_NONE          0 /* plain nn.Embedding lookup (order embeddings) */
#define LEC_ROWS_EUC_SOFTCLIP  1 /* e/|e|*(|e|+K): order_embeddings.py:195-200, oe.py:75-80, oe.py:133-138 */
#define LEC_ROWS_HYP_SHELL     2 /* +1e-15, project into [r_in, 1-1e-5], straight-through: order_embeddings_h.py:205-228 */
#define LEC_ROWS_HYP_TANH      3 /* tanh(clamp(atanh(r_in)+|e|))*e/|e| then projection: oe_h.py:77-104 */
#define LEC_ROWS_HYP_TANH_FEAT 4 /* same on FeatNet output, (1e-6+x)/(1e-6+|x|) projection: oe_h.py:168-224 */

#define LEC_PREC_F32     0
#define LEC_PREC_F64CORE 1

/* negative return codes */
#define LEC_E_NULL      (-1) /* required pointer is NULL */
#define LEC_E_DIM       (-2) /* D < 1, D > LEC_MAX_DIM, ld < D or ld % 4 != 0 */
#define LEC_E_ENUM      (-3) /* unknown geometry / mode / precision / idx_bytes */
#define LEC_E_SIZE      (-4) /* negative count */
#define LEC_E_ALIGN     (-5) /* rows / grad_rows base not 16-byte aligned */
#define LEC_E_K         (-6) /* k out of range for top-k */
#define LEC_E_REPLICAS  (-7) /* grad_replicas < 1 */
#define LEC_E_PEERS     (-8) /* world/rank/slot out of range or slot_packets too small */
#define LEC_E_EMPTY     (-9) /* a negative draw has no candidate (random.choice([]) -> IndexError in the reference) */
#define LEC_E_INDEX     (-10) /* node index outside [0, n_nodes) */
#define LEC_MAX_DIM 1024
#define LEC_MAX_TOPK 8
#define LEC_MAX_LEVELS 8

int lec_abi_version(void);
const char* lec_error_string(int code);
/* kernels launched by this library since load (the bench's gpu_launches claim) */
int64_t lec_launch_count(void);
/* on != 0: the step kernels (pairs_grouped, update_rows, featnet_*) this THREAD launches from now on are programmatic
 * dependents of their predecessor in the stream (their blocks become resident while it drains and wait in
 * griddepcontrol.wait), which hides the launch gap between the kernels of a step.  lec_cone_step does this for its own
 * launches; a host that issues a step as several calls (the joint trainers' engine) switches it on once.  Returns the
 * previous setting. */
int lec_set_pdl(int on);
/* Endpoint ids are range-checked on the device against n_rows, as nn.Embedding checks them on the host (the reference
 * raises IndexError, order_embeddings.py:188-192): a pair with an id outside [0, n_rows) reads and writes nothing out
 * of bounds, gets energy NaN, contributes neither loss nor gradient, and is counted.  This call returns the count for
 * the current device since the last reset in *count_out (HOST pointer).  The one entry point that synchronises: it
 * waits for `stream`. */
int lec_index_errors(int64_t* count_out, int reset, void* stream);

/* ---- row transforms ----------------------------------------------------------------------------
 * Replaces Embedder.forward (order_embeddings.py:188-200, order_embeddings_h.py:205-228,
 * oe_h.py:77-104) and the FeatNet tail after fc1 (oe.py:127-138, oe_h.py:168-224), applied once per
 * table row instead of once per gathered pair endpoint.
 *   in        [n, D] raw rows (row stride D)
 *   rows_out  [n, ld] transformed rows, pad columns written as 0
 *   aux_out   optional [n, 4] doubles (16-byte aligned): the per-row terms of energy `geom` that depend on
 *             one endpoint only -- { |x|^2, 1/|x|, half-aperture term, its dz/dx coefficient } -- computed
 *             in fp64 once per row so that the pair kernels never recompute them per pair.  Required by
 *             lec_pairs_flat / lec_pairs_grouped for LEC_GEOM_EUC and LEC_GEOM_HYP.
 *   zero_out  optional [zero_replicas, n, ld] buffer cleared in the same pass (the gradient
 *             accumulator of the pair kernels), may be NULL
 *   zero_scalar optional double[1] cleared in the same pass (the loss accumulator), may be NULL
 *   zero_stride floats between two replicas of zero_out; 0 = n * ld (a gradient accumulator of exactly these rows).
 *             A row range inside a larger accumulator (the image rows behind the label rows, joint trainers) passes
 *             the accumulator's own replica stride.
 */
int lec_rows_fwd(const float* in, int64_t n, int D, int mode, int geom, float K, float* rows_out, int ld,
                 double* aux_out, float* zero_out, int zero_replicas, int64_t zero_stride, double* zero_scalar,
                 void* stream);

/* Vector-Jacobian product of lec_rows_fwd: grad_in[n, D] (=|+=) J^T grad_rows[n, ld].
 * grad_rows is [grad_replicas, n, ld] (grad_stride floats between replicas, 0 = n * ld); the replicas are summed on
 * the fly.  Replaces autograd through Embedder.forward incl. embedding_dense_backward.  accumulate != 0 adds. */
int lec_rows_bwd(const float* in, const float* grad_rows, int grad_replicas, int64_t grad_stride, int64_t n, int D, int ld,
                 int mode, float K, float* grad_in, int accumulate, void* stream);

/* out[count] = sum over r of in[r, count] (the replica sum on its own, e.g. before an all-reduce). */
int lec_reduce_replicas(const float* in, int replicas, int64_t count, float* out, void* stream);

/* ---- pair energies on gathered rows ------------------------------------------------------------
 * Flat pair list.  Replaces E_operator + positive_pair/negative_pair + the loss sum of
 * EucConesLoss.forward / OrderEmbeddingLoss.forward (order_embeddings.py:971-975, :1029-1042 eval
 * branch, :1056-1102 train branch) for an arbitrary list of (from, to) endpoints.
 *   rows, aux        transformed table and its per-row terms from lec_rows_fwd (aux may be NULL for OE)
 *   from_idx,to_idx  [P] row numbers into rows
 *   w                optional [P] pair weights (NULL = 1)
 *   is_pos           optional [P] uint8, 1 = positive term w*E, 0 = negative term w*max(0, alpha-E)
 *                    (NULL = all positive)
 *   E_out            [P] raw energies
 *   loss_out         optional double[1], the weighted hinge sum is ADDED to it
 *   grad_rows        optional [grad_replicas, n_rows, ld]; if non-NULL d loss / d rows is atomically
 *                    ADDED to it.  The scatter is an L2 vector reduction (REDG.F32x4) whose throughput is
 *                    limited by same-address serialisation on hot rows, so the kernel spreads its
 *                    thread blocks over grad_replicas private copies (block b adds to copy b %
 *                    grad_replicas); the true gradient is their sum (lec_rows_bwd, lec_rsgd_update and
 *                    lec_reduce_replicas sum them).  grad_replicas >= 1.
 */
int lec_pairs_flat(int geom, int precision, const float* rows, const double* aux, int64_t n_rows, int D, int ld,
                   const void* from_idx, const void* to_idx, int idx_bytes, const float* w,
                   const uint8_t* is_pos, int64_t P, float K, float alpha, float* E_out,
                   double* loss_out, float* grad_rows, int grad_replicas, void* stream);

/* Training-layout batch: B positives (u_i, v_i), each with N negatives (u_i, v'_ip) and N negatives
 * (u'_ip, v_i) -- the layout EucConesLoss.forward builds at order_embeddings.py:1063-1091 (SURVEY F6),
 * kept in compact form (only the corrupted endpoint is stored).
 *   pos_from,pos_to   [B]
 *   neg_to            [B, N]  corrupted children v' of u_i   (reference slots 2N*i + p)
 *   neg_from          [B, N]  corrupted parents  u' of v_i   (reference slots 2N*i + N + p)
 *   w_pos [B], w_neg [B, 2N]  optional weights (NULL = 1)
 *   E_pos [B], E_neg [B, 2N]  raw energies in the reference's order
 *   loss_out, grad_rows       as above (grad_rows required unless NULL = forward only)
 */
int lec_pairs_grouped(int geom, int precision, const float* rows, const double* aux, int64_t n_rows, int D,
                      int ld, const void* pos_from, const void* pos_to, const void* neg_to, const void* neg_from,
                      int idx_bytes, int64_t B, int N, const float* w_pos, const float* w_neg, float K,
                      float alpha, float* E_pos, float* E_neg, double* loss_out, float* grad_rows,
                      int grad_replicas, void* stream);

/* Dense operands (no gather): E_operator(x, y) on arbitrary [P, D] tensors, as the reference calls
 * it from check_graph_embedding (order_embeddings.py:550-551) and the scoring loops. */
int lec_energy_dense(int geom, int precision, const float* x, const float* y, int64_t P, int D, float K,
                     float* E_out, void* stream);
/* gx, gy [P, D] = gE[p] * dE/dx, dE/dy (E already includes its own max(0, .)). */
int lec_energy_dense_bwd(int geom, int precision, const float* x, const float* y, const float* gE,
                         int64_t P, int D, float K, float* gx, float* gy, void* stream);

/* ---- Riemannian SGD on the Poincare ball --------------------------------------------------------
 * Replaces order_embeddings_h.py:769-775 (lambda_x :662, exp_map_x :668, mob_add :649, soft_clip :634;
 * joint copy oe_h.py:1604-1644, :1761-1762).  Whole table, in place.
 *   grad [grad_replicas, n, ld_g] Euclidean gradient, replicas summed on the fly (ld_g = D and
 *        grad_replicas = 1 for a dense nn.Embedding grad)
 *   lambda_mode 0: reference conformal factor 2/(1-|x|) (SURVEY F4); 1: textbook 2/(1-|x|^2)
 *   grad_out optional [n, D]: receives the rescaled (Riemannian) gradient as the reference leaves it
 *   in weight.grad; may alias grad when ld_g == D and grad_replicas == 1.
 */
int lec_rsgd_update(float* table, const float* grad, int grad_replicas, int64_t n, int D, int ld_g, float lr,
                    float r_in, int lambda_mode, float* grad_out, void* stream);

/* ---- fused table update (+ data-parallel exchange over NVLink / NVSwitch peer memory) ---------------
 * Everything a training iteration does to the parameter table between the pair kernel and the next iteration's
 * pair kernel, in ONE launch, per table row:
 *   1. sum of the row's gradient replicas (d loss / d rows from lec_pairs_*), replicas cleared
 *   2. world > 1: one-shot all-reduce of the row over peer memory (lec_exchange_t below)
 *   3. vector-Jacobian product of the row transform `row_mode` (autograd through Embedder.forward)
 *   4. the update rule:
 *        LEC_UPD_RSGD  order_embeddings_h.py:764-775 (lambda_x :662, exp_map_x :668, mob_add :649, soft_clip :634;
 *                      joint copy oe_h.py:1604-1644, :1761-1762)
 *        LEC_UPD_SGD   torch.optim.SGD(lr, momentum)   order_embeddings.py:563, oe.py:1712
 *        LEC_UPD_ADAM  torch.optim.Adam(lr)            order_embeddings.py:565, oe.py:1714, oe_h.py:1520-1523
 *        LEC_UPD_NONE  table left alone (grad_out receives d loss / d table)
 *      hyp_rescale != 0 multiplies the gradient by ((1 - |w|) / 2)^2 first (oe_h.py:1766, :1770) and
 *      project_shell != 0 projects the updated row into [r_in, 1 - 1e-5] afterwards (soft_clip, oe_h.py:1771) --
 *      together with LEC_UPD_ADAM that is the reference's default joint hyperbolic update.  RSGD includes both.
 *   5. rows_out != NULL: the row transform of the UPDATED row into rows_out [n, ld] and its aperture terms into
 *      aux_out [n, 4] (as lec_rows_fwd), i.e. the Embedder.forward the NEXT iteration starts with
 * The loss accumulator the pair kernel added into is moved: *loss_step = *loss_acc; *loss_acc = 0 (both optional).
 *   table       [n, D] raw parameter rows, updated in place
 *   grad_rows   [grad_replicas, n, ld], 16-byte aligned (grad_stride floats between replicas when the rows are a range
 *               of a larger accumulator)
 *   state_m/v   [n, ld] optimizer state owned by the caller, zero before the first step: Adam moments (m, v) or the
 *               SGD momentum buffer (m; may be NULL when momentum == 0)
 *   opt_step    1-based step count of the Adam bias correction
 *   grad_out    optional [n, D]: the gradient as the optimizer saw it (what the reference leaves in weight.grad)
 */
#define LEC_UPD_NONE 0
#define LEC_UPD_RSGD 1
#define LEC_UPD_SGD  2
#define LEC_UPD_ADAM 3
typedef struct lec_update {
    int rule, row_mode, geom, lambda_mode /* RSGD: 0 reference 2/(1-|x|) (SURVEY F4), 1 textbook 2/(1-|x|^2) */;
    int hyp_rescale, project_shell;
    float K, lr, r_in;
    float momentum, beta1, beta2, eps; int64_t opt_step;
    float* table; int64_t n; int D; int ld;
    float* grad_rows; int grad_replicas; int64_t grad_stride /* floats between replicas, 0 = n * ld */;
    float* state_m; float* state_v;
    float* rows_out; double* aux_out; float* grad_out;
    double* loss_acc; double* loss_step;
} lec_update_t;

/* The exchange of step 2 replaces nn.DataParallel's reduce_add + broadcast of the label table
 * (order_embeddings.py:360, oe.py:1336,1341): one process per GPU, every rank owns an exchange buffer that all ranks
 * have mapped (CUDA IPC / torch symmetric memory), laid out as
 *     packet slot[2][world][slot_packets]      16-byte packets {value, tag, value, tag}
 * slot_packets >= lec_exchange_packets(n, ld) = n * ld / 2 + 1 (two floats per packet + one packet for the loss).
 * Step t uses slot t % 2 and tag t + 1 (tags increase; buffers start zeroed).  Every rank stores the replica sum of
 * each row into source region [rank] of EVERY rank's buffer (remote stores; the 8-byte halves of a packet are written
 * atomically, so the tag is the arrival flag: no fence, no flag store, one NVLink latency), then polls its OWN buffer
 * until the `world` packets of the chunk carry the tag and adds them in rank order -- the same bits on every rank, so
 * the replicas of the table stay identical.  The rank's loss travels the same way; *loss_global = sum over ranks.
 *   peer_bufs   HOST array of `world` device pointers (rank order)
 *   error       device int, zero at start: set to 1 when a peer's packets do not arrive within timeout_ms (0 = 30 s).
 *               From then on the rows concerned and every later lec_update_rows on this rank leave the table
 *               untouched; the host must treat a non-zero *error as fatal (engine.ConeStep raises).
 *
 * mode LEC_XCHG_TWO_SHOT (tables of megabytes, where sending the whole gradient to every peer would be W-1 table
 * volumes per rank and step): rank r OWNS rows [r * R, (r + 1) * R).  lec_update_rows then issues three launches --
 * scatter (every rank stores the replica sum of each row into its owner's buffer, tile flags follow with release
 * semantics), owner (waits for the `world` partial tiles, adds them in rank order, applies the update rule once per row,
 * stores the updated raw row into every peer's staging area) and receiver (copies the staged rows of the other owners
 * into the local table and runs the row transform) -- a reduce-scatter + all-gather that moves 2 (W-1)/W table volumes
 * per rank; the replicas are identical by construction.  Buffer size: lec_exchange_bytes(n, ld, world, mode);
 * slot_packets is ignored; grad_out is not produced.  `phases` (two-shot only) selects which of the three launches
 * this call issues -- LEC_XCHG_SCATTER | LEC_XCHG_OWNER | LEC_XCHG_RECEIVER, 0 = all -- for a host that wants to put
 * other work between them (or drives several ranks from one stream); a step is complete after all three.
 */
#define LEC_XCHG_SCATTER 1
#define LEC_XCHG_OWNER 2
#define LEC_XCHG_RECEIVER 4
#define LEC_XCHG_ONE_SHOT 0
#define LEC_XCHG_TWO_SHOT 1
typedef struct lec_exchange {
    void* const* peer_bufs; int64_t slot_packets; int world, rank, slot; uint32_t tag;
    double* loss_global; int* error; int64_t timeout_ms;
    int mode, phases;
} lec_exchange_t;
#define LEC_MAX_PEERS 16
int64_t lec_exchange_packets(int64_t n, int ld);
int64_t lec_exchange_bytes(int64_t n, int ld, int world, int mode);
int lec_update_rows(const lec_update_t* u, const lec_exchange_t* x /* NULL or world <= 1: single GPU */, void* stream);

/* ---- one whole training step in one call ---------------------------------------------------------
 * The launch sequence of one label-only cone step (what one iteration of the reference's
 * pass_samples('train') loop does between zero_grad() and the weight update, order_embeddings_h.py:752-775 /
 * order_embeddings.py:619-635) issued from C, so the host pays one FFI call per step instead of one per kernel:
 *     [fused == 0: lec_rows_fwd (clears grad_rows and *loss_acc) ->]  lec_pairs_grouped -> lec_update_rows
 * fused != 0: rows / aux / cleared grad_rows are already current -- a previous step's lec_update_rows (with rows_out)
 * or lec_rows_fwd produced them -- so the step is two launches, each a programmatic dependent of the one before.
 * The pair kernel adds into *upd.loss_acc; the update leaves this rank's loss of the step in *upd.loss_step.
 * Table geometry (n, D, ld, K), rows (upd.rows_out), aux (upd.aux_out) and the gradient replicas are taken from `upd`.
 * ev_pairs_start/stop: optional cudaEvent_t recorded around the pair kernel (for the roofline timing).
 */
typedef struct lec_step {
    int geom, precision, fused;
    float alpha;
    const void* pos_from; const void* pos_to; const void* neg_to; const void* neg_from; int idx_bytes;
    int64_t B; int N;
    const float* w_pos; const float* w_neg;
    float* E_pos; float* E_neg;
    void* ev_pairs_start; void* ev_pairs_stop;
    lec_update_t upd;
    lec_exchange_t xchg;
} lec_step_t;
int lec_cone_step(const lec_step_t* s, void* stream);

/* ---- FeatNet.fc1 on gathered feature rows -----------------------------------------------------------------
 * The image side of the joint trainers: nn.Linear(F, D) over the step's image features (FeatNet.fc1, oe.py:97,113;
 * oe_h.py:127,143), with the gather of those features (get_img_features, oe.py:680-707: a Python dict lookup per
 * filename) fused in.  `features` is the device-resident [n_pool, F] matrix, `sel` [m] row numbers into it (int32 /
 * int64; NULL = rows 0..m-1).  D <= 16, F % 4 == 0, F <= 4096 (lec_featnet_supported; otherwise use cuBLAS).
 *   lec_featnet_fwd    Y[i, :] = weight [D, F] . features[sel[i], :] + bias [D]            Y [m, D]
 *   lec_featnet_wgrad  d weight [d, f] += sum_i gY[i, d] features[sel[i], f],  d bias [d] += sum_i gY[i, d]
 *                      added into one of `grad_replicas` copies (replica stride grad_stride floats) of a flat
 *                      [D*F weights | D biases | pad] buffer: the layout lec_update_rows takes as an [n, 16] "table" of
 *                      plain parameters (row_mode LEC_ROWS_NONE), which sums and clears the replicas.
 * Each is one pass over the m gathered rows (4 F bytes per row); an id outside [0, n_pool) is skipped and counted
 * (lec_index_errors). */
int lec_featnet_supported(int F, int D);
int lec_featnet_fwd(const float* features, int64_t n_pool, int F, const void* sel, int sel_bytes, int64_t m,
                    const float* weight, const float* bias, int D, float* Y, void* stream);
int lec_featnet_wgrad(const float* features, int64_t n_pool, int F, const void* sel, int sel_bytes, int64_t m,
                      const float* gY, int D, float* grad_flat, int grad_replicas, int64_t grad_stride, void* stream);

/* ---- all-pairs image x label scoring ------------------------------------------------------------
 * Replaces the per-image loop of JointEmbeddings.calculate_classification_metrics
 * (oe.py:1764-1779, oe_h.py:2018-2036): e[i, l] = E(x = label_l, y = image_i), then per level
 * torch.topk(k, largest=False).
 *   labels [L, D], images [N, D] (row stride D)
 *   level_start/level_stop  HOST int32[n_levels], label ranges [start, stop)
 *   scores    optional [N, L] full energy matrix
 *   topk_idx  optional int32 [N, n_levels, k] label ids (ascending energy), -1 if fewer than k finite
 *   topk_val  optional float [N, n_levels, k]
 */
int lec_score_topk(int geom, int precision, const float* labels, int64_t L, const float* images,
                   int64_t N, int D, float K, const int32_t* level_start, const int32_t* level_stop,
                   int n_levels, int k, float* scores, int32_t* topk_idx, float* topk_val, void* stream);

/* Same, with the layout of the optional full energy matrix chosen by the caller.  The reference never
 * materialises this matrix (it holds one image's L energies at a time, oe_h.py:2018-2028), so its
 * layout is ours to define:
 *   LEC_SCORES_IMAGE_MAJOR  scores[i * L + l]   (what lec_score_topk writes)
 *   LEC_SCORES_LABEL_MAJOR  scores[l * N + i]   the kernel's threads own images, so this is the layout
 *                           whose stores coalesce (128 B per warp); the host wrapper returns it as the
 *                           transposed view, i.e. still indexed scores[i, l].
 * level ranges must be ascending and disjoint. */
#define LEC_SCORES_IMAGE_MAJOR 0
#define LEC_SCORES_LABEL_MAJOR 1
int lec_score_topk_ex(int geom, int precision, const float* labels, int64_t L, const float* images,
                      int64_t N, int D, float K, const int32_t* level_start, const int32_t* level_stop,
                      int n_levels, int k, float* scores, int scores_layout, int32_t* topk_idx,
                      float* topk_val, void* stream);

/* Tensor-core variant (tcgen05.mma kind::tf32 with the 3xTF32 split, fp32 accumulators in TMEM, fused
 * angle / aperture / top-k epilogue): the <label, image> contraction leaves the FMA pipe, which is what
 * bounds lec_score_topk_ex at every D.  Hyperbolic geometry, LEC_PREC_F32, D <= 128, label-major scores.
 * The label side is repacked once per call into `workspace` (device memory, 128-byte aligned, at least
 * lec_score_workspace_bytes(L, D, n_levels) bytes, owned by the caller -- the library never allocates).
 * lec_score_tc_supported returns 1 when this entry point accepts the combination, else 0 (use
 * lec_score_topk_ex).  Same outputs and conventions as lec_score_topk_ex with LEC_SCORES_LABEL_MAJOR. */
int lec_score_tc_supported(int geom, int precision, int D, int64_t L, int n_levels);
int64_t lec_score_workspace_bytes(int64_t L, int D, int n_levels);
int lec_score_topk_tc(int geom, int precision, const float* labels, int64_t L, const float* images, int64_t N,
                      int D, float K, const int32_t* level_start, const int32_t* level_stop, int n_levels, int k,
                      float* scores, int32_t* topk_idx, float* topk_val, void* workspace, int64_t workspace_bytes,
                      void* stream);

/* ---- negative-edge sampler ----------------------------------------------------------------------
 * Replaces sample_negative_edge (order_embeddings.py:989-1008; joint variant oe.py:755-808) and the
 * B x N x 2 Python loop that calls it (order_embeddings.py:1070-1091, oe.py:846-863).  The reference's
 * dense negative_G (ones - transitive closure - diagonal, order_embeddings.py:417-423, oe.py:465-474) is
 * replaced by two CSR lists of EXCLUDED node ids, each sorted ascending:
 *   row_excl[row_excl_ptr[u] .. row_excl_ptr[u+1])   u itself and every closure descendant of u
 *   col_excl[col_excl_ptr[v] .. col_excl_ptr[v+1])   v itself and every closure ancestor of v
 * so the candidates of "corrupt the child of u" are [0, n_nodes) minus row_excl(u), in ascending order
 * (= np.where(negative_G[u, :] == 1)[0]), and likewise for "corrupt the parent of v" with col_excl(v).
 * pick_per_level != 0 restricts draw p to level (p % level_mod): label levels [level_start, level_stop)
 * for p % level_mod < n_levels (level_mod = n_levels, order_embeddings.py:990-1006); joint graphs pass
 * level_mod = n_levels + 1 and n_labels > 0, the extra slot being the image level (oe.py:786-804: label
 * candidates when the fixed endpoint is an image, image candidates otherwise).
 * Output layout (SURVEY F6): neg_to[i*N + p] = corrupted child of u_i, neg_from[i*N + p] = corrupted parent
 * of v_i; draw order per positive i, per p: row draw, then column draw. */
typedef struct {
    int64_t n_nodes;
    const int64_t* row_excl_ptr; const int32_t* row_excl;
    const int64_t* col_excl_ptr; const int32_t* col_excl;
    int pick_per_level; int n_levels; int level_mod;
    int32_t level_start[LEC_MAX_LEVELS]; int32_t level_stop[LEC_MAX_LEVELS];
    int64_t n_labels; /* joint graphs: node ids >= n_labels are images; 0 = label-only graph */
} lec_sampler_graph;

/* CPython's Mersenne Twister state (Modules/_randommodule.c): random.getstate()[1] = mt[0..623] + (index,) */
typedef struct { uint32_t mt[624]; int32_t index; } lec_mt19937;
/* random.seed(int): key = little-endian 32-bit words of |a| ({0} for 0), init_by_array */
int lec_mt_seed(lec_mt19937* s, const uint32_t* key, int key_words);
uint32_t lec_mt_uint32(lec_mt19937* s);
/* Random._randbelow_with_getrandbits(n), 0 < n < 2^32; LEC_E_EMPTY for n == 0 */
int64_t lec_mt_randbelow(lec_mt19937* s, uint32_t n);
/* EXACT mode, HOST pointers everywhere, runs on the calling thread: consumes `rng` exactly as the
 * reference's random.choice calls would (load random.getstate() before, store it back after), so the
 * indices are bit-exact.  LEC_E_EMPTY where the reference raises IndexError (rng is left mid-stream). */
int lec_sample_negatives(lec_mt19937* rng, const lec_sampler_graph* g, const int64_t* u, const int64_t* v,
                         int64_t B, int N, int64_t* neg_to, int64_t* neg_from);
/* FAST mode, one kernel: same candidate sets, same uniform law, Philox4x32-10 keyed by `seed`, counter
 * (i*N + p, stream_id): the block's low 64 bits make the row draw (draw id 2 (i*N + p)), its high 64 bits the column
 * draw (draw id 2 (i*N + p) + 1); not the reference's stream.  `g` is a HOST struct holding DEVICE
 * pointers; u, v, neg_to, neg_from are device arrays of idx_bytes-wide indices; *status (device int, zeroed
 * by the caller) receives LEC_E_EMPTY / LEC_E_INDEX if any draw failed. */
int lec_sample_negatives_philox(const lec_sampler_graph* g, const void* u, const void* v, int idx_bytes, int64_t B,
                                int N, uint64_t seed, uint64_t stream_id, void* neg_to, void* neg_from, int* status,
                                void* stream);
/* the fast mode's integer draw, on the host (for tests): uniform in [0, n) */
int64_t lec_philox_below(uint64_t seed, uint64_t stream_id, uint64_t draw, uint64_t n);

/* ---- an end-to-end training iteration from host memory ---------------------------------------------
 * Around the loss, one iteration of the reference's train loop moves the batch's indices to the device and the scalar
 * loss back (order_embeddings_h.py:752-775: `for index, data_item in enumerate(self.dataloaders[phase])` ...
 * `loss.item()`; order_embeddings.py:619-635).  lec_host_pipe_submit enqueues all of it with ONE call:
 *     copy stream  [wait until the kernels that last read dev_block are done] -> dev_block <- host_block (`bytes`)
 *                  [-> sample != NULL: lec_sample_negatives_philox draws step->neg_to / neg_from from step->pos_from /
 *                  pos_to on the device; it depends on no kernel of the step before, so it overlaps them] -> event
 *     `stream`     wait for that event -> lec_cone_step(step) -> event
 *     read-back    (a third stream) wait for that event -> *loss_host <- *step->upd.loss_step
 *                  [-> *err_host <- *step->xchg.error when world > 1] -> event
 * and returns without waiting for the GPU.  The index pointers of `step` point into dev_block (the caller lays the
 * block out: pos_from | pos_to | neg_to | neg_from, or just the positives in the sampled mode); host_block, loss_host and
 * err_host are PINNED host memory.  `slot` in [0, depth) names the staging slot: its events order the reuse of dev_block,
 * so the copy of step i+1 overlaps the kernels of step i.  Because the loss is read back BEHIND the main stream (no
 * copy sits between one step's update kernel and the next step's pair kernel), give every slot its own device word
 * step->upd.loss_step: a later step must not overwrite it before it has been read.  A slot must be collected with lec_host_pipe_wait (blocks
 * until its loss has landed) before it is submitted again (LEC_E_SIZE otherwise).  Not thread-safe per pipe. */
typedef struct lec_host_pipe lec_host_pipe_t;
typedef struct lec_host_sample {
    const lec_sampler_graph* graph; uint64_t seed, stream_id; int* status /* device int, see lec_sample_negatives_philox */;
} lec_host_sample_t;
int lec_host_pipe_create(lec_host_pipe_t** out, int depth /* 1..16 */);
void lec_host_pipe_destroy(lec_host_pipe_t* p);
int lec_host_pipe_submit(lec_host_pipe_t* p, int slot, const lec_step_t* step, const lec_host_sample_t* sample,
                         const void* host_block, int64_t bytes, void* dev_block, double* loss_host, int* err_host,
                         void* stream);
int lec_host_pipe_wait(lec_host_pipe_t* p, int slot);

/* ---- evaluation bookkeeping -----------------------------------------------------------------------
 * lec_f1_sweep replaces EmbeddingMetrics.calculate_metrics, 'val' phase (order_embeddings.py:272-287 = oe.py:380-395:
 * every unique energy is a candidate threshold, evaluated by a process pool with two passes over all energies each).
 *   sorted_energies  device float[n]: positive and negative energies together, ascending, NaN last
 *   pos_prefix       device int64[n]: number of POSITIVE-pair energies among sorted_energies[0..i]
 *   out7             device double[7]: {f1, threshold, accuracy, precision, recall, correct_positives, correct_negatives}
 *                    of the first threshold with maximal F1 -- the row calculate_metrics returns; computed with the
 *                    reference's fp64 expression tree, so equal to its Python floats bit for bit
 *   workspace        device, >= lec_f1_workspace_bytes() bytes */
int64_t lec_f1_workspace_bytes(void);
int lec_f1_sweep(const float* sorted_energies, const int64_t* pos_prefix, int64_t n, int64_t n_pos, int64_t n_neg,
                 double* out7, void* workspace, int64_t workspace_bytes, void* stream);

/* Reconstruction check without the energies: lec_recon_* replaces check_graph_embedding (order_embeddings.py:512-559 =
 * oe.py:1923-1990) at any size.  Positives are E(x = rows[u], y = rows[v]) for every v that is a strict descendant of
 * u (tin[u] < tin[v] <= tout[u], the Euler-tour intervals of the forest), negatives every other ordered pair u != v; the
 * result is the row lec_f1_sweep returns for those energies, bit for bit, where the energies are the ones
 * lec_score_topk_ex(..., LEC_PREC_F32, ...) computes for labels = images = rows.  Energies are histogrammed, never
 * stored: round 0 counts every pair into coarse bins, later rounds recount the pairs of the bins that can hold the
 * best threshold by exact value.
 *   rows           device [n, ld] fp32, 16-byte aligned; ld == D or ld % 4 == 0 (the padded rows of lec_rows_fwd)
 *   D              1..64 (what the SIMT scoring kernel supports)
 *   tin, tout      device int32[n]
 *   u_begin/u_end  the apex rows this call evaluates (a rank's share, [0, n) on one GPU); v always spans [0, n)
 *   workspace      device, 16-byte aligned, >= lec_recon_workspace_bytes(1) bytes, zeroed by the caller once before
 *                  round 0.  Its first lec_recon_counter_bytes(workspace_bytes) bytes are the counters a pass adds to;
 *                  ranks that split [0, n) sum that span (all_reduce) after every pass and before lec_recon_finish.
 * A round is lec_recon_pass then lec_recon_finish, which evaluates the round, clears the counters and writes
 *   out7           device double[7]: the best row found so far (final once status[0] == 0)
 *   status         device int64[4]: {1 if another round is needed else 0, coarse bins opened after round 0, n_pos, n_neg}
 * Neither call allocates or synchronises; the round lives in the workspace.  lec_recon_workspace_bytes returns the
 * size for a given number of coarse bins counted per fine round (about 1 MB each); more open bins take more rounds. */
typedef struct lec_recon {
    int geom; float K;
    const float* rows; int64_t n; int D; int ld;
    const int32_t* tin; const int32_t* tout;
    int64_t u_begin, u_end;
    void* workspace; int64_t workspace_bytes;
} lec_recon_t;
int64_t lec_recon_workspace_bytes(int open_bins_per_round);
int64_t lec_recon_counter_bytes(int64_t workspace_bytes);
int lec_recon_pass(const lec_recon_t* r, void* stream);
int lec_recon_finish(const lec_recon_t* r, double* out7, int64_t* status, void* stream);

/* lec_classify_counts replaces the per-image bookkeeping of JointEmbeddings.calculate_classification_metrics
 * (oe.py:1775-1796, oe_h.py:2030-2051) on the output of lec_score_topk*.
 *   topk_idx  device int32 [n_img, n_levels, k]   truth  device int32 [n_img, n_levels] (true label per level, < 0: skip)
 *   k_vals    HOST int32[n_kvals] (the reference's k = [1, 3, 5])
 *   hit            device uint64 [n_kvals, L]   += 1 at the TRUE label when it is among the first k_vals[j] predictions
 *   counts         device uint64 [3, L]         tp (at the true label), fp (at the predicted label), fn (at the true label)
 *   level_correct  device uint64 [n_levels]     correct top-1 predictions per level; tn[l] = level_correct[level(l)] - tp[l]
 * All three outputs are accumulated into (zero them first). */
int lec_classify_counts(const int32_t* topk_idx, const int32_t* truth, int64_t n_img, int n_levels, int k,
                        const int32_t* k_vals, int n_kvals, int64_t L, uint64_t* hit, uint64_t* counts,
                        uint64_t* level_correct, void* stream);

/* Caption-style ranking hinge of the image-label loss variant
 * OrderEmbeddingWithImagesLossvCaption.get_image_label_loss (order_embeddings_images.py:533-542):
 *     S_i = sum_j max(0, alpha + E+_i - E-_ij)        E_pos [B], E_neg [B, M] (row-major), S [B]
 * and, in the same pass, its VJP for an upstream gradient gS [B] (NULL = ones):
 *     gE_pos_i = gS_i * #{j : alpha + E+_i - E-_ij >= 0},   gE_neg_ij = -gS_i * [alpha + E+_i - E-_ij >= 0]
 * (torch.clamp(min=0) passes the gradient at equality; a NaN energy makes S_i NaN and contributes no gradient).
 * S, gE_pos, gE_neg are each optional.  Chains with lec_energy_dense / lec_energy_dense_bwd, which produce E and
 * consume dL/dE. */
int lec_caption_hinge(const float* E_pos, const float* E_neg, int64_t B, int M, float alpha, const float* gS, float* S,
                      float* gE_pos, float* gE_neg, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LEC_B200_H */
