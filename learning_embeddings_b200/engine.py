"""Step engine: one fused training step of a label-only cone model on preallocated buffers.

This is the public fast path (what bench.py drives).  It does what one iteration of the reference's
`pass_samples('train')` loop does between `optimizer.zero_grad()` and the weight update
(order_embeddings_h.py:752-775 for the hyperbolic trainer, order_embeddings.py:619-635 for the
Euclidean one) with the negatives already drawn, as two launches (lec_cone_step):

    loss, dL/drows = cone loss over B*(1+2N) pairs   lec_pairs_grouped   (rows / aux from the previous update)
    table = update(table, J^T sum_ranks dL/drows)    lec_update_rows: replica sum, [all-reduce over NVLink peer
    rows, aux = transform(table)                     memory], VJP of the row transform, RSGD / SGD / Adam, and the
                                                     row transform + aperture terms the NEXT step starts from

Index batches use the compact training layout of include/lec_b200.h (lec_pairs_grouped) as one uint16 / int32
block [pos_from | pos_to | neg_to | neg_from] so a step's indices travel host->device in one copy.
"""

import numpy as np
import torch

from . import _native as N
from . import ops
from . import sharding
from .criterion import inner_radius


def index_dtype_for(n_rows):
    """Narrowest index type the kernels take for a table of n_rows rows: uint16 up to 65 536 rows (ETHEC has
    723), else int32.  The index block is the only per-step host->device traffic, so its width is the
    end-to-end cost of a step."""
    return np.uint16 if n_rows <= 65536 else np.int32


def pack_index_block(pos_from, pos_to, neg_to, neg_from, pin=True, dtype=np.int32, n_rows=None):
    """Host index block [B | B | B*N | B*N] (int32, or uint16 for tables of <= 65 536 rows) for ConeStep.step_host.
    With n_rows the ids are checked against the table here, on the host, the way nn.Embedding checks them in the
    reference (the kernels also check, see lec_index_errors, but only report after the fact)."""
    parts = [np.ascontiguousarray(a).reshape(-1) for a in (pos_from, pos_to, neg_to, neg_from)]
    cat = np.concatenate(parts)
    if cat.size and (cat.min() < 0 or cat.max() > np.iinfo(dtype).max):
        raise ValueError("index out of range for %s" % np.dtype(dtype).name)
    if n_rows is not None and cat.size and cat.max() >= n_rows:
        raise IndexError("endpoint id %d outside the table of %d rows" % (int(cat.max()), int(n_rows)))
    blk = torch.from_numpy(cat.astype(dtype))
    return blk.pin_memory() if (pin and torch.cuda.is_available()) else blk


RULES = {"none": N.UPD_NONE, "rsgd": N.UPD_RSGD, "sgd": N.UPD_SGD, "adam": N.UPD_ADAM, "rsgd_retract": N.UPD_RSGD_RETRACT,
         "rsgd_lorentz": N.UPD_RSGD_LORENTZ}
# Nickel & Kiela's embeddings: geometry -> (pair kernel, its update rule)
_NK = {"poincare": ("lec_pairs_poincare", "rsgd_retract"), "lorentz": ("lec_pairs_lorentz", "rsgd_lorentz")}


class ConeStep:
    """update: "rsgd" (order_embeddings_h.py:764-775), "sgd" / "adam" (torch.optim semantics, order_embeddings.py:563-565),
    "none" (gradient only, left in grad_table), "auto" = rsgd for hyperbolic cones, sgd otherwise.  hyp_rescale /
    project_shell: the joint hyperbolic trainer's gradient rescale and table projection around sgd / adam
    (oe_h.py:1765-1771).  Every rule runs inside the library's fused update kernel (lec_update_rows).

    geom="poincare": Nickel & Kiela's Poincare embeddings -- the softmax loss over each positive and its n_neg
    negatives (lec_pairs_poincare; neg_from is not read, E_neg is [max_groups, n_neg]) and update "rsgd_retract" (the
    default: w <- proj(w - lr (1 - |w|^2)^2 / 4 g)) or "none".  The table is used as it is (no row transform, no aux
    terms); K, alpha and pair weights do not apply.

    geom="lorentz": Nickel & Kiela's Lorentz-model embeddings, the same loss on the hyperboloid distance
    (lec_pairs_lorentz; each table row is the spatial part x of the point (sqrt(1 + |x|^2), x)) and update "rsgd_lorentz"
    (the default: the exponential map x <- cosh(t) x - lr sinh(t)/t (g + <x,g> x), t = lr sqrt(|g|^2 + <x,g>^2)) or
    "none", with the same restrictions as "poincare"."""

    def __init__(self, table, geom, n_neg, max_groups, K=None, alpha=1.0, lr=1e-3, row_mode=None, update="auto",
                 precision=ops.PREC_F64CORE, process_group=None, replicas=None, comm="auto", momentum=0.0,
                 betas=(0.9, 0.999), eps=1e-8, hyp_rescale=False, project_shell=False, exchange=None, exchange_mode=None):
        N.require_cuda(table)
        if table.dtype != torch.float32 or not table.is_contiguous():
            raise N.LecError("ConeStep: table must be a contiguous float32 CUDA tensor (updated in place)")
        self.table = table
        self.geom = geom
        self.n, self.D = table.shape
        self.ld = ops.padded_dim(self.D)
        self.n_neg = int(n_neg)
        nk = geom in _NK   # the softmax loss of Nickel & Kiela: no aux terms, E_neg [max_groups, n_neg]
        self.K = {"euc": 3.0, "hyp": 0.1, "oe": 0.0, "poincare": 0.0, "lorentz": 0.0}[geom] if K is None else float(K)
        self.alpha = float(alpha)
        self.lr = float(lr)
        self.row_mode = {"euc": N.ROWS_EUC_SOFTCLIP, "hyp": N.ROWS_HYP_SHELL, "oe": N.ROWS_NONE, "poincare": N.ROWS_NONE,
                         "lorentz": N.ROWS_NONE}[geom] if row_mode is None else int(row_mode)
        if update == "auto":
            update = _NK[geom][1] if nk else ("rsgd" if geom == "hyp" else "sgd")
        self.update = update
        if self.update not in RULES:
            raise N.LecError("unknown update rule %r" % (self.update,))
        if nk and (self.update not in (_NK[geom][1], "none") or self.row_mode != N.ROWS_NONE):
            raise N.LecError("ConeStep(geom=%r): update must be %r or 'none' on untransformed rows, got update=%r, "
                             "row_mode=%d" % (geom, _NK[geom][1], self.update, self.row_mode))
        if self.update == "rsgd_retract" and geom != "poincare":
            raise N.LecError("update 'rsgd_retract' is the Poincare embeddings' rule (geom='poincare')")
        if self.update == "rsgd_lorentz" and geom != "lorentz":
            raise N.LecError("update 'rsgd_lorentz' is the Lorentz embeddings' rule (geom='lorentz')")
        self.momentum, self.betas, self.eps = float(momentum), (float(betas[0]), float(betas[1])), float(eps)
        self.hyp_rescale, self.project_shell = bool(hyp_rescale), bool(project_shell)
        self.r_in = float(inner_radius(self.K)) if geom == "hyp" else 0.0
        self.precision = int(precision)
        self.pg = process_group
        self.max_groups = int(max_groups)
        dev = table.device
        self.replicas = ops.default_replicas(self.n, self.ld) if replicas is None else int(replicas)
        self.rows = torch.empty((self.n, self.ld), device=dev, dtype=torch.float32)
        self.aux = None if nk else torch.empty((self.n, 4), device=dev, dtype=torch.float64)
        self.grad_rows = torch.empty((self.replicas, self.n, self.ld), device=dev, dtype=torch.float32)
        self.grad_table = torch.empty((self.n, self.D), device=dev, dtype=torch.float32)
        self.E_pos = torch.empty(self.max_groups, device=dev, dtype=torch.float32)
        self.E_neg = torch.empty((self.max_groups, (1 if nk else 2) * self.n_neg), device=dev, dtype=torch.float32)
        # the pair kernel adds into loss_acc; the update kernel moves it to `loss` (this rank's loss of the latest step)
        self.loss = torch.zeros(1, device=dev, dtype=torch.float64)
        self._loss_ptr = self.loss.data_ptr()
        self.loss_acc = torch.zeros(1, device=dev, dtype=torch.float64)
        self.opt_m = self.opt_v = None
        if self.update == "adam" or (self.update == "sgd" and self.momentum != 0.0):
            self.opt_m = torch.zeros((self.n, self.ld), device=dev, dtype=torch.float32)
        if self.update == "adam":
            self.opt_v = torch.zeros((self.n, self.ld), device=dev, dtype=torch.float32)
        self.opt_step = 0
        self.write_grad_table = self.update == "none"   # set to True to keep d loss / d table of every step
        # the update also produces the rows / aux / cleared replicas the next step starts from (two launches per step);
        # only the first step, and the first after invalidate_rows(), runs lec_rows_fwd first (three launches)
        self._rows_valid = False
        # host->device staging: `depth` slots so that the copies of steps i+1, i+2 overlap the kernels of step i (r2: with
        # host-drawn negatives the step is PCIe-bound; depth 2 -> 3: 101 -> 88.6 us per step, no change beyond 3)
        self.depth = 3
        self._idx_bytes_dev = [torch.empty(self.max_groups * (2 + 2 * self.n_neg) * 4, device=dev, dtype=torch.uint8)
                               for _ in range(self.depth)]
        self.loss_host = torch.zeros(self.depth, dtype=torch.float64).pin_memory()
        self.err_host = torch.zeros(self.depth, dtype=torch.int32).pin_memory()
        self._pipe, self._sample_struct, self._sample_graph = None, None, None
        self._copy_stream = None
        self._ev = None          # per slot: (indices copied, kernels done with the slot, loss read back)
        self._inflight = [False] * self.depth
        self._submitted = 0
        self._losses = []
        self.kernel_events = None  # optional (start, stop) pairs around the pair kernel, set by bench
        self._struct = None
        # multi-GPU exchange: "p2p" = one-shot low-latency all-reduce over NVLink peer memory inside the update kernel,
        # "nccl" = all_reduce of the summed gradient between the pair kernel and the update kernel
        self.comm, self.comm_note, self.px = "none", "", exchange
        world = torch.distributed.get_world_size(self.pg) if self.pg is not None else 1
        if exchange is not None:
            self.comm = "p2p"
        elif world > 1:
            self.comm = "nccl"
            if comm in ("p2p", "auto"):
                try:
                    # one-shot packets for label-sized tables, owner-computes two-shot for multi-megabyte ones
                    self.px = sharding.PeerExchange(self.n, self.ld, dev, self.pg, mode=exchange_mode)
                    self.comm = "p2p"
                    self.comm_note = "two-shot (reduce-scatter + owner update + all-gather)" if self.px.mode == sharding.TWO_SHOT \
                        else "one-shot packets inside the update kernel"
                except Exception as e:  # noqa: BLE001 -- any failure of the symmetric-memory setup
                    if comm == "p2p":
                        raise
                    self.comm_note = "p2p unavailable (%s: %s)" % (type(e).__name__, str(e)[:120])
        if self.comm == "nccl":
            self.grad_sum = torch.empty((self.n, self.ld), device=dev, dtype=torch.float32)
        self.loss_global = self.px.loss_global if self.px is not None else torch.zeros(1, device=dev, dtype=torch.float64)

    # -- pieces ---------------------------------------------------------------------------------
    def _split(self, blk, B):
        Nn = self.n_neg
        return blk[:B], blk[B:2 * B], blk[2 * B:2 * B + B * Nn], blk[2 * B + B * Nn:2 * B + 2 * B * Nn]

    def set_lr(self, lr):
        """Learning-rate schedules (the reference decays lr every epoch, order_embeddings_h.py:620) take effect on the
        next step; assigning `engine.lr` directly works too."""
        self.lr = float(lr)

    def _fill_update(self, u, grad_rows=None, replicas=None):
        """lec_update_t for the next step (scalars are re-read every step, so lr / alpha / K may change between steps)."""
        if getattr(u, "_lec_static", None) is self and grad_rows is None:
            # the pointers and shapes of this engine are already in the struct: only what may change between steps
            u.rule, u.K, u.lr, u.r_in, u.opt_step = RULES[self.update], self.K, self.lr, self.r_in, self.opt_step + 1
            u.grad_out = self.grad_table.data_ptr() if self.write_grad_table else None
            return u
        u.rule, u.row_mode, u.geom, u.lambda_mode = RULES[self.update], self.row_mode, N.GEOM[self.geom], 0
        u.hyp_rescale, u.project_shell = int(self.hyp_rescale), int(self.project_shell)
        u.K, u.lr, u.r_in = self.K, self.lr, self.r_in
        u.momentum, u.beta1, u.beta2, u.eps = self.momentum, self.betas[0], self.betas[1], self.eps
        u.opt_step = self.opt_step + 1
        u.table, u.n, u.D, u.ld = self.table.data_ptr(), self.n, self.D, self.ld
        u.grad_rows = (self.grad_rows if grad_rows is None else grad_rows).data_ptr()
        u.grad_replicas = self.replicas if replicas is None else replicas
        u.state_m = self.opt_m.data_ptr() if self.opt_m is not None else None
        u.state_v = self.opt_v.data_ptr() if self.opt_v is not None else None
        u.rows_out, u.aux_out = self.rows.data_ptr(), self.aux.data_ptr() if self.aux is not None else None
        u.grad_out = self.grad_table.data_ptr() if self.write_grad_table else None
        u.loss_acc, u.loss_step = self.loss_acc.data_ptr(), self.loss.data_ptr()
        if grad_rows is None:
            u._lec_static = self
        return u

    def _rows_fwd(self):
        N.check(N.lib().lec_rows_fwd(N._p(self.table), self.n, self.D, self.row_mode, N.GEOM[self.geom], self.K,
                                     N._p(self.rows), self.ld, N._p(self.aux), N._p(self.grad_rows), self.replicas, 0,
                                     N._p(self.loss_acc), N.stream_ptr(self.table.device)), "lec_rows_fwd")

    def forward_backward(self, pos_from, pos_to, neg_to, neg_from, w_pos=None, w_neg=None):
        """rows, loss and d loss / d rows for one batch (no collective, no update): the loss is left in loss_acc, the
        gradient in the replicas; reduce_and_update() finishes the step."""
        lib, st = N.lib(), N.stream_ptr(self.table.device)
        B = int(pos_from.numel())
        if B > self.max_groups:
            raise N.LecError("batch of %d positives exceeds max_groups=%d" % (B, self.max_groups))
        if not self._rows_valid:
            self._rows_fwd()
        self._rows_valid = False
        ev = self.kernel_events
        if ev is not None:
            ev[0].record()
        if self.geom in _NK:
            if w_pos is not None or w_neg is not None:
                raise N.LecError("the softmax loss of geom=%r takes no pair weights" % (self.geom,))
            name = _NK[self.geom][0]
            N.check(getattr(lib, name)(
                self.precision, N._p(self.rows), self.n, self.D, self.ld, N._p(pos_from), N._p(pos_to), N._p(neg_to),
                pos_from.element_size(), B, self.n_neg, N._p(self.E_pos), N._p(self.E_neg), N._p(self.loss_acc),
                N._p(self.grad_rows), self.replicas, st), name)
        else:
            N.check(lib.lec_pairs_grouped(
                N.GEOM[self.geom], self.precision, N._p(self.rows), N._p(self.aux), self.n, self.D, self.ld,
                N._p(pos_from), N._p(pos_to),
                N._p(neg_to), N._p(neg_from), pos_from.element_size(), B, self.n_neg, N._p(w_pos), N._p(w_neg), self.K,
                self.alpha, N._p(self.E_pos), N._p(self.E_neg), N._p(self.loss_acc), N._p(self.grad_rows), self.replicas,
                st), "lec_pairs_grouped")
        if ev is not None:
            ev[1].record()
        return B

    def invalidate_rows(self):
        """Call after changing `table` from outside the engine (loading weights, a manual update): the fused step
        otherwise reuses the transformed rows its previous update left behind."""
        self._rows_valid = False

    def reduce_and_update(self, phases=0):
        """Second half of a step issued as separate calls: [exchange] + update + next rows (lec_update_rows).  `phases`
        (two-shot exchange only): bit mask of the launches to issue now -- 1 scatter, 2 owner, 4 receiver; 0 = all."""
        import ctypes
        lib, st = N.lib(), N.stream_ptr(self.table.device)
        u, x = N.LecUpdate(), N.LecExchange()
        if self.comm == "nccl":
            # sum of the replicas -> one NCCL all-reduce -> the update reads the reduced buffer as a single replica
            N.check(lib.lec_reduce_replicas(N._p(self.grad_rows), self.replicas, self.n * self.ld, N._p(self.grad_sum), st),
                    "lec_reduce_replicas")
            self.grad_rows.zero_()
            torch.distributed.all_reduce(self.grad_sum, group=self.pg)
            self._fill_update(u, self.grad_sum, 1)
        else:
            self._fill_update(u)
            if self.comm == "p2p":
                self.px.fill(x)
                x.phases = int(phases)
        N.check(lib.lec_update_rows(ctypes.byref(u), ctypes.byref(x) if self.comm == "p2p" else None, st), "lec_update_rows")
        if not phases or (phases & 4):
            self._after_step()

    def _after_step(self):
        if self.update != "none":
            self.opt_step += 1
        if self.comm == "p2p":
            self.px.step += 1
        self._rows_valid = True

    def check_exchange(self):
        """Raises if the peer exchange reported a failure (a rank did not deliver its gradient in time).  Synchronises."""
        if self.px is not None and int(self.px.error.item()) != 0:
            raise N.LecError("peer exchange timed out: a rank did not deliver its gradient; the table replicas are no "
                             "longer in step -- restart from a checkpoint")

    def global_loss(self):
        """Loss of the latest step summed over ranks (float64 tensor on the device)."""
        if self.comm == "p2p":
            self.check_exchange()
            return self.loss_global.clone()
        out = self.loss.clone()
        if self.pg is not None and torch.distributed.get_world_size(self.pg) > 1:
            torch.distributed.all_reduce(out, group=self.pg)
        return out

    # -- whole steps ----------------------------------------------------------------------------
    def _fill_step(self, p_from, p_to, n_to, n_from, idx_bytes, B, w_pos=None, w_neg=None, loss_ptr=None):
        """lec_step_t of the next step (pointers as integers).  One cached ctypes struct: pointers and shapes of this
        engine are written once, the per-step fields every time (lr / alpha / K may change between steps)."""
        if B > self.max_groups:
            raise N.LecError("batch of %d positives exceeds max_groups=%d" % (B, self.max_groups))
        s = self._struct
        if s is None:
            s = self._struct = N.LecStep()
            self._upd = s.upd    # ONE wrapper of the embedded struct (every `s.upd` would build a new Python object)
            s.E_pos, s.E_neg, s.N = self.E_pos.data_ptr(), self.E_neg.data_ptr(), self.n_neg
            s.xchg.world = 0
            if self.comm == "p2p":
                self.px.fill(s.xchg)
        s.geom, s.precision, s.alpha = N.GEOM[self.geom], self.precision, self.alpha
        s.fused = 1 if self._rows_valid else 0
        s.pos_from, s.pos_to, s.neg_to, s.neg_from = p_from, p_to, n_to, n_from
        s.idx_bytes, s.B = idx_bytes, B
        s.w_pos = w_pos.data_ptr() if w_pos is not None else None
        s.w_neg = w_neg.data_ptr() if w_neg is not None else None
        self._fill_update(self._upd)
        self._upd.loss_step = self._loss_ptr if loss_ptr is None else loss_ptr   # pipelined steps: one word per slot
        if self.comm == "p2p":
            s.xchg.slot, s.xchg.tag = self.px.slot_and_tag()
        ev = self.kernel_events
        if ev is not None:
            for e in ev:
                if not e.cuda_event:
                    e.record()  # torch creates the cudaEvent lazily
            s.ev_pairs_start, s.ev_pairs_stop = ev[0].cuda_event, ev[1].cuda_event
        else:
            s.ev_pairs_start, s.ev_pairs_stop = None, None
        return s

    def step_device(self, pos_from, pos_to, neg_to, neg_from, w_pos=None, w_neg=None):
        """Indices already on the device (uint16 / int32 / int64).  Returns this rank's device loss (float64[1])."""
        if self.comm == "nccl":
            self.forward_backward(pos_from, pos_to, neg_to, neg_from, w_pos, w_neg)
            self.reduce_and_update()
            return self.loss
        # the whole step as ONE call into the library (lec_cone_step): one FFI crossing, two launches
        import ctypes
        s = self._fill_step(pos_from.data_ptr(), pos_to.data_ptr(), neg_to.data_ptr(), neg_from.data_ptr(),
                            pos_from.element_size(), int(pos_from.numel()), w_pos, w_neg)
        N.check(N.lib().lec_cone_step(ctypes.byref(s), N.stream_ptr(self.table.device)), "lec_cone_step")
        self._after_step()
        return self.loss

    def step_sampled(self, graph, pos_from, pos_to, seed, step):
        """Device-resident training step: negatives are drawn on the GPU (sampler.SamplerGraph.draw_philox: the
        reference's candidate sets and uniform law, Philox stream keyed by (seed, step)) and consumed by the step in the
        same stream -- only the positive edges ever come from the host.  The fast mode: not the `random.choice` stream."""
        B = int(pos_from.numel())
        key = (pos_from.dtype, B)
        if getattr(self, "_neg_key", None) != key:
            dev = self.table.device
            self._neg_bufs = (torch.empty((B, self.n_neg), dtype=pos_from.dtype, device=dev),
                              torch.empty((B, self.n_neg), dtype=pos_from.dtype, device=dev))
            self._neg_key = key
        neg_to, neg_from = graph.draw_philox(pos_from, pos_to, self.n_neg, seed, step, out=self._neg_bufs, check=False)
        return self.step_device(pos_from, pos_to, neg_to.view(-1), neg_from.view(-1))

    def _slot_view(self, slot, n, dtype):
        return self._idx_bytes_dev[slot][:n * dtype.itemsize].view(dtype)

    def step_host(self, index_block, B):
        """index_block: pinned host block from pack_index_block (uint16 / int32).  Copies it in, runs the
        step and reads the scalar loss back (one H2D, one D2H, one sync) -- the synchronous end-to-end path."""
        self._collect()
        n = B * (2 + 2 * self.n_neg)
        dst = self._slot_view(0, n, index_block.dtype)
        dst.copy_(index_block[:n], non_blocking=True)
        self.step_device(*self._split(dst, B))
        self.loss_host[:1].copy_(self.loss, non_blocking=True)
        if self.px is not None:
            self.err_host[:1].copy_(self.px.error, non_blocking=True)
        torch.cuda.current_stream(self.table.device).synchronize()
        self._raise_on(0)
        return float(self.loss_host[0])

    def _raise_on(self, slot):
        if self.px is not None and int(self.err_host[slot]) != 0:
            raise N.LecError("peer exchange timed out: a rank did not deliver its gradient; the table replicas are no "
                             "longer in step -- restart from a checkpoint")

    # -- end-to-end iterations through the library's host pipe (lec_host_pipe_*) ---------------------------------
    def _pipe_slot(self):
        """The staging slot of the next submission, collected if a step is still in flight on it (blocks on that
        step's loss, i.e. on step i - depth)."""
        import ctypes
        lib = N.lib()
        if self._pipe is None:
            h = ctypes.c_void_p()
            N.check(lib.lec_host_pipe_create(ctypes.byref(h), self.depth), "lec_host_pipe_create")
            self._pipe = h
            self._slot_ptr = [b.data_ptr() for b in self._idx_bytes_dev]
            self._loss_np, self._err_np = self.loss_host.numpy(), self.err_host.numpy()
            self._loss_host_ptr = [self.loss_host.data_ptr() + 8 * i for i in range(self.depth)]
            # the step's loss on the device, one word per slot: it is read back behind the main stream
            self._loss_slots = torch.zeros(self.depth, dtype=torch.float64, device=self.table.device)
            self._loss_slot_ptr = [self._loss_slots.data_ptr() + 8 * i for i in range(self.depth)]
            self._err_ptr = [self.err_host.data_ptr() + 4 * i for i in range(self.depth)]
        slot = self._submitted % self.depth
        if self._inflight[slot]:
            self._collect_slot(slot)
        return slot

    def _collect_slot(self, slot):
        N.check(N.lib().lec_host_pipe_wait(self._pipe, slot), "lec_host_pipe_wait")
        self._inflight[slot] = False
        self._raise_on(slot)
        self._losses.append(float(self._loss_np[slot]))

    def _pipe_submit(self, slot, s, sample, host_block, nbytes):
        import ctypes
        N.check(N.lib().lec_host_pipe_submit(self._pipe, slot, ctypes.byref(s), sample, host_block.data_ptr(), nbytes,
                                             self._slot_ptr[slot], self._loss_host_ptr[slot],
                                             self._err_ptr[slot] if self.px is not None else None,
                                             N.stream_ptr(self.table.device)), "lec_host_pipe_submit")
        self._after_step()
        self._inflight[slot] = True
        self._submitted += 1

    def submit_host(self, index_block, B):
        """Pipelined end-to-end step: ONE library call (lec_host_pipe_submit) copies the pinned index block
        host->device on a side stream into one of `depth` staging slots while the previous step's kernels run,
        enqueues the step behind the copy and the read-back of its loss behind the step.  Blocks only when the slot it
        needs is still in flight (i.e. on the loss of step i - depth).  Losses are returned, in order, by drain()."""
        if self.comm == "nccl":
            return self._submit_host_torch(index_block, B)
        slot = self._pipe_slot()
        ib, Nn, base = index_block.element_size(), self.n_neg, self._slot_ptr[slot]
        s = self._fill_step(base, base + B * ib, base + 2 * B * ib, base + (2 + Nn) * B * ib, ib, B,
                            loss_ptr=self._loss_slot_ptr[slot])
        self._pipe_submit(slot, s, None, index_block, B * (2 + 2 * Nn) * ib)

    def submit_host_sampled(self, graph, pos_block, B, seed):
        """Pipelined end-to-end step in the device-sampled mode: only the step's POSITIVE edges travel host->device
        (pos_block = pinned [pos_from | pos_to], uint16 / int32: 4 B bytes instead of 4 B (1 + N)); the negatives are
        drawn on the GPU by the library's Philox sampler (the reference's candidate sets and uniform law, not its
        random.choice stream) right before the step, in the same stream and the same library call.  Losses come back
        through drain()."""
        if self.comm == "nccl":
            return self._submit_host_sampled_torch(graph, pos_block, B, seed)
        import ctypes
        slot = self._pipe_slot()
        ib, Nn, base = pos_block.element_size(), self.n_neg, self._slot_ptr[slot]
        s = self._fill_step(base, base + B * ib, base + 2 * B * ib, base + (2 + Nn) * B * ib, ib, B,
                            loss_ptr=self._loss_slot_ptr[slot])
        smp = self._sample_struct
        if smp is None or self._sample_graph is not graph:
            g, keep, status = graph.device_struct(self.table.device)
            smp = self._sample_struct = N.LecHostSample()
            self._sample_graph, self._sample_keep = graph, (g, keep, status)
            smp.graph, smp.status = ctypes.addressof(g), status.data_ptr()
        smp.seed, smp.stream_id = int(seed), self._submitted
        self._pipe_submit(slot, s, ctypes.byref(smp), pos_block, 2 * B * ib)

    def close(self):
        """Releases the host pipe (its stream and events).  Called by __del__; safe to call twice."""
        if getattr(self, "_pipe", None) is not None:
            self._collect()
            N.lib().lec_host_pipe_destroy(self._pipe)
            self._pipe = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 -- interpreter shutdown
            pass

    # the NCCL exchange is a torch.distributed call between the two halves of a step, so that path keeps the host side
    # in Python (stream switch, copy, events)
    def _submit_host_torch(self, index_block, B):
        dev = self.table.device
        main = torch.cuda.current_stream(dev)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(dev)
            self._ev = [tuple(torch.cuda.Event() for _ in range(3)) for _ in range(self.depth)]
        slot = self._submitted % self.depth
        ev_copied, ev_free, ev_loss = self._ev[slot]
        if self._inflight[slot]:
            ev_loss.synchronize()
            self._raise_on(slot)
            self._losses.append(float(self.loss_host[slot]))
        n = B * (2 + 2 * self.n_neg)
        dst = self._slot_view(slot, n, index_block.dtype)
        with torch.cuda.stream(self._copy_stream):
            if self._inflight[slot]:
                self._copy_stream.wait_event(ev_free)
            dst.copy_(index_block[:n], non_blocking=True)
            ev_copied.record(self._copy_stream)
        main.wait_event(ev_copied)
        self.step_device(*self._split(dst, B))
        ev_free.record(main)
        self.loss_host[slot:slot + 1].copy_(self.loss, non_blocking=True)
        ev_loss.record(main)
        self._inflight[slot] = True
        self._submitted += 1

    def _submit_host_sampled_torch(self, graph, pos_block, B, seed):
        dev = self.table.device
        main = torch.cuda.current_stream(dev)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(dev)
            self._ev = [tuple(torch.cuda.Event() for _ in range(3)) for _ in range(self.depth)]
        slot = self._submitted % self.depth
        ev_copied, ev_free, ev_loss = self._ev[slot]
        if self._inflight[slot]:
            ev_loss.synchronize()
            self._raise_on(slot)
            self._losses.append(float(self.loss_host[slot]))
        dst = self._slot_view(slot, 2 * B, pos_block.dtype)
        with torch.cuda.stream(self._copy_stream):
            if self._inflight[slot]:
                self._copy_stream.wait_event(ev_free)
            dst.copy_(pos_block[:2 * B], non_blocking=True)
            ev_copied.record(self._copy_stream)
        main.wait_event(ev_copied)
        self.step_sampled(graph, dst[:B], dst[B:2 * B], seed, self._submitted)
        ev_free.record(main)
        self.loss_host[slot:slot + 1].copy_(self.loss, non_blocking=True)
        ev_loss.record(main)
        self._inflight[slot] = True
        self._submitted += 1

    def drain(self):
        """Wait for every submitted step; returns their losses in submission order (and forgets them)."""
        self._collect()
        out, self._losses = self._losses, []
        return out

    def _collect(self):
        for k in range(self.depth):
            slot = (self._submitted + k) % self.depth  # oldest first
            if not self._inflight[slot]:
                continue
            if self._pipe is not None:
                self._collect_slot(slot)
            elif self._ev is not None:
                self._ev[slot][2].synchronize()
                self._raise_on(slot)
                self._losses.append(float(self.loss_host[slot]))
                self._inflight[slot] = False


class JointConeStep:
    """One fused training step of a JOINT image+label cone model (the reference's oe.py / oe_h.py trainers,
    `JointEmbeddings.pass_samples('train')`, oe.py:1489-1560 / oe_h.py:1730-1771) on preallocated buffers, seven
    launches of this library and nothing else:

        Y        = fc1(features[img_sel])                    lec_featnet_fwd  (gather fused into the projection)
        img rows = transform(Y), their aperture terms        lec_rows_fwd     (FeatNet tail; clears their gradient rows)
        loss, dL/drows over B*(1+2N) pairs                   lec_pairs_grouped on the concatenated [labels ; images] rows
        dL/dY    = J^T dL/d(img rows)                        lec_rows_bwd
        dL/dfc1  = dL/dY^T features[img_sel], dL/dbias       lec_featnet_wgrad (second and last pass over the features)
        table  <- rule(table, J^T dL/d(label rows))          lec_update_rows  (+ the label rows / aperture terms of the
        fc1    <- Adam(fc1, dL/dfc1)                         lec_update_rows    NEXT step; both with the peer exchange
                                                                               when world_size > 1)

    Endpoints are row numbers of the concatenated table: < n_labels a label, >= n_labels image (index - n_labels) of
    this step's img_sel.  Update rules: Euclidean / order embeddings: Adam on both parameter groups with their own
    learning rates (oe.py:1356-1357, :1714); hyperbolic: the label gradient is rescaled by ((1-|w|)/2)^2, Adam, then the
    table is projected back into the shell (oe_h.py:1765-1771) -- or, with update="rsgd", the exponential-map update
    of oe_h.py:1757-1762 -- while fc1 takes plain Adam.  update="none" leaves the parameters alone and the three
    gradients in g_table / g_w / g_b.

    fc1's weight and bias are kept in ONE flat buffer (fc_w / fc_b are views of it; the constructor copies the
    tensors it is given): the update kernel treats it as an [n, 16] table of plain parameters."""

    FC_LD = 16

    def __init__(self, table, fc_weight, fc_bias, features, geom, n_neg, max_groups, max_images, K=None, alpha=1.0,
                 lr=1e-3, precision=ops.PREC_F64CORE, process_group=None, update="auto", lr_fc=None, comm="auto",
                 exchange=None):
        N.require_cuda(table, fc_weight, fc_bias, features)
        self.table, self.features = table, features
        self.geom = geom
        self.n, self.D = table.shape
        self.ld = ops.padded_dim(self.D)
        self.n_neg, self.max_groups, self.max_images = int(n_neg), int(max_groups), int(max_images)
        self.K = {"euc": 3.0, "hyp": 0.1, "oe": 0.0}[geom] if K is None else float(K)
        self.alpha, self.lr, self.precision = float(alpha), float(lr), int(precision)
        self.lr_fc = float(lr if lr_fc is None else lr_fc)
        self.lab_mode = {"euc": N.ROWS_EUC_SOFTCLIP, "hyp": N.ROWS_HYP_TANH, "oe": N.ROWS_NONE}[geom]
        self.img_mode = {"euc": N.ROWS_EUC_SOFTCLIP, "hyp": N.ROWS_HYP_TANH_FEAT, "oe": N.ROWS_NONE}[geom]
        self.update = "adam" if update == "auto" else update
        if self.update not in ("adam", "rsgd", "none") or (self.update == "rsgd" and geom != "hyp"):
            raise N.LecError("JointConeStep: update must be adam, none, or rsgd (hyperbolic only), got %r" % (update,))
        self.r_in = float(inner_radius(self.K)) if geom == "hyp" else 0.0
        self.pg = process_group
        dev = table.device
        F = features.shape[1]
        self.F = F
        if not N.lib().lec_featnet_supported(F, self.D):
            raise N.LecError("JointConeStep: FeatNet of %d -> %d is outside lec_featnet_* (D <= 16, F %% 4 == 0, F <= 4096)" % (F, self.D))
        nt = self.n + self.max_images
        self.n_total = nt
        self.replicas = ops.default_replicas(nt, self.ld)
        self.Y = torch.empty((self.max_images, self.D), device=dev, dtype=torch.float32)
        self.rows = torch.empty((nt, self.ld), device=dev, dtype=torch.float32)
        self.aux = torch.empty((nt, 4), device=dev, dtype=torch.float64)
        self.grad_rows = torch.zeros((self.replicas, nt, self.ld), device=dev, dtype=torch.float32)
        self.gY = torch.empty((self.max_images, self.D), device=dev, dtype=torch.float32)
        # fc1 as one flat parameter vector [D*F weights | D biases | pad], its gradient replicas and Adam moments
        self.n_fc = (self.D * F + self.D + self.FC_LD - 1) // self.FC_LD
        self.fc_flat = torch.zeros(self.n_fc * self.FC_LD, device=dev, dtype=torch.float32)
        self.fc_w = self.fc_flat[:self.D * F].view(self.D, F)
        self.fc_b = self.fc_flat[self.D * F:self.D * F + self.D]
        with torch.no_grad():
            self.fc_w.copy_(fc_weight)
            self.fc_b.copy_(fc_bias)
        self.fc_replicas = 8
        self.fc_grad = torch.zeros((self.fc_replicas, self.n_fc * self.FC_LD), device=dev, dtype=torch.float32)
        self.g_fc = torch.zeros(self.n_fc * self.FC_LD, device=dev, dtype=torch.float32)
        self.g_w = self.g_fc[:self.D * F].view(self.D, F)
        self.g_b = self.g_fc[self.D * F:self.D * F + self.D]
        self.g_table = torch.zeros((self.n, self.D), device=dev, dtype=torch.float32)
        self.write_grads = self.update == "none"
        self.opt = {k: torch.zeros((self.n, self.ld), device=dev) for k in ("m", "v")}
        self.opt_fc = {k: torch.zeros(self.n_fc * self.FC_LD, device=dev) for k in ("m", "v")}
        self.opt_step = 0
        self.E_pos = torch.empty(self.max_groups, device=dev, dtype=torch.float32)
        self.E_neg = torch.empty((self.max_groups, 2 * self.n_neg), device=dev, dtype=torch.float32)
        self.loss = torch.zeros(1, device=dev, dtype=torch.float64)
        self.loss_acc = torch.zeros(1, device=dev, dtype=torch.float64)
        self.kernel_events = None
        self._rows_valid = False
        self._sel_dev = torch.empty(self.max_images, device=dev, dtype=torch.int64)
        self._idx_bytes_dev = torch.empty(self.max_groups * (2 + 2 * self.n_neg) * 4, device=dev, dtype=torch.uint8)
        self.loss_host = torch.zeros(1, dtype=torch.float64).pin_memory()
        # multi-GPU: two exchanges per step (label table, fc1), each inside its update kernel
        self.comm, self.px, self.px_fc = "none", None, None
        world = torch.distributed.get_world_size(self.pg) if self.pg is not None else 1
        if exchange is not None:
            self.px, self.px_fc = exchange
            self.comm = "p2p"
        elif world > 1:
            if comm == "nccl":
                raise N.LecError("JointConeStep exchanges gradients inside its update kernels (comm='p2p')")
            self.px = sharding.PeerExchange(self.n, self.ld, dev, self.pg)
            self.px_fc = sharding.PeerExchange(self.n_fc, self.FC_LD, dev, self.pg)
            self.comm = "p2p"
        self.loss_global = self.px.loss_global if self.px is not None else self.loss

    def _split(self, blk, B):
        Nn = self.n_neg
        return blk[:B], blk[B:2 * B], blk[2 * B:2 * B + B * Nn], blk[2 * B + B * Nn:2 * B + 2 * B * Nn]

    def invalidate_rows(self):
        self._rows_valid = False

    def _update_struct(self, which):
        cache = self.__dict__.setdefault("_ucache", {})
        if which in cache:
            u = cache[which]
            u.opt_step = self.opt_step + 1
            u.lr = self.lr if which == "table" else self.lr_fc
            return u
        u = cache[which] = N.LecUpdate()
        u.lambda_mode, u.beta1, u.beta2, u.eps, u.momentum = 0, 0.9, 0.999, 1e-8, 0.0
        u.opt_step = self.opt_step + 1
        if which == "table":
            hyp = self.geom == "hyp"
            u.rule = {"adam": N.UPD_ADAM, "rsgd": N.UPD_RSGD, "none": N.UPD_NONE}[self.update]
            u.row_mode, u.geom = self.lab_mode, N.GEOM[self.geom]
            u.hyp_rescale = int(hyp and self.update == "adam")
            u.project_shell = int(hyp and self.update == "adam")
            u.K, u.lr, u.r_in = self.K, self.lr, self.r_in
            u.table, u.n, u.D, u.ld = self.table.data_ptr(), self.n, self.D, self.ld
            u.grad_rows, u.grad_replicas, u.grad_stride = self.grad_rows.data_ptr(), self.replicas, self.n_total * self.ld
            u.state_m, u.state_v = self.opt["m"].data_ptr(), self.opt["v"].data_ptr()
            u.rows_out, u.aux_out = self.rows.data_ptr(), self.aux.data_ptr()
            u.grad_out = self.g_table.data_ptr() if self.write_grads else None
            u.loss_acc, u.loss_step = self.loss_acc.data_ptr(), self.loss.data_ptr()
        else:
            u.rule = N.UPD_NONE if self.update == "none" else N.UPD_ADAM
            u.row_mode, u.geom = N.ROWS_NONE, N.GEOM["oe"]
            u.K, u.lr, u.r_in = 0.0, self.lr_fc, 0.0
            u.table, u.n, u.D, u.ld = self.fc_flat.data_ptr(), self.n_fc, self.FC_LD, self.FC_LD
            u.grad_rows, u.grad_replicas, u.grad_stride = self.fc_grad.data_ptr(), self.fc_replicas, 0
            u.state_m, u.state_v = self.opt_fc["m"].data_ptr(), self.opt_fc["v"].data_ptr()
            u.grad_out = self.g_fc.data_ptr() if self.write_grads else None
        return u

    def step_device(self, img_sel, pos_from, pos_to, neg_to, neg_from):
        import ctypes
        lib, st = N.lib(), N.stream_ptr(self.table.device)
        m, B, n, D, ld = int(img_sel.numel()), int(pos_from.numel()), self.n, self.D, self.ld
        if m > self.max_images or B > self.max_groups:
            raise N.LecError("step of %d images / %d positives exceeds the engine's buffers" % (m, B))
        geom = N.GEOM[self.geom]
        prev_pdl = lib.lec_set_pdl(1)
        try:
            vp = ctypes.c_void_p
            p_Y, p_gY = vp(self.Y.data_ptr()), vp(self.gY.data_ptr())
            p_rows_img = vp(self.rows.data_ptr() + 4 * n * ld)
            p_aux_img = vp(self.aux.data_ptr() + 8 * 4 * n)
            p_grad_img = vp(self.grad_rows.data_ptr() + 4 * n * ld)
            N.check(lib.lec_featnet_fwd(N._p(self.features), self.features.shape[0], self.F, N._p(img_sel),
                                        img_sel.element_size(), m, N._p(self.fc_w), N._p(self.fc_b), D, p_Y, st),
                    "lec_featnet_fwd")
            if not self._rows_valid:
                # first step (or the table changed behind the engine's back): label rows, cleared label gradient and loss
                N.check(lib.lec_rows_fwd(N._p(self.table), n, D, self.lab_mode, geom, self.K, N._p(self.rows), ld,
                                         N._p(self.aux), N._p(self.grad_rows), self.replicas, self.n_total * ld,
                                         N._p(self.loss_acc), st), "lec_rows_fwd")
            N.check(lib.lec_rows_fwd(p_Y, m, D, self.img_mode, geom, self.K, p_rows_img, ld, p_aux_img,
                                     p_grad_img, self.replicas, self.n_total * ld, N._p(None), st),
                    "lec_rows_fwd")
            ev = self.kernel_events
            if ev is not None:
                ev[0].record()
            N.check(lib.lec_pairs_grouped(
                geom, self.precision, N._p(self.rows), N._p(self.aux), self.n_total, D, ld, N._p(pos_from), N._p(pos_to),
                N._p(neg_to), N._p(neg_from), pos_from.element_size(), B, self.n_neg, N._p(None), N._p(None), self.K,
                self.alpha, N._p(self.E_pos), N._p(self.E_neg), N._p(self.loss_acc), N._p(self.grad_rows), self.replicas, st),
                "lec_pairs_grouped")
            if ev is not None:
                ev[1].record()
            N.check(lib.lec_rows_bwd(p_Y, p_grad_img, self.replicas, self.n_total * ld, m, D, ld,
                                     self.img_mode, self.K, p_gY, 0, st), "lec_rows_bwd")
            N.check(lib.lec_featnet_wgrad(N._p(self.features), self.features.shape[0], self.F, N._p(img_sel),
                                          img_sel.element_size(), m, p_gY, D, N._p(self.fc_grad), self.fc_replicas,
                                          self.fc_grad.shape[1], st), "lec_featnet_wgrad")
            xcache = self.__dict__.setdefault("_xcache", {})
            for which, px in (("table", self.px), ("fc", self.px_fc)):
                u = self._update_struct(which)
                x = None
                if px is not None:
                    x = xcache.get(which)
                    if x is None:
                        x = xcache[which] = N.LecExchange()
                        px.fill(x)
                    x.slot, x.tag = px.slot_and_tag()
                N.check(lib.lec_update_rows(ctypes.byref(u), ctypes.byref(x) if x is not None else None, st), "lec_update_rows")
                if px is not None:
                    px.step += 1
        finally:
            lib.lec_set_pdl(prev_pdl)
        if self.update != "none":
            self.opt_step += 1
        self._rows_valid = True
        return self.loss

    def check_exchange(self):
        for px in (self.px, self.px_fc):
            if px is not None and int(px.error.item()) != 0:
                raise N.LecError("peer exchange timed out: a rank did not deliver its gradient; the parameter replicas "
                                 "are no longer in step -- restart from a checkpoint")

    def step_host(self, img_sel_host, index_block, B):
        """Pinned host inputs (int64 image selection, uint16/int32 index block) -> step -> loss on the host."""
        m = int(img_sel_host.numel())
        n = B * (2 + 2 * self.n_neg)
        sel = self._sel_dev[:m]
        sel.copy_(img_sel_host, non_blocking=True)
        dst = self._idx_bytes_dev[:n * index_block.dtype.itemsize].view(index_block.dtype)
        dst.copy_(index_block[:n], non_blocking=True)
        self.step_device(sel, *self._split(dst, B))
        self.loss_host.copy_(self.loss, non_blocking=True)
        torch.cuda.current_stream(self.table.device).synchronize()
        if self.px is not None:
            self.check_exchange()
        return float(self.loss_host[0])
