"""GloveEngine: host-side driver of the sm_100a kernels behind the C ABI (include/glove_b200.h).

This replaces, for the training path, what the reference builds inside ``model_fn`` + ``tf.estimator`` +
``tf.data`` [ref src/models/estimator.py:13-56, src/models/train_utils.py:13-54, src/models/data_utils.py:4-26]:

* the four Keras ``Embedding`` variables + global bias [ref src/models/model_utils.py:31-39] live in two packed
  device tables (see the header for the layout);
* ``make_csv_dataset``'s shuffle/batch is a device-resident COO + keyed on-GPU shuffle + batch plans;
* one ``session.run(train_op)`` is one ``glove_train_step``.

PyTorch is used only for device memory, streams and ``torch.distributed`` plumbing.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import os
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from ._lib import lib, check

ADAM_BETA1, ADAM_BETA2, KERAS_EPSILON = 0.9, 0.999, 1e-7


def adam_alpha_table(learning_rate: float, n_steps: int, beta1: float = ADAM_BETA1, beta2: float = ADAM_BETA2):
    """alpha[s] = lr * sqrt(1 - beta2^(s+1)) / (1 - beta1^(s+1)) in fp32 -- legacy Keras Adam._prepare_local."""
    t = np.arange(1, n_steps + 1, dtype=np.float32)
    b1p = np.power(np.float32(beta1), t).astype(np.float32)
    b2p = np.power(np.float32(beta2), t).astype(np.float32)
    return (np.float32(learning_rate) * np.sqrt(np.float32(1) - b2p).astype(np.float32)
            / (np.float32(1) - b1p)).astype(np.float32)


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class GloveEngine:
    def __init__(self, vocab_size: int, embedding_size: int = 64, *, optimizer: str = "Adam",
                 learning_rate: float = 0.001, l2_reg: float = 0.01, reg_scale: float = 2.0, neg_factor: float = 1.0,
                 head: str = "glove", adam_mode: str = "replay", batch_size: int = 1024, plan_steps: int = 16,
                 max_steps: int = 16384, device="cuda:0", dp_rank: int = 0, dp_world: int = 1, loss_cap: int = 4096,
                 dp_mode: str = "replicated"):
        if not torch.cuda.is_available():
            raise RuntimeError("GloveEngine needs a CUDA device (sm_100a); there is no CPU fallback")
        if optimizer not in _lib.OPTIMIZERS:
            raise ValueError("unsupported optimizer %r (supported: %s)" % (optimizer, sorted(_lib.OPTIMIZERS)))
        if head not in _lib.HEADS:
            raise ValueError("unsupported head %r" % head)
        if adam_mode not in _lib.ADAM_MODES:
            raise ValueError("unsupported adam_mode %r" % adam_mode)
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        self.V, self.d, self.B, self.K = int(vocab_size), int(embedding_size), int(batch_size), int(plan_steps)
        self.optimizer, self.head, self.adam_mode = optimizer, head, adam_mode
        self.learning_rate, self.l2_reg, self.reg_scale, self.neg_factor = learning_rate, l2_reg, reg_scale, neg_factor
        self.dp_rank, self.dp_world = dp_rank, dp_world
        if dp_mode not in ("replicated", "sharded"):
            raise ValueError("unsupported dp_mode %r" % dp_mode)
        # "sharded": the tables are split row-wise, rank r owns the ids with id % world == r (local row id // world)
        self.sharded = dp_mode == "sharded" and dp_world > 1
        self.V_global = int(vocab_size)
        self.V_rows = (self.V_global + dp_world - 1) // dp_world if self.sharded else self.V_global  # rows held here
        self.opt_id = _lib.OPTIMIZERS[optimizer]
        self.S = lib.glove_table_stride(self.d)
        self.P = lib.glove_table_planes(self.opt_id)
        if self.S // 4 > 128:
            raise ValueError("embedding_size %d > 510 is not supported" % self.d)
        f32 = dict(dtype=torch.float32, device=self.device)
        self.row_table = torch.empty(self.V_rows * self.P * self.S, **f32)
        self.col_table = torch.empty(self.V_rows * self.P * self.S, **f32)
        for side, t in enumerate((self.row_table, self.col_table)):
            check(lib.glove_table_init(_ptr(t), self.V_rows, self.d, self.opt_id, side, _stream()), "glove_table_init")
        self.V = self.V_rows   # every table-shaped operation below works on the rows held here
        # row-sharded tables: optional frequency-balanced owner map (balance_owners).  label = the id the kernels see
        # (owner = label % world, local row = label // world); None = identity (owner = id % world)
        self._label = None      # device int64 [V_global]: original id -> label
        self._unlabel = None    # numpy int64 [V_global]: label -> original id
        self.scalars = torch.zeros(8, dtype=torch.int32, device=self.device)
        if optimizer == "Adagrad":
            self._write_scalars(g_s0=0.1)
        self.max_steps = int(max_steps)
        self.alpha_host = adam_alpha_table(learning_rate, self.max_steps)
        self.alpha = torch.from_numpy(self.alpha_host).to(self.device)
        self.loss_cap = int(loss_cap)
        self.loss_out = torch.zeros(self.loss_cap, **f32)
        u8 = dict(dtype=torch.uint8, device=self.device)
        self.plan_bytes = lib.glove_plan_bytes(self.K, self.B)
        self.plans = [torch.empty(self.plan_bytes, **u8) for _ in range(2)]
        self.plan_first = [None, None]
        self._plan_counts = [None, None]
        self._plan_shards = [None, None]
        self._plan_need = [None, None]
        self.shard_exchange = "alltoall"
        self.prep_ws = torch.empty(lib.glove_prepare_workspace_bytes(self.K, self.B), **u8)
        self.step_ws = torch.zeros(lib.glove_step_workspace_bytes(self.B, self.d), **u8)   # must start zeroed
        self._plan_override = None
        self.coo = None
        self.nnz = 0
        self.shuffle_key = 0
        self.host_step = 0
        self.sample_idx = None  # explicit [n_steps, B] injected batch order (parity tests)
        self._args = [self._make_args(i) for i in range(2)]
        self.grad = None
        # overlap machinery: plan construction and the Adam catch-up of the NEXT step run on side streams
        self.overlap = True
        self._side = torch.cuda.Stream(device=self.device)
        self._prep_stream = torch.cuda.Stream(device=self.device)
        self._ev_step_done = [torch.cuda.Event(), torch.cuda.Event()]   # completion of step s -> slot s & 1
        self._ev_catchup = None                                         # (step, event) of the launched catch-up
        self._ev_plan = [None, None]                                    # plan buffer ready
        self._keep = [None, None]
        self._norm_cache = None
        self.last_topk_fallbacks = None
        # K steps as ONE CUDA graph launch (glove_step_graph_*): one graph per plan buffer, built on first use
        self.use_graph = False
        self._graphs = [None, None]
        self._ring = None       # shared plan construction over peer memory (enable_plan_sharing)
        self._ev_coo = None     # the COO / injected batch order are complete on the device

    def __del__(self):
        for g in getattr(self, "_graphs", [None, None]):
            if g is not None:
                try:
                    lib.glove_step_graph_destroy(g)
                except Exception:
                    pass
        self._graphs = [None, None]
        pipe = getattr(self, "_host_pipe", None)
        if pipe is not None:
            try:
                lib.glove_host_pipe_destroy(pipe)
            except Exception:
                pass
            self._host_pipe = None

    # ---- state ---------------------------------------------------------------------------------------------------
    def _write_scalars(self, **kw):
        host = self.scalars.cpu().numpy().copy()
        s = _lib.GloveScalars.from_buffer(host)
        for k, v in kw.items():
            setattr(s, k, v)
        self.scalars.copy_(torch.from_numpy(host))

    def read_scalars(self) -> Dict[str, float]:
        host = self.scalars.cpu().numpy().copy()
        s = _lib.GloveScalars.from_buffer(host)
        return {k: getattr(s, k) for k, _ in _lib.GloveScalars._fields_}

    def balance_owners(self, row, col, hot: int = 65536):
        """Row-sharded tables: replace the ``id % world`` ownership by a frequency-balanced one.  With Zipf ids the owner of
        id 0 carries ~1.45x the mean work at 8 shards; here the ``hot`` most frequent ids (by their triple counts in the
        COO ``row`` / ``col``) are dealt greedily to the least loaded owner (cost of an id = expected triples per step +
        the per-row cost of a touched row), the rest round-robin, every owner keeping exactly as many rows as before.
        Inside an owner, ids keep their order, so ties in the top-k still break towards the lower ORIGINAL id.  It is a pure
        relabelling applied at the engine boundary (COO ids in, tables / top-k ids out): no kernel sees it, and results are
        bit-identical to the unbalanced sharding (an item's arithmetic does not depend on where its row lives; the loss is
        an order-independent sum).  Must be called on every rank with the same COO, before set_coo / load_state /
        init_uniform."""
        assert self.sharded, "balance_owners is for row-sharded tables"
        N, V = self.dp_world, self.V_global
        r = torch.as_tensor(row).to(self.device).to(torch.int64)
        c = torch.as_tensor(col).to(self.device).to(torch.int64)
        freq = (torch.bincount(r, minlength=V) + torch.bincount(c, minlength=V)).cpu().numpy().astype(np.float64)
        from .parallel import balanced_labels
        label, self._unlabel, load = balanced_labels(freq, N, self.B, int(r.numel()), hot)
        self._label = torch.from_numpy(label).to(self.device)
        self._norm_cache = None
        return load                                              # relative load of the hot part per owner (diagnostics)

    def owned_ids(self) -> np.ndarray:
        """Original ids of the table rows held by this rank, in local-row order (row-sharded tables)."""
        lab = np.arange(self.dp_rank, self.V_global, self.dp_world, dtype=np.int64) if self.sharded else np.arange(self.V_global)
        return lab if self._unlabel is None else self._unlabel[lab]

    def load_state(self, R, C, rb, cb, g=0.0):
        """Inject initial tables (reference layout: R, C [V,d]; rb, cb [V]; scalar g)."""
        self._join_side()
        for side, (table, emb, bias) in enumerate(((self.row_table, R, rb), (self.col_table, C, cb))):
            emb, bias = np.asarray(emb, np.float32), np.asarray(bias, np.float32).reshape(-1)
            if self.sharded and emb.shape[0] == self.V_global:      # global arrays: keep the rows this rank owns
                emb, bias = self._local_rows(emb), self._local_rows(bias)
            e = torch.as_tensor(np.ascontiguousarray(emb, np.float32)).to(self.device)
            b = torch.as_tensor(np.ascontiguousarray(bias, np.float32).reshape(-1)).to(self.device)
            assert e.shape == (self.V, self.d) and b.shape == (self.V,)
            check(lib.glove_pack_plane(_ptr(table), self.V, self.d, self.P, 0, side, _ptr(e), _ptr(b), _stream()), "glove_pack_plane")
        self._write_scalars(g=float(g))
        torch.cuda.synchronize()

    def _local_rows(self, a):
        """Rows of a global [V, ...] array owned by this rank (owned_ids()), zero-padded to V_rows."""
        loc = a[self.owned_ids()]
        if loc.shape[0] < self.V_rows:
            pad = np.zeros((self.V_rows - loc.shape[0],) + loc.shape[1:], loc.dtype)
            loc = np.concatenate([loc, pad], 0)
        return loc

    def set_step(self, step: int):
        """Resume at a given global_step (checkpoint restore / steady-state benchmarking)."""
        self._join_side()
        self._write_scalars(step=int(step))
        self.host_step = int(step)
        self.plan_first = [None, None]
        self._ring_reset()

    def set_plane(self, side: str, plane: int, emb: torch.Tensor, bias: torch.Tensor):
        """Write optimizer slot plane ``plane`` (1 = Adam m / Adagrad acc, 2 = Adam v) of ``side`` in {'row','col'}."""
        self._join_side()
        table = self.row_table if side == "row" else self.col_table
        check(lib.glove_pack_plane(_ptr(table), self.V, self.d, self.P, plane, 0 if side == "row" else 1,
                                   _ptr(emb.contiguous()), _ptr(bias.contiguous()), _stream()), "glove_pack_plane")

    def set_last_step(self, side: str, ls: torch.Tensor):
        self._join_side()
        table = self.row_table if side == "row" else self.col_table
        ls = ls.to(device=self.device, dtype=torch.int32).contiguous()
        check(lib.glove_set_last_step(_ptr(table), self.V, self.d, self.P, 0 if side == "row" else 1, _ptr(ls), _stream()),
              "glove_set_last_step")
        torch.cuda.synchronize()

    def get_last_step(self, side: str) -> torch.Tensor:
        table = self.row_table if side == "row" else self.col_table
        out = torch.empty(self.V, dtype=torch.int32, device=self.device)
        check(lib.glove_get_last_step(_ptr(table), self.V, self.d, self.P, 0 if side == "row" else 1, _ptr(out), _stream()),
              "glove_get_last_step")
        return out

    def init_uniform(self, seed: int = 0):
        """Keras Embedding default initialiser U(-0.05, 0.05) on all four tables, global bias zero
        [ref src/models/model_utils.py:7-15,39]."""
        gen = torch.Generator(device=self.device).manual_seed(seed)
        for side, table in enumerate((self.row_table, self.col_table)):
            # the GLOBAL table is drawn (same stream on every rank) and, when sharded, only the owned rows are kept
            e = torch.empty(self.V_global, self.d, dtype=torch.float32, device=self.device).uniform_(-0.05, 0.05, generator=gen)
            b = torch.empty(self.V_global, dtype=torch.float32, device=self.device).uniform_(-0.05, 0.05, generator=gen)
            if self.sharded:
                e2 = torch.zeros(self.V, self.d, dtype=torch.float32, device=self.device)
                b2 = torch.zeros(self.V, dtype=torch.float32, device=self.device)
                ids = torch.from_numpy(self.owned_ids()).to(self.device)
                e2[: ids.numel()] = e[ids]
                b2[: ids.numel()] = b[ids]
                e, b = e2, b2
            check(lib.glove_pack_plane(_ptr(table), self.V, self.d, self.P, 0, side, _ptr(e), _ptr(b), _stream()), "glove_pack_plane")
        torch.cuda.synchronize()

    def _unpack(self, table, plane):
        e = torch.empty(self.V, self.d, dtype=torch.float32, device=self.device)
        b = torch.empty(self.V, dtype=torch.float32, device=self.device)
        side = 0 if table is self.row_table else 1
        check(lib.glove_unpack_plane(_ptr(table), self.V, self.d, self.P, plane, side, _ptr(e), _ptr(b), _stream()), "glove_unpack_plane")
        return e, b

    def get_state(self, slots: bool = False, flush: bool = True) -> Dict[str, np.ndarray]:
        """Reference-layout view of the variables (after replaying lazy Adam state up to the current step)."""
        if flush:
            self.flush()
        out = {}
        for name, bname, table in (("R", "rb", self.row_table), ("C", "cb", self.col_table)):
            e, b = self._unpack(table, 0)
            out[name], out[bname] = e.cpu().numpy(), b.cpu().numpy()
            if slots:
                for p in range(1, self.P):
                    e, b = self._unpack(table, p)
                    out["%s/s%d" % (name, p - 1)], out["%s/s%d" % (bname, p - 1)] = e.cpu().numpy(), b.cpu().numpy()
        sc = self.read_scalars()
        out["g"] = np.float32(sc["g"])
        out["step"] = sc["step"]
        if sc["error"]:
            raise _lib.GloveError("device-side error flag %d set (1: plan / step mismatch, 2: non-finite loss, 3: shard blocks "
                                  "too unbalanced for the snapshot buffer)" % sc["error"])
        return out

    def row_embeddings(self) -> torch.Tensor:
        """[V, d] device tensor of the row table (the only table the exporter / top-k uses,
        ref src/models/model_utils.py:86-95)."""
        self.flush()
        return self._unpack(self.row_table, 0)[0]

    def bias_vectors(self):
        """(row biases, col biases) of the rows held here as numpy [V] (after replaying lazy Adam state): what the
        reference's summaries histogram [ref src/models/model_utils.py:116-118]."""
        self.flush()
        out = []
        for side, t in enumerate((self.row_table, self.col_table)):
            out.append(t.view(self.V, self.P, self.S)[:, 0, self.d + side].cpu().numpy())
        return out[0], out[1]

    def _join_side(self):
        """Order the current stream after everything in flight on the side streams (catch-up, plan prefetch): required
        before the tables are read or written from outside the step sequence."""
        main = torch.cuda.current_stream()
        main.wait_stream(self._side)
        main.wait_stream(self._prep_stream)
        if self._ring is not None:
            main.wait_stream(self._ring["pull_stream"])
        self._ev_catchup = None

    def flush(self):
        self._join_side()
        if self.optimizer != "Adam" or self.adam_mode == "lazy":
            return
        fn = lib.glove_flush_lazy_state if self.adam_mode == "replay" else lib.glove_flush_lazy_state_exact
        for side, t in enumerate((self.row_table, self.col_table)):
            check(fn(_ptr(t), self.V, self.d, self.opt_id, side, _ptr(self.alpha), self.max_steps,
                     self.host_step, ADAM_BETA1, ADAM_BETA2, KERAS_EPSILON, _stream()), "glove_flush_lazy_state")
        if self.overlap and self.adam_mode in ("replay_exact", "dense"):
            # the sweep rewrites rows that the look-ahead catch-up of a later step replays too: that catch-up waits for the
            # completion event of an earlier step, so both slots are moved BEHIND the sweep
            for ev in self._ev_step_done:
                ev.record(torch.cuda.current_stream())

    # ---- input ---------------------------------------------------------------------------------------------------
    def set_coo(self, row, col, col_a, col_b, shuffle_key: int = 0):
        """Device-resident COO triple buffer.  (col_a, col_b) = (glove_value, glove_weight) for the glove head,
        (value, neg_weight) for the logistic head."""
        def dev(x, dt):
            t = torch.as_tensor(x)
            return t.to(device=self.device, dtype=dt).contiguous()
        self.coo = (dev(row, torch.int32), dev(col, torch.int32), dev(col_a, torch.float32), dev(col_b, torch.float32))
        self.nnz = int(self.coo[0].numel())
        if self.nnz and self._label is not None:       # balanced owner map: the kernels see labels (checked against V first)
            for t in self.coo[:2]:
                if int(t.min()) < 0 or int(t.max()) >= self.V_global:
                    self.coo, self.nnz = None, 0
                    raise ValueError("set_coo: ids must lie in [0, %d)" % self.V_global)
            self.coo = (self._label[self.coo[0].long()].to(torch.int32), self._label[self.coo[1].long()].to(torch.int32)) + self.coo[2:]
        if self.nnz:
            # ids index the packed tables and are packed into vbits-wide sort keys: refuse out-of-range ids here, once
            lo = int(torch.minimum(self.coo[0].min(), self.coo[1].min()))
            hi = int(torch.maximum(self.coo[0].max(), self.coo[1].max()))
            if lo < 0 or hi >= self.V_global:
                self.coo, self.nnz = None, 0
                raise ValueError("set_coo: ids must lie in [0, %d): min %d, max %d" % (self.V_global, lo, hi))
        self.shuffle_key = int(shuffle_key) & 0xFFFFFFFF
        self.plan_first = [None, None]
        self._ev_coo = torch.cuda.Event()
        self._ev_coo.record(torch.cuda.current_stream())
        self._ring_reset()

    def set_batches(self, sample_idx):
        """Inject an explicit batch order: int64 [n_steps, B] indices into the COO, used from the current step on."""
        idx = torch.as_tensor(np.ascontiguousarray(sample_idx, np.int64)).to(self.device)
        assert idx.dim() == 2 and idx.shape[1] == self.B
        self.sample_idx = idx.contiguous()
        self.sample_idx_first = self.host_step
        self.plan_first = [None, None]
        self._ev_coo = torch.cuda.Event()
        self._ev_coo.record(torch.cuda.current_stream())
        self._ring_reset()

    def _make_args(self, which):
        a = _lib.StepArgs()
        a.struct_size = ctypes.sizeof(_lib.StepArgs)
        a.row_table, a.col_table = self.row_table.data_ptr(), self.col_table.data_ptr()
        a.scalars = self.scalars.data_ptr()
        a.plan = self.plans[which].data_ptr()
        a.workspace, a.workspace_bytes = self.step_ws.data_ptr(), self.step_ws.numel()
        a.alpha, a.alpha_len = self.alpha.data_ptr(), self.max_steps
        a.loss_out, a.loss_cap = self.loss_out.data_ptr(), self.loss_cap
        a.plan_K, a.V, a.d, a.B = self.K, self.V_global, self.d, self.B
        a.n_shards, a.shard = (self.dp_world, self.dp_rank) if self.sharded else (1, 0)
        a.head, a.optimizer = _lib.HEADS[self.head], self.opt_id
        a.adam_mode = _lib.ADAM_MODES[self.adam_mode]
        a.learning_rate, a.l2_reg, a.reg_scale, a.neg_factor = self.learning_rate, self.l2_reg, self.reg_scale, self.neg_factor
        a.beta1, a.beta2, a.epsilon = ADAM_BETA1, ADAM_BETA2, KERAS_EPSILON
        a.dp_rank, a.dp_world = self.dp_rank, self.dp_world
        return a

    def prepare(self, first_step: int, which: int, dst: Optional[int] = None):
        """Build the plan for steps [first_step, first_step + K) into plan buffer ``which`` (or, with ``dst``, into the
        device address ``dst`` -- a build buffer of the shared plan construction -- leaving the buffer bookkeeping alone)."""
        assert self.coo is not None, "set_coo() first"
        sidx = None
        if self.sample_idx is not None:
            off = first_step - self.sample_idx_first
            n = self.sample_idx.shape[0]
            if off < 0 or off >= n:
                raise IndexError("no injected batches for step %d" % first_step)
            chunk = self.sample_idx[off:off + self.K]
            if chunk.shape[0] < self.K:  # pad the tail of the plan by repeating the last batch (never executed)
                chunk = torch.cat([chunk, chunk[-1:].expand(self.K - chunk.shape[0], -1)], 0)
            sidx = chunk.contiguous().view(-1)
        row, col, ca, cb = self.coo
        check(lib.glove_prepare_batches_sharded(ctypes.c_void_p(dst) if dst is not None else _ptr(self.plans[which]),
                                                _ptr(self.prep_ws), self.prep_ws.numel(),
                                                _ptr(row), _ptr(col), _ptr(ca), _ptr(cb), self.nnz, _ptr(sidx),
                                                int(first_step) * self.B, self.shuffle_key, int(first_step), self.K,
                                                self.B, self.V_global, self.dp_world if self.sharded else 1, _stream()),
              "glove_prepare_batches")
        if dst is not None:
            return sidx       # the caller keeps the index chunk alive until the stream has consumed it
        self._keep[which] = sidx  # keep the index chunk alive until the stream has consumed it
        self.plan_first[which] = first_step
        self._plan_counts[which] = None
        self._plan_shards[which] = None
        self._plan_need[which] = None
        self._ev_plan[which] = None

    def _prefetch_plan(self, step: int):
        """Build the plan of the chunk AFTER the one `step` is in, on the side stream, while this chunk trains."""
        nxt_first = (step // self.K + 1) * self.K
        which = (nxt_first // self.K) & 1
        if self.plan_first[which] == nxt_first or nxt_first >= self.max_steps:
            return
        if self.sample_idx is not None and nxt_first - self.sample_idx_first >= self.sample_idx.shape[0]:
            return
        main = torch.cuda.current_stream()
        if self._ring is not None:
            self._ring_pull_chunk(nxt_first // self.K, which)
            return
        # the buffer being overwritten belonged to the chunk before the current one: every step of it has completed
        # before the current chunk's first step was enqueued on `main`, so ordering after `main` here is sufficient
        self._prep_stream.wait_stream(main)
        with torch.cuda.stream(self._prep_stream):
            self.prepare(nxt_first, which)
            ev = torch.cuda.Event()
            ev.record(self._prep_stream)
        self._ev_plan[which] = ev

    def _plan_for(self, step: int) -> int:
        ov = self._plan_override
        if ov is not None and ov[1] <= step < ov[1] + self.K:       # a chunk planned from host buffers, any alignment
            return ov[0]
        first = (step // self.K) * self.K
        which = (step // self.K) & 1
        if self.plan_first[which] != first and self._ring is not None:
            self._ring_pull_chunk(first // self.K, which)
            torch.cuda.current_stream().wait_event(self._ev_plan[which])
        elif self.plan_first[which] != first:
            torch.cuda.current_stream().wait_stream(self._prep_stream)   # one prepare at a time (shared workspace)
            self.prepare(first, which)
            ev = torch.cuda.Event()                                     # the catch-up stream reads the plan too
            ev.record(torch.cuda.current_stream())
            self._ev_plan[which] = ev
        elif self._ev_plan[which] is not None:      # built on the side stream: order the consumer after it
            torch.cuda.current_stream().wait_event(self._ev_plan[which])   # (kept: the catch-up stream waits on it too)
        return which

    def _before_step(self, which):
        """Overlap hooks run before step `host_step` is enqueued: (1) start the catch-up of step+1 on the side stream
        (it only needs step-1 to have finished), (2) make this step wait for its own catch-up, (3) prefetch the next plan."""
        s = self.host_step
        if not self.overlap:
            return
        main = torch.cuda.current_stream()
        if self._ev_catchup is not None and self._ev_catchup[0] == s:
            main.wait_event(self._ev_catchup[1])
        self._ev_catchup = None
        k_next = s + 1 - self.plan_first[which] if self.plan_first[which] is not None else 0
        if (self.optimizer == "Adam" and self.adam_mode in ("replay_exact", "dense") and 0 < k_next < self.K
                and s + 1 < self.max_steps and s >= 1):
            self._side.wait_event(self._ev_step_done[(s - 1) & 1])
            if self._ev_plan[which] is not None:                        # ... and not before its plan is complete
                self._side.wait_event(self._ev_plan[which])
            check(lib.glove_catchup_step(ctypes.byref(self._args[which]), s + 1, ctypes.c_void_p(self._side.cuda_stream)),
                  "glove_catchup_step")
            ev = torch.cuda.Event()
            ev.record(self._side)
            self._ev_catchup = (s + 1, ev)
        if s % self.K == 0 and self._plan_override is None:
            self._prefetch_plan(s)

    def _after_step(self):
        if self.overlap:
            self._ev_step_done[self.host_step & 1].record(torch.cuda.current_stream())

    def _dense_flush(self):
        """adam_mode == 'dense' (the literal dense sweep): bring every row up to date after the step that has just been
        counted.  The sweep rewrites rows that the catch-up of a later step may replay, so the step's completion event --
        what that catch-up waits for -- is recorded again BEHIND the sweep (a host that runs ahead of the device would
        otherwise let the two overlap)."""
        if self.adam_mode != "dense":
            return
        self.flush()
        if self.overlap:
            self._ev_step_done[(self.host_step - 1) & 1].record(torch.cuda.current_stream())

    # ---- shared plan construction (row-sharded tables over peer memory) ------------------------------------------------
    # Every rank of a row-sharded job needs the plan of the GLOBAL batch but dereferences only the ~1/world of it that
    # describes its own segments, and building it (two radix sorts + ~30 passes over K * B_global elements) costs as much as
    # the steps themselves from 4 GPUs on.  With plan sharing the chunks are dealt round-robin: in "round" R (chunks
    # R*world .. R*world + world - 1) rank q builds ONLY chunk R*world + q, into one of two build buffers in symmetric
    # memory, a whole round ahead of its use and at the same time as every other rank builds its own; when the round
    # opens (one barrier over the peer-mapped signal pads, off the step stream) every rank copies its slice of each chunk
    # out of the builder's buffer over NVLink (glove_plan_pull_slice) into its local double-buffered plans.  Per rank and
    # step the construction cost is that of ONE GPU's batch, whatever the world size.
    #   build stream:  [wait: last barrier -- everyone has left the buffer]  prepare(my chunk of round R+1) -> built[R+1]
    #   pull stream:   [wait: built[R]]  barrier  | per chunk: [wait: steps of chunk c-2 done]  pull slice -> plan ready
    def enable_plan_sharing(self, group=None, _emulate=None):
        """Collective (call on every rank, after enable_peer_gather): allocates the two build buffers in symmetric memory and
        switches plan construction to the shared scheme.  ``_emulate`` = (peer base pointers, barrier callable) lets N
        engines on ONE GPU stand in for N ranks (tests)."""
        assert self.sharded, "plan sharing is for row-sharded tables"
        self._join_side()
        torch.cuda.synchronize()
        if _emulate is None:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem
            buf = symm_mem.empty(2 * self.plan_bytes, dtype=torch.uint8, device=self.device)
            hdl = symm_mem.rendezvous(buf, group if group is not None else dist.group.WORLD)
            ptrs, barrier = [int(p) for p in hdl.buffer_ptrs], hdl.barrier
        else:
            buf = torch.empty(2 * self.plan_bytes, dtype=torch.uint8, device=self.device)
            hdl, (ptrs, barrier) = None, _emulate
        self._ring = dict(buf=buf, hdl=hdl, ptrs=ptrs, barrier=barrier, built={}, opened=set(), ev_barrier=None, keep={},
                          build_stream=torch.cuda.Stream(device=self.device), pull_stream=torch.cuda.Stream(device=self.device),
                          builder=self._ring_build_resident)
        self.plan_first = [None, None]
        torch.cuda.synchronize()
        if _emulate is None:
            barrier()
            torch.cuda.synchronize()

    def _ring_reset(self):
        """Forget every built / opened round (the batch order changed).  A peer may still be copying out of this rank's build
        buffers: nothing is rebuilt before every rank has passed the barrier enqueued here."""
        ring = self._ring
        if ring is None:
            return
        ring["built"].clear(); ring["opened"].clear(); ring["keep"].clear()
        ps = ring["pull_stream"]
        ps.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(ps):
            ring["barrier"]()
            ring["ev_barrier"] = torch.cuda.Event()
            ring["ev_barrier"].record(ps)

    def _ring_build_resident(self, R, dst):
        """builder of the device-resident COO: my chunk of round R (steps [c*K, (c+1)*K), c = R*world + rank)"""
        first = (R * self.dp_world + self.dp_rank) * self.K
        if first >= self.max_steps:
            return None
        if self.sample_idx is not None and not 0 <= first - self.sample_idx_first < self.sample_idx.shape[0]:
            return None
        return self.prepare(first, 0, dst=dst)

    def _ring_build(self, R):
        ring = self._ring
        if R in ring["built"]:
            return
        bs = ring["build_stream"]
        if self._ev_coo is not None:
            bs.wait_event(self._ev_coo)
        if ring["ev_barrier"] is not None:      # every rank has finished copying out of the buffer this build overwrites
            bs.wait_event(ring["ev_barrier"])
        with torch.cuda.stream(bs):
            ring["keep"][R & 1] = ring["builder"](R, ring["buf"].data_ptr() + (R & 1) * self.plan_bytes)
            ev = torch.cuda.Event()
            ev.record(bs)
        ring["built"][R] = ev
        for r in [r for r in ring["built"] if r != R and (r & 1) == (R & 1)]:   # the buffer held another round: gone
            del ring["built"][r]
            ring["opened"].discard(r)

    def _ring_open(self, R):
        ring = self._ring
        if R in ring["opened"]:
            return
        if R not in ring["built"]:
            # cold start, or a round out of order (a plan of earlier steps asked for again): its build overwrites a buffer
            # that a peer may still be copying a later chunk from -- start over behind a barrier
            self._ring_reset()
        self._ring_build(R)                      # normally a no-op: built one round ago
        ps = ring["pull_stream"]
        ps.wait_event(ring["built"][R])
        with torch.cuda.stream(ps):
            ring["barrier"]()                    # every rank's chunk of round R is complete ...
            ring["ev_barrier"] = torch.cuda.Event()
            ring["ev_barrier"].record(ps)        # ... and nobody reads the buffers of round R-1 any more
        ring["opened"].add(R)
        ring["opened"].discard(R - 2)
        self._ring_build(R + 1)                  # look-ahead: a whole round of training hides it

    def _ring_pull(self, R, j, which, first_step, after=None):
        """Copy this rank's slice of chunk j of round R (built by rank j) into plan buffer ``which``."""
        ring = self._ring
        self._ring_open(R)
        ps = ring["pull_stream"]
        if after is not None:
            ps.wait_event(after)                 # the steps that read plan buffer `which` before have finished
        with torch.cuda.stream(ps):
            src = ring["ptrs"][j] + (R & 1) * self.plan_bytes
            check(lib.glove_plan_pull_slice(_ptr(self.plans[which]), ctypes.c_void_p(src), self.K, self.B, self.dp_world,
                                            self.dp_rank, ctypes.c_void_p(ps.cuda_stream)), "glove_plan_pull_slice")
            ev = torch.cuda.Event()
            ev.record(ps)
        self.plan_first[which] = first_step
        self._plan_counts[which] = self._plan_shards[which] = self._plan_need[which] = None
        self._ev_plan[which] = ev
        return ev

    def _ring_pull_chunk(self, c, which):
        """device-resident COO: chunk c = steps [c*K, (c+1)*K) of the keyed shuffle / the injected batch order"""
        # plan buffer `which` belonged to chunk c-2, whose steps were all enqueued before this call
        from .parallel import shared_plan_slot
        self._ring["pull_stream"].wait_stream(torch.cuda.current_stream())
        R, builder, _ = shared_plan_slot(c, self.dp_world)
        self._ring_pull(R, builder, which, c * self.K)

    # ---- train ---------------------------------------------------------------------------------------------------
    def step(self):
        """One TRAIN step (``session.run(train_op)`` in the reference).  Asynchronous; the loss lands in
        ``loss_out[step % loss_cap]``."""
        if self.host_step >= self.max_steps:
            raise RuntimeError("max_steps exhausted; construct the engine with a larger max_steps")
        if self.sharded:
            self._step_sharded()
            return
        which = self._plan_for(self.host_step)
        self._before_step(which)
        if self.dp_world > 1:
            self._step_dp(which)
            return
        check(lib.glove_train_step(ctypes.byref(self._args[which]), _stream()), "glove_train_step")
        self._after_step()
        self.host_step += 1
        self._dense_flush()

    def step_chunk_graph(self) -> int:
        """The K steps of the plan chunk that starts at the current step as ONE CUDA graph launch (captured once per plan
        buffer, valid for every later chunk that buffer serves).  Returns the number of steps enqueued (K), or 0 when the
        graph path does not apply here (not at a chunk boundary, fewer than K steps left, data-parallel modes whose steps
        need host-side collectives -- everything but 'peer-sync' sharding --, exact-replay modes that interleave other
        streams with the steps): the caller then falls back to ``step()``."""
        s = self.host_step
        shard_ok = self.sharded and self.shard_exchange in ("peer-sync", "peer-push")
        if (s % self.K or s + self.K > self.max_steps or (self.dp_world > 1 and not shard_ok) or self._plan_override is not None
                or self.adam_mode in ("replay_exact", "dense")):
            return 0
        if self.sample_idx is not None and s + self.K - self.sample_idx_first > self.sample_idx.shape[0]:
            return 0
        which = self._plan_for(s)
        self._ev_catchup = None
        if self.overlap:
            self._prefetch_plan(s)
        if self._graphs[which] is None:
            g = ctypes.c_void_p(0)
            check(lib.glove_step_graph_create(ctypes.byref(self._args[which]), self.K, ctypes.byref(g)), "glove_step_graph_create")
            self._graphs[which] = g
        check(lib.glove_step_graph_launch(self._graphs[which], _stream()), "glove_step_graph_launch")
        self.host_step += self.K
        if self.overlap:   # both completion slots: whichever parity a later catch-up asks about, the chunk has finished
            self._ev_step_done[0].record(torch.cuda.current_stream())
            self._ev_step_done[1].record(torch.cuda.current_stream())
        return self.K

    def grad_step(self):
        """Data-parallel half-step 1: this rank's gradient partial sums for every global segment (dense, slot order).
        Returns (grad_rows, grad_cols, grad_scalars) device tensors to be all-reduced."""
        which = self._plan_for(self.host_step)
        gr, gc, gs = self._grad_buffers()
        check(lib.glove_grad_step(ctypes.byref(self._args[which]), _ptr(gr), _ptr(gc), _ptr(gs), _stream()), "glove_grad_step")
        return gr, gc, gs

    def _grad_buffers(self):
        """One contiguous buffer [scalars(4, padded to 8) | rows B*S | cols B*S] so that a step needs ONE collective when
        the touched slots of both sides are packed next to each other (see _step_dp)."""
        if self.grad is None:
            self._grad_flat = torch.zeros(8 + 2 * self.B * self.S, dtype=torch.float32, device=self.device)
            n = self.B * self.S
            self.grad = (self._grad_flat[8:8 + n], self._grad_flat[8 + n:8 + 2 * n], self._grad_flat[0:4])
        return self.grad

    def apply_step(self):
        """Data-parallel half-step 2: apply the optimizer on every replica from the all-reduced buffers."""
        which = self._plan_for(self.host_step)
        gr, gc, gs = self.grad
        check(lib.glove_apply_step(ctypes.byref(self._args[which]), _ptr(gr), _ptr(gc), _ptr(gs), _stream()), "glove_apply_step")
        self._after_step()
        self.host_step += 1
        self._dense_flush()

    # ---- row-sharded data parallel (cfg4): owner-computes ------------------------------------------------------------
    def _shard_info(self, step):
        """(first owned slot per shard [2][world+1], padded block size [2]) of the batch of `step` (host copy, cached)."""
        which = self._plan_for(step)
        if self._plan_shards[which] is None:
            out = (ctypes.c_int32 * 20)()
            infos = []
            for k in range(self.K):
                check(lib.glove_plan_shard_info(_ptr(self.plans[which]), self.K, self.B, k, out, _stream()), "glove_plan_shard_info")
                infos.append(([list(out[0:9]), list(out[10:19])], [out[9], out[19]]))
            self._plan_shards[which] = infos
        return self._plan_shards[which][step - self.plan_first[which]]

    def snapshot_view(self, side: int) -> torch.Tensor:
        """float32 [snapshot_rows, S] view of the step workspace's snapshot of `side`."""
        rows = lib.glove_step_snapshot_rows(self.B)
        off = lib.glove_step_snapshot_offset(self.B, self.d, side)
        return self.step_ws[off: off + rows * self.S * 4].view(torch.float32).view(rows, self.S)

    def _shard_scalars(self):
        if getattr(self, "_sscal", None) is None:
            self._sscal = torch.zeros(4, dtype=torch.float32, device=self.device)
        return self._sscal

    def shard_stage(self):
        which = self._plan_for(self.host_step)
        self._before_step(which)
        own, upad = self._shard_info(self.host_step)
        if self.dp_world * max(upad) > lib.glove_step_snapshot_rows(self.B):
            raise _lib.GloveError("shard blocks too unbalanced for the snapshot buffer (%d x %d rows)" % (self.dp_world, max(upad)))
        check(lib.glove_shard_stage_step(ctypes.byref(self._args[which]), _stream()), "glove_shard_stage_step")
        return upad

    def set_peer_workspaces(self, ptrs, direct: bool = False, sync: bool = False, push: bool = False):
        """Row-sharded tables over peer memory: ``ptrs[r]`` = base of rank r's step workspace as mapped in THIS process.
        From now on the requested snapshot rows are pulled from their owners by one kernel (``shard_exchange='peer'``) or,
        with ``direct``, read by the update kernel itself while it computes (``'peer-direct'``); no NCCL data movement.
        ``sync`` (``'peer-sync'``): the pull variant with the step's two synchronisation points done on the device through
        the same peer memory (epoch flags + the loss sums): no barrier, no all-reduce, one C call (or one graph node
        sequence) per step."""
        arr = (ctypes.c_void_p * len(ptrs))(*[int(p) for p in ptrs])
        check(lib.glove_shard_set_peers(ctypes.byref(self._args[0]), arr, len(ptrs), _stream()), "glove_shard_set_peers")
        # 'peer-push' (the stage kernel writes each row straight into the snapshots of the shards that read it; needs the
        # closed-form Adam stage) falls back to the pull for the other optimizers
        push = push and self.optimizer == "Adam" and self.adam_mode == "replay"
        for a in self._args:
            a.peer_gather = 1 if direct else (4 if push else 3 if sync else 2)
        self.shard_exchange = "peer-direct" if direct else ("peer-push" if push else "peer-sync" if sync else "peer")

    def shard_wait_staged(self):
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_wait_staged(ctypes.byref(self._args[which]), _stream()), "glove_shard_wait_staged")

    def shard_signal_staged(self):
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_signal_staged(ctypes.byref(self._args[which]), _stream()), "glove_shard_signal_staged")

    def shard_finish_sync(self):
        """peer-sync: announce this rank's loss sums, wait for every peer's, finish the step (device-side all-reduce)."""
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_finish_sync(ctypes.byref(self._args[which]), _ptr(self._shard_scalars()), _stream()), "glove_shard_finish_sync")
        self._after_step()
        self.host_step += 1

    def shard_pull(self):
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_pull_step(ctypes.byref(self._args[which]), _stream()), "glove_shard_pull_step")

    def enable_peer_gather(self, group=None, direct: bool = False, sync: bool = False, push: bool = False):
        """Collective: moves the step workspace into symmetric (peer-mapped) memory and registers every rank's mapping."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        assert self.sharded, "peer gather is the exchange of the row-sharded scheme"
        self._join_side()
        torch.cuda.synchronize()
        ws = symm_mem.empty(self.step_ws.numel(), dtype=torch.uint8, device=self.device)
        ws.zero_()                                                     # the step workspace must start zeroed
        self._symm = symm_mem.rendezvous(ws, group if group is not None else dist.group.WORLD)
        self.step_ws = ws
        self._args = [self._make_args(i) for i in range(2)]
        self.set_peer_workspaces(list(self._symm.buffer_ptrs), direct, sync or push, push)
        torch.cuda.synchronize()
        self._symm.barrier()

    def shard_update(self):
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_update_step(ctypes.byref(self._args[which]), _ptr(self._shard_scalars()), _stream()), "glove_shard_update_step")

    def shard_finish(self):
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_finish_step(ctypes.byref(self._args[which]), _ptr(self._shard_scalars()), _stream()), "glove_shard_finish_step")
        self._after_step()
        self.host_step += 1
        self._dense_flush()

    def _need_counts(self, step):
        """(rows to send to each peer, rows to receive from each owner) of the request-only exchange of `step`."""
        which = self._plan_for(step)
        if self._plan_need[which] is None:
            out = (ctypes.c_int32 * (2 * self.K * 8 * 9))()
            check(lib.glove_plan_need_info(_ptr(self.plans[which]), self.K, self.B, out, _stream()), "glove_plan_need_info")
            self._plan_need[which] = np.ctypeslib.as_array(out).reshape(2, self.K, 8, 9).copy()
        need = self._plan_need[which][:, step - self.plan_first[which]]      # [side][requester][owner]
        N, me = self.dp_world, self.dp_rank
        send = [int(sum(need[s][r][me + 1] - need[s][r][me] for s in (0, 1))) for r in range(N)]
        recv = [int(sum(need[s][me][q + 1] - need[s][me][q] for s in (0, 1))) for q in range(N)]
        if min(send) < 0 or min(recv) < 0:
            raise _lib.GloveError("corrupt request lists in the plan")
        return send, recv

    def shard_pack(self):
        if getattr(self, "_xbuf", None) is None:
            rows = 2 * lib.glove_step_snapshot_rows(self.B)
            self._xbuf = [torch.empty(rows, self.S, dtype=torch.float32, device=self.device) for _ in range(2)]  # send, recv
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_pack_step(ctypes.byref(self._args[which]), _ptr(self._xbuf[0]), _stream()), "glove_shard_pack_step")
        return self._need_counts(self.host_step)

    def shard_unpack(self):
        which = self._plan_for(self.host_step)
        check(lib.glove_shard_unpack_step(ctypes.byref(self._args[which]), _ptr(self._xbuf[1]), _stream()), "glove_shard_unpack_step")

    def _step_sharded(self):
        """Owner-computes: stage own rows -> exchange snapshot rows -> fused update of the own segments (in place) ->
        all-reduce of the 3 loss scalars -> finish.  No gradient exchange.  `shard_exchange`:
        'alltoall' (default) sends every owner's rows only to the shards whose work items need them (request lists from the
        plan, one all_to_all_single with uneven splits); 'allgather' sends every block to everyone (equal-sized native);
        'peer' (after enable_peer_gather) moves nothing ahead of time: the update kernel reads remote rows over NVLink."""
        import torch.distributed as dist
        if self.shard_exchange in ("peer-sync", "peer-push"):
            # the whole step is device work: stage -> announce -> pull (waits owner by owner) -> update -> announce + wait +
            # finish, with flags and loss sums exchanged through the peer-mapped workspaces
            # (padded owner blocks that do not fit the snapshot are refused by the kernels themselves -- error flag 3, the step
            # counter stops -- so the host does not read the block sizes back, which would drain the stream once per chunk)
            which = self._plan_for(self.host_step)
            self._before_step(which)
            check(lib.glove_shard_train_step(ctypes.byref(self._args[which]), _stream()), "glove_shard_train_step")
            self._after_step()
            self.host_step += 1
            return
        upad = self.shard_stage()
        N, r = self.dp_world, self.dp_rank
        if self.shard_exchange in ("peer", "peer-direct"):
            # no NCCL data movement: once every rank has staged its rows (barrier), one kernel pulls the requested rows
            # from their owners' snapshots over NVLink ('peer'), or the update kernel reads them there while it computes
            # ('peer-direct'); the all-reduce below keeps the next stage from overwriting a block that a peer still reads
            self._symm.barrier()
            if self.shard_exchange == "peer":
                self.shard_pull()
        elif self.shard_exchange == "alltoall":
            send, recv = self.shard_pack()
            dist.all_to_all_single(self._xbuf[1][: sum(recv)], self._xbuf[0][: sum(send)], recv, send)
            self.shard_unpack()
        else:
            for side in (0, 1):
                snap, u = self.snapshot_view(side), upad[side]
                if u:
                    dist.all_gather_into_tensor(snap[: N * u], snap[r * u:(r + 1) * u])   # in place (send = recv + rank*count)
        self.shard_update()
        dist.all_reduce(self._shard_scalars())
        self.shard_finish()

    def _step_dp(self, which):
        import torch.distributed as dist
        gr, gc, gs = self.grad_step()
        # exchange only the touched rows: the buffers are dense in slot order and the per-batch segment counts of the
        # whole plan were fetched once when the plan was built
        n_r, n_c = self._counts_for(self.host_step)
        # [scalars | touched row slots] is contiguous; the touched col slots follow B*S later: two collectives per step
        dist.all_reduce(self._grad_flat[: 8 + n_r * self.S])
        dist.all_reduce(gc[: n_c * self.S])
        self.apply_step()

    def _counts_for(self, step):
        which = self._plan_for(step)
        if self._plan_counts[which] is None:
            out = (ctypes.c_int32 * 4)()
            counts = []
            for k in range(self.K):
                check(lib.glove_plan_batch_counts(_ptr(self.plans[which]), self.K, self.B, k, out, _stream()), "glove_plan_batch_counts")
                counts.append((out[0], out[1]))
            self._plan_counts[which] = counts
        return self._plan_counts[which][step - self.plan_first[which]]

    def step_profiled(self):
        """One TRAIN step with per-kernel device timings (ms): (stage, update, 0).  Synchronises."""
        self._join_side()
        which = self._plan_for(self.host_step)
        ms = (ctypes.c_float * 3)()
        check(lib.glove_train_step_profiled(ctypes.byref(self._args[which]), _stream(), ms), "glove_train_step_profiled")
        self._after_step()
        self.host_step += 1
        self._dense_flush()
        return tuple(ms)

    def train_steps_host(self, host_row, host_col, host_a, host_b, host_losses):
        """End-to-end boundary: n * plan_steps TRAIN steps on the explicit triples held in HOST (pinned) tensors
        (numel = steps * B); H2D copies, plan builds, steps and the D2H loss read all happen inside ONE C-ABI call
        (glove_train_steps_host), pipelined chunk against chunk."""
        if getattr(self, "_host_staging", None) is None:
            pipe = ctypes.c_void_p(0)
            check(lib.glove_host_pipe_create(ctypes.byref(pipe)), "glove_host_pipe_create")
            self._host_pipe = pipe
            self._host_staging = torch.empty(lib.glove_host_staging_bytes(self.K, self.B), dtype=torch.uint8, device=self.device)
            self._host_plans = torch.empty(lib.glove_host_plan_bytes(self.K, self.B), dtype=torch.uint8, device=self.device)
        steps = host_row.numel() // self.B
        assert steps * self.B == host_row.numel() and steps % self.K == 0 and not host_row.is_cuda
        assert host_losses.numel() >= steps
        self._join_side()
        check(lib.glove_train_steps_host(self._host_pipe, ctypes.byref(self._args[0]), _ptr(self._host_plans), _ptr(self.prep_ws),
                                         self.prep_ws.numel(), _ptr(self._host_staging), self._host_staging.numel(),
                                         _ptr(host_row), _ptr(host_col), _ptr(host_a), _ptr(host_b), steps,
                                         _ptr(host_losses), _stream()), "glove_train_steps_host")
        self.host_step += steps
        self.plan_first = [None, None]
        if self.overlap:   # both completion slots (see step_chunk_graph): a later catch-up waits on a current event
            self._ev_step_done[0].record(torch.cuda.current_stream())
            self._ev_step_done[1].record(torch.cuda.current_stream())

    def train_chunk_from_host(self, host_row, host_col, host_a, host_b):
        """One chunk of K*B explicit triples from pinned HOST tensors (see train_chunks_from_host)."""
        return self.train_chunks_from_host([(host_row, host_col, host_a, host_b)])

    def train_chunks_from_host(self, chunks, sliced: bool = False):
        """End-to-end path for any world size (data-parallel aware): every chunk is K*B explicit triples in pinned HOST
        tensors (row, col, colA, colB); it is copied to a device staging COO, planned in file order and trained for K
        steps.  The copy + plan of chunk c+1 run on the side stream while the steps of chunk c run (two plan buffers, two
        staging sets).  Returns the losses of all steps (numpy; synchronises).  At world size 1 prefer train_steps_host
        (the same pipeline behind one C-ABI call).

        ``sliced`` (world > 1): every rank feeds only ITS share of each batch -- chunk tensors of K * B / world elements,
        laid out [K][B / world], the triples [rank * B / world, (rank + 1) * B / world) of every step -- and the ranks
        all-gather the chunk on the device (one NCCL all-gather per chunk on its own communicator, off the step stream):
        1 / world of the bytes cross each rank's PCIe link instead of the whole global batch."""
        n = self.K * self.B
        N = self.dp_world if sliced else 1
        if sliced and N > 1 and self._ring is not None and self._ring["hdl"] is not None and len(chunks) % N == 0:
            return self._train_chunks_shared_plans(chunks)
        if self._ring is not None:
            self._ring_reset()      # the build buffers are about to be bypassed: plans of the resident COO are rebuilt afterwards
        if sliced and N > 1:
            import torch.distributed as dist
            assert self.B % N == 0
            if getattr(self, "_gather_group", None) is None:
                self._gather_group = dist.new_group(backend="nccl") if dist.get_backend() == "nccl" else dist.group.WORLD
                self._slice_buf = [torch.empty(4 * (n // N), dtype=torch.int32, device=self.device) for _ in range(2)]
                self._gather_buf = torch.empty(N * 4 * (n // N), dtype=torch.int32, device=self.device)
        self._join_side()
        if getattr(self, "_stage_coo", None) is None:
            i32 = dict(dtype=torch.int32, device=self.device)
            f32 = dict(dtype=torch.float32, device=self.device)
            self._stage_coo = [(torch.empty(n, **i32), torch.empty(n, **i32), torch.empty(n, **f32), torch.empty(n, **f32))
                               for _ in range(2)]
            self._stage_idx = torch.arange(n, dtype=torch.int64, device=self.device)
        first0 = self.host_step
        main = torch.cuda.current_stream()
        ready, done = [None, None], [None, None]
        self._prep_stream.wait_stream(main)          # earlier steps may still read the plan buffers

        def stage(c):
            which = c & 1
            with torch.cuda.stream(self._prep_stream):
                if done[which] is not None:           # plan + staging set `which` belonged to chunk c-2
                    self._prep_stream.wait_event(done[which])
                if sliced and N > 1:
                    import torch.distributed as dist
                    m = n // N
                    sl = self._slice_buf[which]
                    for j, src in enumerate(chunks[c]):           # H2D of this rank's share only
                        assert src.numel() == m and not src.is_cuda
                        sl[j * m:(j + 1) * m].copy_(src.view(torch.int32), non_blocking=True)
                    dist.all_gather_into_tensor(self._gather_buf, sl, group=self._gather_group)
                    from .parallel import assemble_chunk
                    g = assemble_chunk(self._gather_buf, N, self.K, self.B // N)          # [array][step][rank][triple]
                    for j, dst in enumerate(self._stage_coo[which]):
                        dst.view(torch.int32).view(self.K, N, self.B // N).copy_(g[j])
                else:
                    for dst, src in zip(self._stage_coo[which], chunks[c]):
                        assert src.numel() == n and not src.is_cuda
                        dst.copy_(src, non_blocking=True)
                row, col, ca, cb = self._stage_coo[which]
                if self._label is not None:                        # balanced owner map: the kernels see labels
                    row.copy_(self._label[row.long()]); col.copy_(self._label[col.long()])
                check(lib.glove_prepare_batches_sharded(_ptr(self.plans[which]), _ptr(self.prep_ws), self.prep_ws.numel(),
                                                        _ptr(row), _ptr(col), _ptr(ca), _ptr(cb), n, _ptr(self._stage_idx), 0, 0,
                                                        first0 + c * self.K, self.K, self.B, self.V_global,
                                                        self.dp_world if self.sharded else 1,
                                                        ctypes.c_void_p(self._prep_stream.cuda_stream)), "glove_prepare_batches")
                ready[which] = torch.cuda.Event()
                ready[which].record(self._prep_stream)

        stage(0)
        for c in range(len(chunks)):
            if c + 1 < len(chunks):
                stage(c + 1)
            which, first = c & 1, first0 + c * self.K
            main.wait_event(ready[which])
            self._plan_counts[which] = self._plan_shards[which] = self._plan_need[which] = None
            self._ev_plan[which] = ready[which]
            self.plan_first = [None, None]
            self.plan_first[which] = first
            self._plan_override = (which, first)
            a = self._args[which]
            for _ in range(self.K):
                if self.sharded:
                    self._step_sharded()
                    continue
                if self.dp_world > 1:
                    import torch.distributed as dist
                    gr, gc, gs = self._grad_buffers()
                    check(lib.glove_grad_step(ctypes.byref(a), _ptr(gr), _ptr(gc), _ptr(gs), _stream()), "glove_grad_step")
                    dist.all_reduce(gr); dist.all_reduce(gc); dist.all_reduce(gs)
                    check(lib.glove_apply_step(ctypes.byref(a), _ptr(gr), _ptr(gc), _ptr(gs), _stream()), "glove_apply_step")
                else:
                    self._before_step(which)
                    check(lib.glove_train_step(ctypes.byref(a), _stream()), "glove_train_step")
                    self._after_step()
                self.host_step += 1
            done[which] = torch.cuda.Event()
            done[which].record(main)
        self._plan_override = None
        self.plan_first = [None, None]
        main.wait_stream(self._prep_stream)
        idx = torch.arange(first0, first0 + len(chunks) * self.K, device=self.device) % self.loss_cap
        return self.loss_out[idx].cpu().numpy()      # D2H of the losses (synchronises)

    def _train_chunks_shared_plans(self, chunks):
        """train_chunks_from_host(sliced=True) with shared plan construction: the chunks are taken in rounds of `world`; of
        every round each rank copies its shares of all chunks to the device, ONE all-to-all hands rank q every share of
        chunk q (instead of all-gathering every chunk to everyone), rank q plans that chunk alone, and the ranks pull their
        slices of the plans as the steps reach them.  Copies, exchange and planning of round R+1 run under the steps of
        round R."""
        import torch.distributed as dist
        from .parallel import assemble_chunk
        ring, N, K, me = self._ring, self.dp_world, self.K, self.dp_rank
        assert self.B % N == 0
        n, m = K * self.B, K * self.B // N
        self._join_side()
        if getattr(self, "_gather_group", None) is None:
            self._gather_group = dist.new_group(backend="nccl") if dist.get_backend() == "nccl" else dist.group.WORLD
        if getattr(self, "_ring_io", None) is None:
            i32 = dict(dtype=torch.int32, device=self.device)
            self._ring_io = [(torch.empty(N * 4 * m, **i32), torch.empty(N * 4 * m, **i32)) for _ in range(2)]   # send, recv
            self._ring_coo = [tuple(torch.empty(n, dtype=dt, device=self.device) for dt in (torch.int32, torch.int32, torch.float32, torch.float32))
                              for _ in range(2)]
            self._stage_idx = torch.arange(n, dtype=torch.int64, device=self.device)
        first0 = self.host_step
        main = torch.cuda.current_stream()
        self._ring_reset()

        def build(R, dst):
            if R * N >= len(chunks):
                return None
            send, recv = self._ring_io[R & 1]
            sv = send.view(N, 4, m)
            for q in range(N):                                     # H2D of this rank's share of every chunk of the round
                for j, src in enumerate(chunks[R * N + q]):
                    assert src.numel() == m and not src.is_cuda
                    sv[q, j].copy_(src.view(torch.int32), non_blocking=True)
            dist.all_to_all_single(recv, send, group=self._gather_group)    # rank q receives every rank's share of chunk q
            g = assemble_chunk(recv, N, K, self.B // N)            # [array][step][rank][triple]
            coo = self._ring_coo[R & 1]
            for j, t in enumerate(coo):
                t.view(torch.int32).view(K, N, self.B // N).copy_(g[j])
            row, col, ca, cb = coo
            if self._label is not None:                            # balanced owner map: the kernels see labels
                row.copy_(self._label[row.long()]); col.copy_(self._label[col.long()])
            check(lib.glove_prepare_batches_sharded(ctypes.c_void_p(dst), _ptr(self.prep_ws), self.prep_ws.numel(), _ptr(row), _ptr(col),
                                                    _ptr(ca), _ptr(cb), n, _ptr(self._stage_idx), 0, 0, first0 + (R * N + me) * K, K,
                                                    self.B, self.V_global, N, _stream()), "glove_prepare_batches")
            return None

        ring["builder"] = build
        ready, done = [None, None], [None, None]
        ring["pull_stream"].wait_stream(main)            # earlier steps may still read the plan buffers

        def pull(c):
            ready[c & 1] = self._ring_pull(c // N, c % N, c & 1, first0 + c * K, after=done[c & 1])

        try:
            pull(0)
            for c in range(len(chunks)):
                if c + 1 < len(chunks):
                    pull(c + 1)
                which, first = c & 1, first0 + c * K
                main.wait_event(ready[which])
                self.plan_first = [None, None]
                self.plan_first[which] = first
                self._plan_override = (which, first)
                for _ in range(K):
                    self._step_sharded()
                done[which] = torch.cuda.Event()
                done[which].record(main)
        finally:
            self._plan_override = None
            self.plan_first = [None, None]
            ring["builder"] = self._ring_build_resident
        main.wait_stream(ring["pull_stream"])
        main.wait_stream(ring["build_stream"])
        self._ring_reset()
        idx = torch.arange(first0, first0 + len(chunks) * K, device=self.device) % self.loss_cap
        return self.loss_out[idx].cpu().numpy()      # D2H of the losses (synchronises)

    def batch_counts(self, step: int):
        which = self._plan_for(step)
        out = (ctypes.c_int32 * 4)()
        check(lib.glove_plan_batch_counts(_ptr(self.plans[which]), self.K, self.B, step - self.plan_first[which], out,
                                          _stream()), "glove_plan_batch_counts")
        return tuple(out)

    def train(self, n_steps: int):
        """Run n_steps; returns their losses as a numpy array (synchronises)."""
        start = self.host_step
        losses = []
        done = 0
        while done < n_steps:
            chunk = min(n_steps - done, self.loss_cap)
            left = chunk
            while left:
                k = self.step_chunk_graph() if (self.use_graph and left >= self.K) else 0
                if not k:
                    self.step()
                    k = 1
                left -= k
            torch.cuda.synchronize()
            idx = (torch.arange(start + done, start + done + chunk, device=self.device) % self.loss_cap)
            losses.append(self.loss_out[idx].cpu().numpy())
            done += chunk
        sc = self.read_scalars()
        if sc["error"] or sc["step"] != self.host_step:
            raise _lib.GloveError("device step counter %d != host %d (error flag %d)" % (sc["step"], self.host_step, sc["error"]))
        return np.concatenate(losses) if losses else np.zeros(0, np.float32)

    # ---- predict -------------------------------------------------------------------------------------------------
    def topk(self, query_ids, k: int, exact_fp32: bool = False):
        """Cosine top-k of the ROW embeddings of ``query_ids`` against the whole row table
        (get_predictions, ref src/models/model_utils.py:81-110).  Returns (sim [n,k] f32, idx [n,k] i32) as numpy:
        similarities descending, ties -> lower id.  ``exact_fp32`` forces the CUDA-core scan.

        Row-sharded tables: every rank runs the same call with the same global ``query_ids``; the query rows are
        gathered from their owners (one all-reduce), each rank ranks ALL queries against its own rows, and the per-rank
        top-k lists are all-gathered and merged (ties -> lower global id)."""
        if self.sharded:
            import torch.distributed as dist
            qrows = self.topk_shard_query_rows(query_ids)
            dist.all_reduce(qrows)
            sim, idx = self.topk_shard_local(qrows, k, exact_fp32)
            n, kk = sim.shape
            all_sim = torch.empty(self.dp_world * n * kk, dtype=torch.float32, device=self.device)
            all_idx = torch.empty(self.dp_world * n * kk, dtype=torch.int32, device=self.device)
            dist.all_gather_into_tensor(all_sim, sim.reshape(-1))
            dist.all_gather_into_tensor(all_idx, idx.reshape(-1))
            return self.topk_shard_merge(all_sim.view(self.dp_world, n, kk), all_idx.view(self.dp_world, n, kk), k)
        self.flush()
        qh = np.ascontiguousarray(query_ids, np.int64).reshape(-1)
        if qh.size and (qh.min() < 0 or qh.max() >= self.V):      # the kernels index the table with these: refuse, never clamp
            raise ValueError("topk: query ids must lie in [0, %d): min %d, max %d" % (self.V, qh.min(), qh.max()))
        q = torch.as_tensor(qh.astype(np.int32)).to(self.device)
        n = int(q.numel())
        inv, nb = self._normalised_table()
        sim, idx = self._topk_call(inv, nb, self.row_table, self.P, nb, q, n, k, exact_fp32)
        torch.cuda.synchronize()
        return sim.cpu().numpy().reshape(n, k), idx.cpu().numpy().reshape(n, k)

    def _normalised_table(self):
        if self._norm_cache is None or self._norm_cache[0] != self.host_step:
            Kp, Vp = lib.glove_topk_kpad(self.d), lib.glove_topk_vpad(self.V)
            inv = torch.empty(self.V, dtype=torch.float32, device=self.device)
            nb = torch.empty(Vp * Kp, dtype=torch.bfloat16, device=self.device)
            check(lib.glove_normalize_rows(_ptr(self.row_table), self.V, self.d, self.P, _ptr(nb), _ptr(inv), _stream()),
                  "glove_normalize_rows")
            self._norm_cache = (self.host_step, inv, nb)
        return self._norm_cache[1], self._norm_cache[2]

    def _topk_call(self, inv, nb, qtable, qplanes, qnb, q, n, k, exact_fp32):
        sim = torch.empty(n * k, dtype=torch.float32, device=self.device)
        idx = torch.empty(n * k, dtype=torch.int32, device=self.device)
        ws = torch.empty(max(lib.glove_topk_workspace_bytes(self.V, self.d, n, k), 256), dtype=torch.uint8, device=self.device)
        use_tc = not exact_fp32
        check(lib.glove_topk_cosine_queries(_ptr(self.row_table), self.V, self.d, self.P, _ptr(nb) if use_tc else None, _ptr(inv),
                                            _ptr(qtable), qplanes, _ptr(qnb) if use_tc else None, _ptr(q), n, k, _ptr(sim),
                                            _ptr(idx), _ptr(ws), ws.numel(), _stream()), "glove_topk_cosine")
        if use_tc and self.tc_path_covers(k):
            cnt = ctypes.c_int32(0)
            check(lib.glove_topk_flagged(_ptr(ws), self.V, self.d, n, k, ctypes.byref(cnt), _stream()), "glove_topk_flagged")
            self.last_topk_fallbacks = int(cnt.value)
        return sim, idx

    # ---- row-sharded top-k, in the three phases between which the collectives sit (topk() strings them together) -----
    def topk_shard_query_rows(self, query_ids):
        """[n, S] fp32: the packed plane-0 rows of the queries this rank owns, zero elsewhere (sum over ranks = all rows)."""
        self.flush()
        q = torch.as_tensor(np.ascontiguousarray(query_ids, np.int64)).to(self.device)
        if self._label is not None:
            q = self._label[q]
        out = torch.zeros(q.numel(), self.S, dtype=torch.float32, device=self.device)
        mine = (q % self.dp_world) == self.dp_rank
        rows = self.row_table.view(self.V, self.P, self.S)[:, 0, :]
        out[mine] = rows[q[mine] // self.dp_world]
        return out

    def topk_shard_local(self, qrows, k: int, exact_fp32: bool = False):
        """Top-k of every query (rows of ``qrows``) against the rows held here; ids are returned GLOBAL, pad rows removed.
        One spare candidate is kept when this shard holds a pad row, so that dropping it cannot cost a real one."""
        n = int(qrows.shape[0])
        has_pad = self.V * self.dp_world > self.V_global
        kk = min(k + 1, 32, self.V) if has_pad else min(k, self.V)
        inv, nb = self._normalised_table()
        Kp = lib.glove_topk_kpad(self.d)
        qnb = torch.empty(lib.glove_topk_vpad(n) * Kp, dtype=torch.bfloat16, device=self.device)
        qrows = qrows.contiguous()
        check(lib.glove_normalize_rows(_ptr(qrows), n, self.d, 1, _ptr(qnb), None, _stream()), "glove_normalize_rows")
        ids = torch.arange(n, dtype=torch.int32, device=self.device)
        sim, idx = self._topk_call(inv, nb, qrows, 1, qnb, ids, n, kk, exact_fp32)
        sim, idx = sim.view(n, kk), idx.view(n, kk)
        gid = idx.to(torch.int64) * self.dp_world + self.dp_rank
        bad = (idx < 0) | (gid >= self.V_global)
        sim = torch.where(bad, torch.full_like(sim, float("-inf")), sim)
        if self._unlabel is not None:                  # labels -> original ids BEFORE the merge (ties -> lower original id)
            un = torch.from_numpy(self._unlabel).to(self.device)
            gid = un[torch.where(bad, torch.zeros_like(gid), gid)]
        gid = torch.where(bad, torch.full_like(gid, -1), gid).to(torch.int32)
        if kk < k + 1:                                                   # same list width on every rank
            pad = k + 1 - kk
            sim = torch.cat([sim, torch.full((n, pad), float("-inf"), device=self.device)], 1)
            gid = torch.cat([gid, torch.full((n, pad), -1, dtype=torch.int32, device=self.device)], 1)
        return sim.contiguous(), gid.contiguous()

    def topk_shard_merge(self, all_sim, all_idx, k: int):
        """[world, n, kk] candidate lists -> (sim [n,k], idx [n,k]) numpy."""
        world, n, kk = all_sim.shape
        cs = all_sim.permute(1, 0, 2).reshape(n, world * kk).contiguous()
        ci = all_idx.permute(1, 0, 2).reshape(n, world * kk).contiguous()
        sim = torch.empty(n * k, dtype=torch.float32, device=self.device)
        idx = torch.empty(n * k, dtype=torch.int32, device=self.device)
        check(lib.glove_topk_merge(_ptr(cs), _ptr(ci), n, world * kk, k, _ptr(sim), _ptr(idx), _stream()), "glove_topk_merge")
        torch.cuda.synchronize()
        return sim.cpu().numpy().reshape(n, k), idx.cpu().numpy().reshape(n, k)

    # ---- intrinsic evaluation (evaluate_embeddings) ----------------------------------------------------------------
    def _single_table(self, what):
        if self.sharded:
            raise RuntimeError("%s needs the whole row table on one GPU: load the checkpoint into a one-GPU engine "
                               "(row-sharded engines are not evaluated in place)" % what)

    def analogy(self, abc, k: int = 1, method: str = "add", restrict: Optional[int] = None, exact_fp32: bool = False):
        """Word analogies a : b :: c : ? over the row table (glove_analogy_topk).  ``abc`` int [n, 3]; ``method`` "add"
        (3CosAdd) or "mul" (3CosMul); the candidates are the first ``restrict`` rows (default all), a, b and c excluded.
        Returns (score [n,k] f32, idx [n,k] i32) as numpy, scores descending, ties -> lower id.  ``exact_fp32`` makes
        3CosAdd skip the tensor-core candidate pass (3CosMul is always an exact fp32 scan)."""
        self._single_table("analogy")
        if method not in _lib.ANALOGY_METHODS:
            raise ValueError("analogy: method must be one of %s, not %r" % (sorted(_lib.ANALOGY_METHODS), method))
        V = self.V if restrict is None else int(restrict)
        if not 1 <= V <= self.V:
            raise ValueError("analogy: restrict=%d not in [1, %d]" % (V, self.V))
        abc = np.ascontiguousarray(abc, np.int64).reshape(-1, 3)
        n = abc.shape[0]
        if n == 0:
            return np.zeros((0, k), np.float32), np.zeros((0, k), np.int32)
        if abc.min() < 0 or abc.max() >= V:     # the kernels index the table with these: refuse, never clamp
            raise ValueError("analogy: word ids must lie in [0, %d): min %d, max %d" % (V, abc.min(), abc.max()))
        self.flush()
        inv, nb = self._normalised_table()
        m = _lib.ANALOGY_METHODS[method]
        q = torch.as_tensor(abc.astype(np.int32)).to(self.device)
        score = torch.empty(n * k, dtype=torch.float32, device=self.device)
        idx = torch.empty(n * k, dtype=torch.int32, device=self.device)
        ws = torch.empty(max(lib.glove_analogy_workspace_bytes(V, self.d, n, k, m), 256), dtype=torch.uint8, device=self.device)
        use_tc = method == "add" and not exact_fp32
        check(lib.glove_analogy_topk(_ptr(self.row_table), V, self.d, self.P, _ptr(nb) if use_tc else None, _ptr(inv),
                                     _ptr(q), n, m, k, _ptr(score), _ptr(idx), _ptr(ws), ws.numel(), _stream()),
              "glove_analogy_topk")
        torch.cuda.synchronize()
        return score.cpu().numpy().reshape(n, k), idx.cpu().numpy().reshape(n, k)

    def pair_cosine(self, pairs) -> np.ndarray:
        """Cosine of the row embeddings of each pair (int [n, 2]) as numpy f32 [n]: bit for bit the similarity that
        ``topk([w1])`` reports for w2."""
        self._single_table("pair_cosine")
        pairs = np.ascontiguousarray(pairs, np.int64).reshape(-1, 2)
        n = pairs.shape[0]
        if n == 0:
            return np.zeros(0, np.float32)
        if pairs.min() < 0 or pairs.max() >= self.V:
            raise ValueError("pair_cosine: word ids must lie in [0, %d): min %d, max %d" % (self.V, pairs.min(), pairs.max()))
        self.flush()
        inv, _ = self._normalised_table()
        p = torch.as_tensor(pairs.astype(np.int32)).to(self.device)
        out = torch.empty(n, dtype=torch.float32, device=self.device)
        check(lib.glove_pair_cosine(_ptr(self.row_table), self.V, self.d, self.P, _ptr(inv), _ptr(p), n, _ptr(out), _stream()),
              "glove_pair_cosine")
        torch.cuda.synchronize()
        return out.cpu().numpy()

    def tc_path_covers(self, k: int) -> bool:
        """Shapes the tcgen05 candidate pass handles (everything else runs the exact fp32 scan)."""
        return lib.glove_topk_kpad(self.d) <= 320 and k <= 24 and self.V >= 1024

    # ---- eval ----------------------------------------------------------------------------------------------------
    def eval_sums(self, batch_size: Optional[int] = None, first: int = 0, count: Optional[int] = None) -> np.ndarray:
        """Per-batch metric sums, double [n_batches, 8] (see glove_eval_loss)."""
        self.flush()
        batch_size = batch_size or self.B
        count = self.nnz - first if count is None else count
        nb = (count + batch_size - 1) // batch_size
        out = torch.zeros(nb * 8, dtype=torch.float64, device=self.device)
        ws = torch.empty(lib.glove_eval_workspace_bytes(count, batch_size), dtype=torch.uint8, device=self.device)
        row, col, ca, cb = self.coo
        check(lib.glove_eval_loss(_ptr(self.row_table), _ptr(self.col_table), _ptr(self.scalars), self.P, self.d,
                                  _ptr(row), _ptr(col), _ptr(ca), _ptr(cb), first, count, batch_size,
                                  _lib.HEADS[self.head], _ptr(out), _ptr(ws), ws.numel(), _stream()), "glove_eval_loss")
        return out.cpu().numpy().reshape(nb, 8)

    def eval_metrics(self, batch_size: Optional[int] = None) -> Dict[str, float]:
        """RegressionHead EVAL metrics over one pass of the COO in file order [ref src/models/estimator.py:87-92]."""
        batch_size = batch_size or self.B
        s = self.eval_sums(batch_size)
        n = self.nnz
        sizes = np.full(len(s), batch_size, np.float64)
        sizes[-1] = n - batch_size * (len(s) - 1)
        g = float(self.read_scalars()["g"])
        lam, d = self.l2_reg, self.d
        reg = self.reg_scale * ((lam / d) * s[:, 4] / sizes + (lam / d) * s[:, 5] / sizes + lam * s[:, 6] / sizes
                                + lam * s[:, 7] / sizes + lam * g * g)
        if self.head == "glove":
            data = s[:, 0] / sizes
            return {"average_loss": float(s[:, 0].sum() / s[:, 1].sum()), "loss": float(np.mean(data + reg)),
                    "label/mean": float(s[:, 2].sum() / s[:, 1].sum()),
                    "prediction/mean": float(s[:, 3].sum() / s[:, 1].sum()),
                    "regularization_loss": float(np.mean(reg))}
        data = s[:, 0] / sizes + self.neg_factor * s[:, 2] / sizes
        return {"loss": float(np.mean(data + reg)), "regularization_loss": float(np.mean(reg)),
                "pos/average_loss": float(s[:, 0].sum() / max(s[:, 1].sum(), 1e-30)),
                "neg/average_loss": float(s[:, 2].sum() / max(s[:, 3].sum(), 1e-30))}
