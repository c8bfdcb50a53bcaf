"""Device-side state and step orchestration of the AAE hot path.

``AAEEngine`` owns the weights, the four Adam states and the per-batch workspaces in HBM and
enqueues the kernels of one ``partial_fit`` (reference: aaerec/aae.py:745-766 -> ae_step 676-711,
disc_step 713-732, gen_step 734-743) and of ``predict`` (aae.py:840-870) through the C ABI in
``include/aae_b200.h``.  PyTorch is used for memory, streams, CUDA graphs and (multi-GPU)
``torch.distributed`` only -- every numeric op on the path is one of our kernels.

HBM layout (fp32, row-major)
  W1t  [Vloc,H]  enc.lin1.weight transposed (+ m1,v1 for enc_optim, m2,v2 for gen_optim)
  Wd3  [Vloc,H]  dec.lin3.weight (+ m,v), bd3 [Vloc] (+ m,v)
  enc/dec/disc   small layers packed in one block each (see aae_b200.h), with moment/grad blocks
Item-sharded over ``world`` ranks: rank r owns items [v_begin, v_end); small layers replicated and
computed redundantly (identical inputs and RNG on every rank), so the only exchanges are the
all-reduce of h1pre partial sums and of (dh2, loss) -- SURVEY.md 8(e).
"""
import ctypes as C
import gc
import os

import numpy as np
import torch

from . import _native as N
from ._native import call, ptr, AaeDims

# Philox stream ids of the 12 dropout layers of one step, in the reference's draw order (A11)
_DROP_ORDER = ("ae_e1", "ae_e2", "ae_d1", "ae_d2", "disc_r1", "disc_r2", "disc_f1", "disc_f2",
               "gen_e1", "gen_e2", "gen_q1", "gen_q2")


from .dist import shard_range, gather_item_shards, gather_topk_candidates  # noqa: E402,F401


def enc_block_sizes(H, C_):
    return [("enc.lin1.bias", H), ("enc.lin2.weight", H * H), ("enc.lin2.bias", H),
            ("enc.lin3.weight", C_ * H), ("enc.lin3.bias", C_)]


def dec_block_sizes(H, Cp):
    return [("dec.lin1.weight", H * Cp), ("dec.lin1.bias", H), ("dec.lin2.weight", H * H), ("dec.lin2.bias", H)]


def disc_block_sizes(H, C_):
    return [("disc.lin1.weight", H * C_), ("disc.lin1.bias", H), ("disc.lin2.weight", H * H),
            ("disc.lin2.bias", H), ("disc.lin3.weight", H), ("disc.lin3.bias", 1)]


def _on_device(fn):
    """Run an engine entry point with the engine's GPU as the CUDA current device: the C ABI launches on the current
    device, so ``device='cuda:1'`` must not depend on the caller having called ``torch.cuda.set_device``."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **kw):
        if torch.cuda.current_device() == self.dev.index:
            return fn(self, *a, **kw)
        with torch.cuda.device(self.dev):
            return fn(self, *a, **kw)
    return wrapper


class _Branch(object):
    """Fork of the current stream onto ``engine.side2`` (see AAEEngine._branch)."""

    def __init__(self, eng):
        self.eng = eng
        self.ctx = None

    def __enter__(self):
        eng = self.eng
        if not eng.branches:
            return self
        cur = torch.cuda.current_stream(eng.dev)
        eng._ev_fork2.record(cur)
        eng.side2.wait_event(eng._ev_fork2)
        self.ctx = torch.cuda.stream(eng.side2)
        self.ctx.__enter__()
        return self

    def __exit__(self, *a):
        if self.ctx is None:
            return False
        self.eng._ev_join2.record(self.eng.side2)
        self.ctx.__exit__(*a)
        self.ctx = None
        return False


class AAEEngine(object):
    has_encoder = True      # False: no sparse first layer / W1t (the decoder-only engine of engine_siblings.py)

    def enc_sizes(self):
        return enc_block_sizes(self.H, self.C)

    def dec_sizes(self):
        return dec_block_sizes(self.H, self.Cp)

    def disc_sizes(self):
        return disc_block_sizes(self.H, self.C)

    # Every change of the output layer sets _wp_dirty; it also bumps the weight version that the compact candidate copy
    # (``_compact``) is checked against.
    @property
    def _wp_dirty(self):
        return self._wp_stale

    @_wp_dirty.setter
    def _wp_dirty(self, v):
        self._wp_stale = bool(v)
        if v:
            self._wver = getattr(self, "_wver", 0) + 1

    def __init__(self, n_items, n_hidden=100, n_code=50, cond_dim=0, gen_lr=1e-3, reg_lr=1e-3,
                 dropout=(.2, .2), prior_scale=None, normalize_inputs=True, device=None,
                 rank=0, world=1, group=None, impl="auto", seed=0, max_batch=128, max_nnz=None,
                 use_graph=True, overlap_sweep=True, adversarial=True, exchange="auto", inference_only=False):
        self.inference_only = bool(inference_only)
        N.require_device(0 if device is None else (torch.device(device).index or 0))
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.dev.index is None:
            self.dev = torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(self.dev):
            self._construct(n_items, n_hidden, n_code, cond_dim, gen_lr, reg_lr, dropout, prior_scale,
                            normalize_inputs, rank, world, group, impl, seed, max_batch, max_nnz, use_graph,
                            overlap_sweep, adversarial, exchange)

    def _construct(self, n_items, n_hidden, n_code, cond_dim, gen_lr, reg_lr, dropout, prior_scale, normalize_inputs,
                   rank, world, group, impl, seed, max_batch, max_nnz, use_graph, overlap_sweep, adversarial, exchange):
        self.V, self.H, self.C, self.D = int(n_items), int(n_hidden), int(n_code), int(cond_dim)
        self.Cp = self.C + self.D
        self.gen_lr, self.reg_lr = float(gen_lr), float(reg_lr)
        self.dropout = (float(dropout[0]), float(dropout[1]))
        self.prior_scale = 1.0 if prior_scale is None else float(prior_scale)
        self.normalize = 1 if normalize_inputs else 0
        self.rank, self.world, self.group = int(rank), int(world), group
        self.v_begin, self.v_end = shard_range(self.V, self.rank, self.world)
        self.Vloc = self.v_end - self.v_begin
        self.seed = int(seed)
        # adversarial=False: the plain AutoEncoder of aae.py:221-458 -- the reconstruction phase alone (enc_optim and
        # dec_optim at one learning rate; pass reg_lr=0 so that the unused second Adam state of W1t stays exactly zero)
        self.adversarial = bool(adversarial)
        self.use_graph = bool(use_graph)
        self.peer = None
        self._exchange_kind = "none"
        self.overlap_sweep = bool(overlap_sweep) and os.environ.get("AAE_B200_NO_OVERLAP", "") == ""
        self.branches = os.environ.get("AAE_B200_NO_BRANCH", "") == ""   # parallel graph branches (debug switch)
        # 64-thread sweep CTAs per SM that run beside the decoder-output kernel (0: the stand-alone wide sweep)
        self.sweep_ctas = int(os.environ.get("AAE_B200_SWEEP_CTAS", "4"))   # measured at the MPD shape: 2 -> 1517, 4 -> 1443, 8 -> 1467 us per step
        # W1t Adam policy: rows outside the batch are swept in G time-blocked groups (1 = dense sweep every step)
        # (measured at V=2M: 2.01 / 1.82 / 1.67 ms per step for G = 8 / 16 / 32 -- the group sweep runs exposed behind
        # the decoder kernel; V=200k: no difference)
        self.w1_groups = max(1, min(32, int(os.environ.get("AAE_B200_W1_GROUPS", "32"))))
        self.impl = self._pick_impl(impl)
        self.steps_done = 0
        self._launches_per_step = 0
        self._phase_cursor = 0
        self._phase_ctx_live = None
        self._epoch = None
        self._gwork = None
        self._wp = None             # padded [Vloc,104] copy of the output layer for the TMA-fed predict filter
        self._wp_dirty = True
        self._cmp = None            # compact [A,H] copy of the shard's eligible rows of the output layer (``_compact``)
        self._xstage = None         # pinned + device staging of the batch's exclusion CSR (``_upload_exclusions``)
        self._topk_out = None
        f32 = dict(dtype=torch.float32, device=self.dev)
        H, Cc, Cp, Vl = self.H, self.C, self.Cp, max(self.Vloc, 1)
        z = lambda *s: torch.zeros(*s, **f32)
        # inference-only engines (set-sharded predict replicas) carry the weights without the six [V,H] Adam tensors
        zm = (lambda *s: torch.zeros(*((1,) + tuple(s[1:])), **f32)) if self.inference_only else z
        Vw = Vl if self.has_encoder else 1
        self.W1t = z(Vw, H)
        self.W1_m1, self.W1_v1, self.W1_m2, self.W1_v2 = (zm(Vw, H) for _ in range(4))
        self.Wd3 = z(Vl, H)
        self.Wd3_m, self.Wd3_v = (zm(Vl, H) for _ in range(2))
        self.bd3 = z(Vl)
        self.bd3_m, self.bd3_v = (zm(Vl) for _ in range(2))
        self.n_enc = max(1, sum(s for _, s in self.enc_sizes()))
        self.n_dec = max(1, sum(s for _, s in self.dec_sizes()))
        self.n_disc = max(1, sum(s for _, s in self.disc_sizes()))
        self.enc, self.enc_m1, self.enc_v1, self.enc_m2, self.enc_v2, self.g_enc = (z(self.n_enc) for _ in range(6))
        self.dec, self.dec_m, self.dec_v, self.g_dec = (z(self.n_dec) for _ in range(4))
        self.disc, self.disc_m, self.disc_v, self.g_disc = (z(self.n_disc) for _ in range(4))
        self.state = torch.zeros(C.sizeof(N.StepState), dtype=torch.uint8, device=self.dev)
        self.slot_of = torch.full((Vl,), -1, dtype=torch.int32, device=self.dev)
        # time-blocked dense Adam of W1t (w1_blocked.cu): last applied step per row, per-step claim marks, and the
        # ring of per-step Adam constants
        self.w1_last = torch.zeros(Vl, dtype=torch.int32, device=self.dev)
        self.w1_claim = torch.zeros(Vl, dtype=torch.int32, device=self.dev)
        self.ktab = torch.zeros(64 * 4, **f32)
        self._w1_dirty = False
        self.loss_sums = torch.zeros(3, dtype=torch.float64, device=self.dev)
        self._topk_work = None
        self._n_bad = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.topk_fallbacks = 0
        self.losses = torch.zeros(3, **f32)
        self._ws_B = 0
        self._ws_nnz = 0
        self._graphs = {}
        # torch hands out streams from a small round-robin pool: make sure the three we use together (capture
        # stream + two side streams) are different CUDA streams, or a fork would alias the capturing stream
        self._cap_stream, self.side, self.side2 = self._distinct_streams(3)
        self._ev_fork = torch.cuda.Event()
        self._ev_join = torch.cuda.Event()
        self._ev_prep = torch.cuda.Event()
        self._ev_k3 = torch.cuda.Event()
        self._ev_fork2 = torch.cuda.Event()
        self._ev_join2 = torch.cuda.Event()
        self._init_state()
        self._ensure_ws(max_batch, max_nnz or max_batch * 64)
        if self.world > 1:
            self._setup_exchange(exchange, max(int(max_batch), 128) * self.H)

    # ------------------------------------------------------------------ plumbing
    def _setup_exchange(self, exchange, n_max):
        """Item shards exchange [B,H] partial sums three times per step: through our own one-shot all-reduce kernel
        over NVLink peer memory (``PeerExchange``; graph-capturable), or -- when CUDA IPC mapping is not possible or
        ``exchange='nccl'`` / AAE_B200_EXCHANGE=nccl -- through NCCL all-reduces (eager, no CUDA graph)."""
        kind = os.environ.get("AAE_B200_EXCHANGE", exchange)
        if kind in ("auto", "peer"):
            try:
                from .dist import PeerExchange
                self.peer = PeerExchange(self.rank, self.world, self.group, n_max, self.dev)
                self._exchange_kind = "peer"
            except Exception as e:   # noqa: BLE001
                if kind == "peer":
                    raise
                if self.rank == 0:
                    print("aaerec_b200: peer-memory exchange unavailable (%s); using NCCL all-reduce" % (e,))
                self.peer = None
        if self.peer is None:
            self._exchange_kind = "nccl"
            self.use_graph = self.use_graph and os.environ.get("AAE_B200_NCCL_GRAPH", "") == "1"

    def _init_state(self):
        """Step state for step 1 (aae_step_finish advances it at the end of every step), loss sums cleared."""
        call("aae_step_state_init", ptr(self.state), self.gen_lr, self.reg_lr, C.c_uint64(self.seed), self._stream())
        call("aae_step_tick", ptr(self.state), self._stream())
        call("aae_ktab_write", ptr(self.state), ptr(self.ktab), self._stream())
        self.loss_sums.zero_()
        self.w1_last.zero_()
        self.w1_claim.zero_()
        self._w1_dirty = False

    def _distinct_streams(self, n):
        seen = {torch.cuda.current_stream(self.dev).cuda_stream, torch.cuda.default_stream(self.dev).cuda_stream}
        out = []
        for _ in range(256):
            st = torch.cuda.Stream(device=self.dev)
            if st.cuda_stream not in seen:
                seen.add(st.cuda_stream)
                out.append(st)
                if len(out) == n:
                    return out
        raise RuntimeError("could not obtain %d distinct CUDA streams" % n)

    def _pick_impl(self, impl):
        names = {"simt": 0, "fp32": 0, "tc": 1, "tc3": 1, "parity": 1, "tf32": 2, "fast": 2}
        if impl == "auto":
            return -1          # resolved per batch: tensor-core kernel when the shape is inside its envelope
        if isinstance(impl, int):
            return impl
        return names[impl]

    def impl_for(self, B):
        """Decoder-output kernel for a batch of B rows: 1 = tcgen05 3xTF32 (n_hidden % 4 == 0, n_hidden <= 124; any
        batch size: batches beyond one row chunk are walked chunk by chunk, aae_dec_out_train_ws), 0 = fp32 CUDA cores
        (any shape up to n_hidden 512)."""
        if self.impl >= 0:
            return self.impl
        ok = self.H % 4 == 0 and self.H <= 124
        if ok and B > 128 and int(N.load().aae_dec_out_train_work_floats(B, self.H, max(self.Vloc, 1), 1)) == 0:
            ok = False      # n_hidden outside the pipelined kernel's envelope: no chunked path
        return 1 if ok else 0

    def impl_for_scores(self):
        """Scores / fused v1 kernel: 1 = tcgen05 3xTF32 (n_hidden % 4 == 0, n_hidden <= 108: a [Wd3 | bd3] row of at
        most 112 floats fits its operand tile), 0 = fp32 CUDA cores (any n_hidden up to 512)."""
        if self.impl >= 0:
            return self.impl
        return 1 if (self.H % 4 == 0 and self.H <= 108) else 0

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def _ensure_ws(self, B, nnz):
        if B <= self._ws_B and nnz <= self._ws_nnz:
            return
        # grow geometrically: every growth synchronises, drops the captured graphs and re-pins the staging slots
        if self._ws_B:
            B = max(self._ws_B, B if B <= self._ws_B else max(B, int(1.5 * self._ws_B)))
            nnz = max(self._ws_nnz, nnz if nnz <= self._ws_nnz else max(nnz, int(1.5 * self._ws_nnz)))
        nnz = max(nnz, 1)
        torch.cuda.synchronize(self.dev)
        if self.peer is not None and B * self.H > self.peer.n_max:
            # the exchange buffers are sized for the largest [B,H] message: re-create them (collective: every rank
            # sees the same batch sizes) instead of silently issuing NCCL calls inside a graph capture
            from .dist import PeerExchange
            self.peer.close()
            self.peer = PeerExchange(self.rank, self.world, self.group, max(B, 128) * self.H, self.dev)
        self._graphs.clear()
        f32 = dict(dtype=torch.float32, device=self.dev)
        i32 = dict(dtype=torch.int32, device=self.dev)
        H, Cc, Cp, D = self.H, self.C, self.Cp, self.D
        z = lambda *s: torch.zeros(*s, **f32)
        # CSR rows of the batch, packed: indptr block (padded to 16 bytes) directly followed by the column indices, so
        # that the host-buffer entry moves a batch with ONE H2D copy (aae_upload_batch)
        off = (B + 1 + 3) // 4 * 4
        self._batch = torch.zeros(off + nnz, **i32)
        self.indptr = self._batch[: B + 1]
        self.indices = self._batch[off: off + nnz]
        self.cond = z(B, max(D, 1))
        self.masks = z(12, B, H)
        self.z_real = z(B, Cc)
        self.uniq = torch.zeros(nnz, **i32)
        self.n_uniq = torch.zeros(1, **i32)
        self.csc_cnt, self.csc_pos, self.csc_off, self.csc_row = (torch.zeros(nnz + 1, **i32) for _ in range(4))
        self.h1pre, self.a1, self.a2, self.dd1, self.h2, self.dh2 = (z(B, H) for _ in range(6))
        self.zc = z(B, Cp)
        self.g_d2, self.g_d1, self.g_e2, self.g_h1 = (z(B, H) for _ in range(4))
        self.g_z = z(B, Cc)
        self.h1pre2, self.ga1, self.ga2, self.gg_e2, self.gg_h1 = (z(B, H) for _ in range(5))
        self.gg_z = z(B, Cc)
        self.disc_acts = z(B, 2 * (Cc + 2 * H))
        self.disc_grads = z(B, 2 * (2 * H + 1))
        # pinned staging ring for the host-buffer (end-to-end) entry
        self._pin = []
        for _ in range(8):
            packed = torch.zeros(off + nnz, dtype=torch.int32).pin_memory()
            self._pin.append(dict(
                packed=packed, indptr=packed[: B + 1], indices=packed[off: off + nnz],
                cond=torch.zeros(B, max(D, 1), dtype=torch.float32).pin_memory(),
                ev=None))
        self._pin_i = 0
        # zero-copy staging for train_step_host: two pinned (mapped) slots that the step's graph reads / writes itself
        self._zc = []
        for _ in range(2):
            self._zc.append(dict(packed=torch.zeros(off + nnz, dtype=torch.int32).pin_memory(),
                                 cond=torch.zeros(B, max(D, 1), dtype=torch.float32).pin_memory(),
                                 losses=torch.zeros(4, dtype=torch.float32).pin_memory(), ev=None))
        self._zc_i = 0
        self._zc_off = off
        self._ws_B, self._ws_nnz = B, nnz

    # ------------------------------------------------------------------ parameters
    @_on_device
    def load_params(self, params):
        """``params``: torch-layout state dict (keys ``enc.lin1.weight`` ... as in the reference's
        modules, aae.py:104-213); values numpy arrays or tensors (full, unsharded)."""
        def t(name):
            return torch.as_tensor(np.asarray(params[name]) if not torch.is_tensor(params[name]) else params[name],
                                   dtype=torch.float32)
        lo, hi = self.v_begin, self.v_end
        W1 = t("enc.lin1.weight")            # [H,V]
        assert W1.shape == (self.H, self.V), (W1.shape, self.H, self.V)
        self.W1t.copy_(W1[:, lo:hi].t().contiguous())
        Wd3 = t("dec.lin3.weight")           # [V,H]
        self.Wd3.copy_(Wd3[lo:hi].contiguous())
        self.bd3.copy_(t("dec.lin3.bias")[lo:hi])
        for blk, sizes in ((self.enc, enc_block_sizes(self.H, self.C)), (self.dec, dec_block_sizes(self.H, self.Cp)),
                           (self.disc, disc_block_sizes(self.H, self.C))):
            off = 0
            for name, sz in sizes:
                if name not in params and name.startswith("disc.") and not self.adversarial:
                    blk[off:off + sz].zero_()      # the plain AutoEncoder has no discriminator
                    off += sz
                    continue
                v = t(name).reshape(-1)
                assert v.numel() == sz, (name, v.numel(), sz)
                blk[off:off + sz].copy_(v)
                off += sz
        for m in (self.W1_m1, self.W1_v1, self.W1_m2, self.W1_v2, self.Wd3_m, self.Wd3_v, self.bd3_m, self.bd3_v,
                  self.enc_m1, self.enc_v1, self.enc_m2, self.enc_v2, self.dec_m, self.dec_v, self.disc_m, self.disc_v):
            m.zero_()
        self._init_state()
        self.steps_done = 0
        self._wp_dirty = True

    INIT_BLOCK = 65536      # items per generator block of init_uniform

    @_on_device
    def init_uniform(self, seed=42):
        """Random-init weights of the reference architecture directly in HBM (nn.Linear's law: U(-1/sqrt(fan_in),
        1/sqrt(fan_in)) for weight and bias), without building the full [V,H] matrices on the host -- for synthetic
        benchmarks at vocabulary sizes where a host-side state dict is impractical (MPD shape, 2M items).  The
        item-sharded layers are drawn in blocks of INIT_BLOCK items, each block from its own generator seeded by
        (seed, tensor, block index): the full matrices are therefore the SAME for every world size, and a rank fills
        exactly the rows of its item range (so an N-GPU run can be checked against a 1-GPU run).  The replicated small
        layers are drawn identically on every rank."""
        gs = torch.Generator(device=self.dev).manual_seed(int(seed))                      # same on every rank

        def fill(t, fan_in, g):
            bound = 1.0 / float(np.sqrt(fan_in))
            t.uniform_(-bound, bound, generator=g)

        def fill_items(t, fan_in, tensor_id):
            bound = 1.0 / float(np.sqrt(fan_in))
            blk = self.INIT_BLOCK
            width = (self.H,) if t.dim() == 2 else ()
            for b in range(self.v_begin // blk, (max(self.v_end, 1) - 1) // blk + 1):
                g = torch.Generator(device=self.dev).manual_seed(int(seed) * 1000003 + tensor_id * 7919 + b * 31 + 17)
                full = torch.empty((blk,) + width, dtype=torch.float32, device=self.dev)
                full.uniform_(-bound, bound, generator=g)
                lo, hi = max(self.v_begin, b * blk), min(self.v_end, (b + 1) * blk)
                if hi > lo:
                    t[lo - self.v_begin: hi - self.v_begin].copy_(full[lo - b * blk: hi - b * blk])
        fill_items(self.W1t, self.V, 1)
        fill_items(self.Wd3, self.H, 2)
        fill_items(self.bd3, self.H, 3)
        fan = {"enc.lin1.bias": self.V, "enc.lin2": self.H, "enc.lin3": self.H, "dec.lin1": self.Cp, "dec.lin2": self.H,
               "disc.lin1": self.C, "disc.lin2": self.H, "disc.lin3": self.H}
        for blk, sizes in ((self.enc, enc_block_sizes(self.H, self.C)), (self.dec, dec_block_sizes(self.H, self.Cp)),
                           (self.disc, disc_block_sizes(self.H, self.C))):
            off = 0
            for name, sz in sizes:
                key = name if name in fan else name.rsplit(".", 1)[0]
                fill(blk[off:off + sz], fan[key], gs)
                off += sz
        for m in (self.W1_m1, self.W1_v1, self.W1_m2, self.W1_v2, self.Wd3_m, self.Wd3_v, self.bd3_m, self.bd3_v,
                  self.enc_m1, self.enc_v1, self.enc_m2, self.enc_v2, self.dec_m, self.dec_v, self.disc_m, self.disc_v):
            m.zero_()
        self._init_state()
        self.steps_done = 0
        self._wp_dirty = True

    def _gather_items(self, local):
        """All-gather an item-sharded [Vloc, ...] tensor into [V, ...] (state export / dense predict)."""
        return gather_item_shards(local[: self.Vloc], self.V, self.world, self.group)

    @_on_device
    def state_dict(self):
        """Weights in the reference's torch layout (full, gathered over shards), on the host."""
        self.flush_w1()
        torch.cuda.synchronize(self.dev)
        self.check_exchange()
        out = {}
        out["enc.lin1.weight"] = self._gather_items(self.W1t[: self.Vloc]).t().contiguous().cpu()
        out["dec.lin3.weight"] = self._gather_items(self.Wd3[: self.Vloc]).contiguous().cpu()
        out["dec.lin3.bias"] = self._gather_items(self.bd3[: self.Vloc]).contiguous().cpu()
        shapes = {"enc.lin2.weight": (self.H, self.H), "enc.lin3.weight": (self.C, self.H),
                  "dec.lin1.weight": (self.H, self.Cp), "dec.lin2.weight": (self.H, self.H),
                  "disc.lin1.weight": (self.H, self.C), "disc.lin2.weight": (self.H, self.H),
                  "disc.lin3.weight": (1, self.H)}
        for blk, sizes in ((self.enc, enc_block_sizes(self.H, self.C)), (self.dec, dec_block_sizes(self.H, self.Cp)),
                           (self.disc, disc_block_sizes(self.H, self.C))):
            off = 0
            for name, sz in sizes:
                v = blk[off:off + sz].cpu()
                out[name] = v.reshape(shapes[name]) if name in shapes else v.clone()
                off += sz
        return out

    @_on_device
    def make_replica(self, max_batch=1024):
        """Set-sharded predict (SURVEY 8(e) 'Predict: ... or set-sharded replicas'): a single-rank, inference-only engine
        on this GPU holding the FULL weights (item shards all-gathered once, collective), so that every rank can rank
        its own slice of the query rows with zero communication.  Query sets are independent; the weights (1.6 GB at the
        MPD shape) fit every GPU."""
        self.flush_w1()
        rep = AAEEngine(self.V, self.H, self.C, cond_dim=self.D, dropout=self.dropout, prior_scale=self.prior_scale,
                        normalize_inputs=bool(self.normalize), device=self.dev, rank=0, world=1,
                        impl={-1: "auto"}.get(self.impl, self.impl), seed=self.seed, max_batch=max_batch,
                        use_graph=False, adversarial=self.adversarial, inference_only=True)
        rep.W1t.copy_(self._gather_items(self.W1t[: self.Vloc]))
        rep.Wd3.copy_(self._gather_items(self.Wd3[: self.Vloc]))
        rep.bd3.copy_(self._gather_items(self.bd3[: self.Vloc]))
        rep.enc.copy_(self.enc)
        rep.dec.copy_(self.dec)
        rep.disc.copy_(self.disc)
        rep._w1_dirty = False
        rep._wp_dirty = True
        return rep

    def optim_state(self, which):
        """Adam moments of one of the reference's four optimizers (aae.py:798-804) in torch's parameter names and
        layouts: {name: (exp_avg, exp_avg_sq)} host tensors, gathered over item shards."""
        self.flush_w1()
        torch.cuda.synchronize(self.dev)
        shapes = {"enc.lin2.weight": (self.H, self.H), "enc.lin3.weight": (self.C, self.H),
                  "dec.lin1.weight": (self.H, self.Cp), "dec.lin2.weight": (self.H, self.H),
                  "disc.lin1.weight": (self.H, self.C), "disc.lin2.weight": (self.H, self.H),
                  "disc.lin3.weight": (1, self.H)}

        def block(m, v, sizes):
            out, off = {}, 0
            for name, sz in sizes:
                a, b = m[off:off + sz].cpu(), v[off:off + sz].cpu()
                if name in shapes:
                    a, b = a.reshape(shapes[name]), b.reshape(shapes[name])
                out[name] = (a, b)
                off += sz
            return out

        def items(t, transpose=False):
            g = self._gather_items(t[: self.Vloc])
            return (g.t().contiguous() if transpose else g.contiguous()).cpu()
        if which in ("enc", "gen"):
            m, v = (self.enc_m1, self.enc_v1) if which == "enc" else (self.enc_m2, self.enc_v2)
            wm, wv = (self.W1_m1, self.W1_v1) if which == "enc" else (self.W1_m2, self.W1_v2)
            out = {"enc.lin1.weight": (items(wm, True), items(wv, True))}
            out.update(block(m, v, enc_block_sizes(self.H, self.C)))
            return out
        if which == "dec":
            out = block(self.dec_m, self.dec_v, dec_block_sizes(self.H, self.Cp))
            out["dec.lin3.weight"] = (items(self.Wd3_m), items(self.Wd3_v))
            out["dec.lin3.bias"] = (items(self.bd3_m), items(self.bd3_v))
            return out
        if which == "disc":
            return block(self.disc_m, self.disc_v, disc_block_sizes(self.H, self.C))
        raise KeyError(which)

    # ------------------------------------------------------------------ batch staging
    @_on_device
    def upload_csr(self, indptr_np, indices_np, cond_np=None):
        """Host CSR rows (int32, row-relative indptr starting at 0) -> device batch buffers,
        through pinned staging; returns (B, nnz).  This is the H2D leg of the end-to-end path."""
        B = int(indptr_np.shape[0]) - 1
        nnz = int(indptr_np[-1])
        self._ensure_ws(B, nnz)
        slot = self._pin[self._pin_i]
        self._pin_i = (self._pin_i + 1) % len(self._pin)
        if slot["ev"] is not None:
            slot["ev"].synchronize()
        slot["indptr"][: B + 1].numpy()[:] = indptr_np
        slot["indices"][:nnz].numpy()[:] = indices_np[:nnz]
        call("aae_upload_batch", ptr(slot["indptr"]), ptr(slot["indices"]), B, nnz, ptr(self.indptr),
             ptr(self.indices), self._stream())
        if self.D and cond_np is not None:
            slot["cond"][:B].numpy()[:] = cond_np
            self.cond[:B].copy_(slot["cond"][:B], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        slot["ev"] = ev
        return B, nnz

    @_on_device
    def set_batch_device(self, indptr_dev, indices_dev, cond_dev=None):
        """Batch already resident in HBM (bench 'value' leg): device-to-device into the fixed buffers."""
        B = indptr_dev.numel() - 1
        nnz = indices_dev.numel()
        self._ensure_ws(B, nnz)
        self.indptr[: B + 1].copy_(indptr_dev, non_blocking=True)
        if nnz:
            self.indices[:nnz].copy_(indices_dev, non_blocking=True)
        if self.D:
            self.cond[:B].copy_(cond_dev, non_blocking=True)
        return B, nnz

    @_on_device
    def set_epoch_data(self, indptr, indices, cond=None):
        """Device-side epoch feed: keep the whole training (or query) matrix in HBM -- CSR with sorted unique
        columns -- and, optionally, the float32 condition matrix [n, D]; batches are then built on the device by
        ``gather_batch`` from a row permutation (aae.py:815-823 without the host round trip)."""
        indptr = np.ascontiguousarray(indptr, dtype=np.int64)
        indices = np.ascontiguousarray(indices, dtype=np.int32)
        ep = dict(n=int(indptr.shape[0]) - 1,
                  indptr=torch.from_numpy(indptr).to(self.dev),
                  indices=torch.from_numpy(indices if indices.size else np.zeros(1, np.int32)).to(self.dev),
                  lens=np.diff(indptr), cond=None, perm=None)
        if cond is not None:
            cond = np.ascontiguousarray(cond, dtype=np.float32)
            assert cond.shape == (ep["n"], self.D), (cond.shape, ep["n"], self.D)
            ep["cond"] = torch.from_numpy(cond).to(self.dev)
        self._epoch = ep
        return ep

    @_on_device
    def set_epoch_perm(self, perm):
        """Row order of the coming epoch (host permutation, e.g. the reference's np.random shuffle); None = identity.
        Returns the nnz of every batch boundary prefix (int64 cumulative lengths in that order)."""
        ep = self._epoch
        if perm is None:
            ep["perm"] = None
            lens = ep["lens"]
        else:
            perm = np.ascontiguousarray(perm, dtype=np.int32)
            assert perm.shape[0] == ep["n"]
            ep["perm"] = torch.from_numpy(perm).to(self.dev)
            lens = ep["lens"][perm]
        csum = np.zeros(ep["n"] + 1, dtype=np.int64)
        np.cumsum(lens, out=csum[1:])
        ep["csum"] = csum
        return csum

    @_on_device
    def gather_batch(self, row0, B):
        """Build the batch of rows perm[row0 : row0+B) of the resident matrix in the device batch buffers."""
        ep = self._epoch
        nnz = int(ep["csum"][row0 + B] - ep["csum"][row0])
        self._ensure_ws(B, nnz)
        call("aae_batch_gather", ptr(ep["indptr"]), ptr(ep["indices"]), ptr(ep["perm"]), C.c_int64(row0), B,
             ptr(self.indptr), ptr(self.indices), ptr(ep["cond"]) if ep["cond"] is not None else None, self.D,
             ptr(self.cond) if ep["cond"] is not None else None, self._stream())
        return B, nnz

    @_on_device
    def corrupt_batch(self, B, p, noise=None):
        """Denoising-autoencoder corruption of the batch in the device buffers (dae.py:48-52): every entry is dropped
        with probability ``p``; ``noise`` = the reference's [B,V] uniform draws (oracle-RNG mode) or None (Philox)."""
        if getattr(self, "_tmp_batch", None) is None or self._tmp_batch.numel() != self._batch.numel():
            self._tmp_batch = torch.empty_like(self._batch)
        self._tmp_batch.copy_(self._batch, non_blocking=True)
        off = self.indices.data_ptr() - self._batch.data_ptr()
        nz = None
        if noise is not None:
            nz = torch.as_tensor(noise, dtype=torch.float32).to(self.dev).contiguous()
            assert nz.shape == (B, self.V)
        call("aae_batch_corrupt", ptr(self._tmp_batch), C.c_void_p(self._tmp_batch.data_ptr() + off), B, self.V,
             C.c_float(p), ptr(nz), ptr(self.state), ptr(self.indptr), ptr(self.indices), self._stream())
        self._keep_alive = nz

    @_on_device
    def set_cond_rows(self, rows_dev, B):
        """Condition rows of the batch (generic conditions, encoded through their Python protocol): device float32
        [B, D] into the step's fixed condition buffer."""
        self._ensure_ws(B, 0)
        self.cond[:B].copy_(rows_dev, non_blocking=True)

    @_on_device
    def snapshot_dec_lin1(self):
        """dec.lin1.weight [H, C+D] as it is before the step (the backward of the step uses it; the step's own Adam
        update overwrites it) -- needed only to hand generic trainable conditions their gradient."""
        n = self.H * self.Cp
        if getattr(self, "_wd1_snap", None) is None:
            self._wd1_snap = torch.empty(n, dtype=torch.float32, device=self.dev)
        self._wd1_snap.copy_(self.dec[:n])

    @_on_device
    def cond_grad(self, B):
        """dL/d(condition rows) [B, D] of the reconstruction phase just run: g_d1 (gradient at dec.lin1's output, written
        by aae_ae_bwd) times the condition columns of the pre-step dec.lin1.weight.  The one torch op on this path; it
        exists only for conditions that train their own parameters (aae.py:703-709)."""
        Wd1 = self._wd1_snap.view(self.H, self.Cp)
        return self.g_d1[:B] @ Wd1[:, self.C:]

    @_on_device
    def set_rng_draws(self, B, draws):
        """Oracle-RNG mode: inject the 12 dropout masks and z_real drawn by torch in the reference's
        order (``oracle.aae_oracle.draw_step_rng``)."""
        order = [("ae_enc", 0), ("ae_enc", 1), ("ae_dec", 0), ("ae_dec", 1), ("disc_real", 0), ("disc_real", 1),
                 ("disc_fake", 0), ("disc_fake", 1), ("gen_enc", 0), ("gen_enc", 1), ("gen_disc", 0), ("gen_disc", 1)]
        have = False
        for i, (k, j) in enumerate(order):
            if k not in draws:      # plain AutoEncoder: only the four masks of the reconstruction phase exist
                continue
            m = draws[k][j]
            if m is not None:
                self.masks[i, :B].copy_(torch.as_tensor(m, dtype=torch.float32), non_blocking=False)
                have = True
        if "z_real" in draws:
            self.z_real[:B].copy_(torch.as_tensor(draws["z_real"], dtype=torch.float32))
        return have

    # ------------------------------------------------------------------ one partial_fit
    def _drops(self, B, injected):
        p1, p2 = self.dropout
        out = {}
        for i, name in enumerate(_DROP_ORDER):
            p = p1 if i % 2 == 0 else p2
            if injected and p > 0:
                out[name] = N.drop(self.masks[i, :B], p, i + 1)
            else:
                out[name] = N.drop(None, p, i + 1)
        return out

    def _branch(self):
        """Context manager: work enqueued inside runs on a second side stream that forks from the current
        stream here and is joined by the next ``_join()`` (a parallel branch of the captured graph)."""
        return _Branch(self)

    def _join(self):
        if self.branches:
            torch.cuda.current_stream(self.dev).wait_event(self._ev_join2)

    def _allreduce(self, t, exchange=0, extra=None):
        """Sum of the shards' partial results, in place: exchange ids 0 (ae-phase h1pre), 1 (dh2 + loss partial),
        2 (disc/gen-phase h1pre), 3 (predict)."""
        if self.world == 1:
            return
        if self.peer is not None:
            if t.numel() > self.peer.n_max:
                raise RuntimeError("exchange message of %d floats exceeds the peer buffers (%d): _ensure_ws must "
                                   "have regrown them" % (t.numel(), self.peer.n_max))
            self.peer.allreduce(t, exchange, extra)
            N.count_launch(1)
            return
        import torch.distributed as dist
        dist.all_reduce(t, group=self.group)
        if extra is not None:
            dist.all_reduce(extra, group=self.group)

    def check_exchange(self):
        """Raise if a peer-memory exchange timed out (its result was poisoned with NaN on the device): called at the
        host's synchronisation points (losses, state export, predict)."""
        if self.peer is not None and self.peer.error():
            raise RuntimeError("aaerec_b200: a peer-memory exchange timed out (a rank died or the ranks diverged); "
                               "the step's results are invalid")

    def close(self):
        """Release the peer-exchange mappings and buffer (item-sharded engines)."""
        if self.peer is not None:
            try:
                torch.cuda.synchronize(self.dev)
                self.peer.close()
            finally:
                self.peer = None

    def __del__(self):
        try:
            self.close()
        except Exception:   # noqa: BLE001 -- interpreter shutdown
            pass

    def _gather_exchange(self, B, out, exchange):
        """h1pre of an item-sharded engine: local partial sums of X.W1^T + all-reduce + bias.  One fused kernel over
        the peer buffers when the batch fits it (<= 256 rows, n_hidden % 4 == 0), else aae_bag_fwd + the exchange."""
        s = self._stream
        if self.peer is not None and B <= 256 and self.H % 4 == 0 and B * self.H <= self.peer.n_max \
                and os.environ.get("AAE_B200_FUSED_GATHER", "1") != "0":
            call("aae_peer_bag_allreduce", self.peer.peers, exchange, ptr(self.indptr), ptr(self.indices), B,
                 ptr(self.W1t), ptr(self.enc), self.H, self.normalize, self.v_begin, self.v_end, ptr(out),
                 C.c_int64(self.peer.n_max), s())
            return
        call("aae_bag_fwd", ptr(self.indptr), ptr(self.indices), B, ptr(self.W1t), ptr(self.enc), self.H, self.normalize,
             self.v_begin, self.v_end, 1 if self.rank == 0 else 0, ptr(out), s())
        self._allreduce(out[:B], exchange)

    def launches_per_step(self):
        """Kernels of ours launched by one train_step (counted while enqueueing; a graph replay
        launches the same kernel nodes)."""
        return self._launches_per_step

    def _enqueue_step(self, B, injected):
        n0 = N.launch_count()
        self._enqueue_step_impl(B, injected)
        self._launches_per_step = N.launch_count() - n0

    def _enqueue_step_impl(self, B, injected):
        """One partial_fit as 15 launches (single GPU), 11 of them on the dependent chain:
        w1_catchup -> [ae_fwd+gather] -> K3 -> ae_bwd -> w1_rows_update || ae_wgrad -> [disc_phase+gather] -> disc_wgrad
        -> [gen_phase+gather] -> w1_rows_update || gen_wgrad -> step_finish, with batch_prepare on a side branch and the
        W1 group sweep (+ its `last` stamp) on a side branch under the step's latency-bound tail.  Item-sharded runs
        gather in a kernel fused with the exchange of the partial sums (aae_peer_bag_allreduce)."""
        ctx = self._phase_ctx(B, injected)
        self._enqueue_ae(ctx)
        if self.adversarial:
            self._enqueue_adversarial(B, ctx["dims"], ctx["bag"], ctx["dr"], ctx["fused"], ctx["cap"], injected)
        self._enqueue_finish(ctx)

    def _phase_ctx(self, B, injected):
        fused = self.world == 1
        lo, hi = self.v_begin, self.v_end
        return dict(B=B, injected=injected, dims=AaeDims(B, self.H, self.C, self.D), dr=self._drops(B, injected),
                    fused=fused, cap=self.uniq.numel(), n_total=float(B) * float(self.V),
                    bag=N.bag(self.indptr, self.indices, self.W1t, self.normalize, lo, hi) if fused else N.bag())

    def _sweep(self):
        call("aae_w1_sweep_blocked", ptr(self.slot_of), self.Vloc, self.H, ptr(self.W1t), ptr(self.W1_m1),
             ptr(self.W1_v1), ptr(self.W1_m2), ptr(self.W1_v2), ptr(self.w1_last), ptr(self.state), ptr(self.ktab),
             self.w1_groups, 0, self.sweep_ctas if self.overlap_sweep else 0, self._stream())

    def _enqueue_ae(self, ctx):
        """ae_step (aae.py:676-711): reconstruction forward, fused decoder output layer, backward, enc_optim and
        dec_optim."""
        s = self._stream
        B, dims, dr, bag, fused, cap = ctx["B"], ctx["dims"], ctx["dr"], ctx["bag"], ctx["fused"], ctx["cap"]
        H = self.H
        st = ptr(self.state)
        lo, hi = self.v_begin, self.v_end
        n_total = ctx["n_total"]
        cur = torch.cuda.current_stream(self.dev)
        # ---- side branch: slots + transposed batch view, then the zero-gradient Adam decay of every row that is
        # not in the batch (both optimizer states, one pass)
        self._ev_fork.record(cur)
        self.side.wait_event(self._ev_fork)
        with torch.cuda.stream(self.side):
            call("aae_batch_prepare", ptr(self.indptr), ptr(self.indices), B, lo, hi, ptr(self.slot_of), ptr(self.uniq),
                 ptr(self.n_uniq), ptr(self.csc_cnt), ptr(self.csc_pos), ptr(self.csc_off), ptr(self.csc_row), cap, s())
            self._ev_prep.record(self.side)
        # rows of this batch: pending zero-gradient steps applied before the encoder reads them
        call("aae_w1_catchup", ptr(self.indptr), ptr(self.indices), B, lo, hi, ptr(self.w1_claim), ptr(self.W1t),
             ptr(self.W1_m1), ptr(self.W1_v1), ptr(self.W1_m2), ptr(self.W1_v2), ptr(self.w1_last), H, st,
             ptr(self.ktab), s())
        if not fused:
            self._gather_exchange(B, self.h1pre, 0)
        call("aae_ae_fwd_bag", dims, bag, ptr(self.h1pre), ptr(self.cond), ptr(self.enc), ptr(self.dec), dr["ae_e1"],
             dr["ae_e2"], dr["ae_d1"], dr["ae_d2"], st, ptr(self.a1), ptr(self.a2), ptr(self.zc), ptr(self.dd1),
             ptr(self.h2), ptr(self.dh2), s())
        self._dec_out_train(B, n_total)
        if self.overlap_sweep:
            # the decoder kernel owns the SMs and starves beside a bandwidth-bound neighbour (measured: 190 -> 375 us),
            # so the sweep runs under the latency-bound tail of the step instead, sized to leave the SMs open
            self._ev_k3.record(cur)
            self.side.wait_event(self._ev_k3)
            with torch.cuda.stream(self.side):
                self._sweep()
        if self.world > 1:
            self._allreduce(self.dh2[:B], 1, self.loss_sums[:1])
        call("aae_ae_bwd", dims, ptr(self.dh2), ptr(self.enc), ptr(self.dec), dr["ae_e1"], dr["ae_e2"], dr["ae_d1"],
             dr["ae_d2"], st, ptr(self.a1), ptr(self.a2), ptr(self.dd1), ptr(self.h2), ptr(self.g_d2), ptr(self.g_d1),
             ptr(self.g_z), ptr(self.g_e2), ptr(self.g_h1), s())
        # the small-layer weight gradients (+ enc_optim / dec_optim, fused into the reduction) and the sparse
        # first-layer update are independent: two branches of the step's graph
        with self._branch():
            call("aae_ae_wgrad", dims, ptr(self.a1), ptr(self.a2), ptr(self.zc), ptr(self.dd1), ptr(self.g_d2),
                 ptr(self.g_d1), ptr(self.g_z), ptr(self.g_e2), ptr(self.g_h1), None, None,
                 N.adam_block(self.enc, self.enc_m1, self.enc_v1, 0),
                 N.adam_block(self.dec, self.dec_m, self.dec_v, 0), st, s())
        cur.wait_event(self._ev_prep)
        call("aae_w1_rows_update", ptr(self.uniq), ptr(self.n_uniq), cap, ptr(self.csc_off), ptr(self.csc_row),
             ptr(self.indptr), self.normalize, ptr(self.g_h1), ptr(self.W1t), ptr(self.W1_m1), ptr(self.W1_v1), H, st,
             0, None if self.adversarial else ptr(self.w1_last), s())
        self._join()

    def _dec_out_train(self, B, n_total):
        """The n_items-wide decoder output layer, fused forward + BCE + backward + dec_optim (K3)."""
        impl = self.impl_for(B)
        need = int(N.load().aae_dec_out_train_work_floats(B, self.H, self.Vloc, impl))
        if need and (self._gwork is None or self._gwork.numel() < need):
            # gradient scratch of the chunked tensor-core path (allocated outside any graph capture: _run warms up
            # eagerly first)
            self._gwork = torch.empty(need, dtype=torch.float32, device=self.dev)
        call("aae_dec_out_train_ws", ptr(self.h2), B, self.H, ptr(self.Wd3), ptr(self.bd3), ptr(self.Wd3_m),
             ptr(self.Wd3_v), ptr(self.bd3_m), ptr(self.bd3_v), self.v_begin, self.Vloc, ptr(self.indptr),
             ptr(self.indices), n_total, ptr(self.state), ptr(self.dh2), ptr(self.loss_sums), impl,
             ptr(self._gwork) if need else None, C.c_int64(need), self._stream())
        if need:
            N.count_launch((B + 103) // 104 - 1)

    def _enqueue_finish(self, ctx):
        cur = torch.cuda.current_stream(self.dev)
        if self.overlap_sweep:
            self._ev_join.record(self.side)
            cur.wait_event(self._ev_join)
        else:
            cur.wait_event(self._ev_prep)
            self._sweep()
        call("aae_step_finish", ptr(self.slot_of), ptr(self.uniq), ptr(self.n_uniq), ctx["cap"], ptr(self.loss_sums), 3,
             ctx["n_total"], ctx["B"], ptr(self.losses), ptr(self.state), ptr(self.ktab), self._stream())

    def _enqueue_adversarial(self, B, dims, bag, dr, fused, cap, injected):
        """disc_step (aae.py:713-732) and gen_step (aae.py:734-743) of one partial_fit."""
        self._enqueue_disc(B, dims, bag, dr, fused, injected)
        self._enqueue_gen(B, dims, bag, dr, cap)

    def _enqueue_disc(self, B, dims, bag, dr, fused, injected):
        """disc_step (aae.py:713-732): eval-mode encoder on the batch, prior sample, discriminator loss, disc_optim.
        Also computes the pre-dropout first encoder layer that gen_step shares (identical weights and input)."""
        s = self._stream
        H, st = self.H, ptr(self.state)
        lo, hi = self.v_begin, self.v_end
        if not fused:
            self._gather_exchange(B, self.h1pre2, 2)
        call("aae_disc_phase_bag", dims, bag, ptr(self.h1pre2), ptr(self.z_real) if injected else None,
             C.c_float(self.prior_scale), ptr(self.enc), ptr(self.disc), dr["disc_r1"], dr["disc_r2"], dr["disc_f1"],
             dr["disc_f2"], st, ptr(self.disc_acts), ptr(self.disc_grads), ptr(self.loss_sums[1:]), s())
        call("aae_disc_wgrad", dims, ptr(self.disc_acts), ptr(self.disc_grads), None,
             N.adam_block(self.disc, self.disc_m, self.disc_v, 1), st, s())

    def _enqueue_gen(self, B, dims, bag, dr, cap):
        """gen_step (aae.py:734-743): train-mode encoder against the updated discriminator, gen_optim."""
        s = self._stream
        H, st = self.H, ptr(self.state)
        call("aae_gen_phase_bag", dims, bag, ptr(self.h1pre2), ptr(self.enc), ptr(self.disc), dr["gen_e1"],
             dr["gen_e2"], dr["gen_q1"], dr["gen_q2"], st, ptr(self.ga1), ptr(self.ga2), ptr(self.gg_z), ptr(self.gg_e2),
             ptr(self.gg_h1), ptr(self.loss_sums[2:]), s())
        with self._branch():
            call("aae_gen_wgrad", dims, ptr(self.ga1), ptr(self.ga2), ptr(self.gg_z), ptr(self.gg_e2),
                 ptr(self.gg_h1), None, N.adam_block(self.enc, self.enc_m2, self.enc_v2, 1), st, s())
        call("aae_w1_rows_update", ptr(self.uniq), ptr(self.n_uniq), cap, ptr(self.csc_off), ptr(self.csc_row),
             ptr(self.indptr), self.normalize, ptr(self.gg_h1), ptr(self.W1t), ptr(self.W1_m2), ptr(self.W1_v2), H, st,
             1, ptr(self.w1_last), s())
        self._join()

    # ------------------------------------------------------------------ the three phases as separate calls
    @_on_device
    def phase_step(self, phase, B, injected=False):
        """ae_step / disc_step / gen_step of the reference (aae.py:676-743) as separate, eager calls on the batch in the
        device buffers.  The four Adam optimizers share one step counter (they all step once per partial_fit,
        aae.py:745-766), so the phases must be called in the reference's order ae -> disc -> gen; the counter advances
        after gen (after ae for the plain AutoEncoder).  Returns the phase's loss (synchronises)."""
        order = ("ae", "disc", "gen") if self.adversarial else ("ae",)
        want = order[self._phase_cursor]
        if phase != want:
            raise RuntimeError("phase %r called out of order (expected %r): the optimizers share one Adam step "
                               "counter, so ae_step, disc_step, gen_step run in partial_fit's order" % (phase, want))
        if phase == "ae":
            self._phase_ctx_live = self._phase_ctx(B, injected)
        ctx = self._phase_ctx_live
        if ctx is None or ctx["B"] != B:
            raise RuntimeError("phase %r: batch differs from the one ae_step saw" % (phase,))
        idx = order.index(phase)
        if phase == "ae":
            self._enqueue_ae(ctx)
        elif phase == "disc":
            self._enqueue_disc(B, ctx["dims"], ctx["bag"], ctx["dr"], ctx["fused"], injected)
        else:
            self._enqueue_gen(B, ctx["dims"], ctx["bag"], ctx["dr"], ctx["cap"])
        denom = ctx["n_total"] if phase == "ae" else float(B)
        loss = float(self.loss_sums[idx].item()) / denom
        self._phase_cursor = (self._phase_cursor + 1) % len(order)
        if self._phase_cursor == 0:
            self._enqueue_finish(ctx)
            self._phase_ctx_live = None
            self.steps_done += 1
            self._w1_dirty = True
        self._wp_dirty = True
        return loss

    def _run(self, key, enqueue):
        """Enqueue ``enqueue()`` eagerly, or (graph mode) capture it once per ``key`` and replay the graph."""
        if not self.use_graph:
            enqueue()
            return
        g = self._graphs.get(key)
        if g is None:
            # warm up once eagerly so that lazy module loading / attribute setting is done
            snap = self._snapshot()
            enqueue()
            torch.cuda.synchronize(self.dev)
            self._restore(snap)
            g = torch.cuda.CUDAGraph()
            # no cyclic garbage collection while capturing: collecting an old engine's CUDA graph in the
            # middle of a capture invalidates it (torch collects once on entering the capture)
            gc_was_on = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.graph(g, stream=self._cap_stream):
                    enqueue()
            finally:
                if gc_was_on:
                    gc.enable()
            self._restore(snap)
            self._graphs[key] = g
        g.replay()

    @_on_device
    def train_step(self, B, injected=False):
        """Enqueue one partial_fit on the batch currently in the device batch buffers.  Losses
        (R, D, G) land in ``self.losses`` (device float32[3])."""
        if B <= 0:
            return
        if self.inference_only:
            raise RuntimeError("this engine was built inference_only (a predict replica): it cannot train")
        self._run((B, bool(injected)), lambda: self._enqueue_step(B, injected))
        self.steps_done += 1
        self._w1_dirty = True
        self._wp_dirty = True

    @_on_device
    def train_step_host(self, indptr_np, indices_np, cond_np=None, injected=False, rng_draws=None,
                        cond_on_device=False):
        """One partial_fit straight from host CSR rows (int32, row-relative indptr): the end-to-end entry.  The batch
        is written into one of two pinned slots and moved with one H2D copy; the step's CUDA graph itself pushes the
        three losses back into the slot's pinned ``losses`` (``aae_copy_words_sel``) -- no D2H hop behind the step.  Returns the slot: ``slot['losses']`` is valid once ``slot['ev']`` has completed;
        ``slot['prev_losses']`` holds the (complete) losses of the step that used the slot before, two steps ago."""
        B = int(indptr_np.shape[0]) - 1
        nnz = int(indptr_np[-1])
        if B <= 0:
            return None
        if self.inference_only:
            raise RuntimeError("this engine was built inference_only (a predict replica): it cannot train")
        self._ensure_ws(B, nnz)
        si = self.steps_done & 1          # the graph's copy kernels pick the slot from the device step counter: t = steps_done + 1
        slot = self._zc[si]
        slot["prev_losses"] = None
        if slot["ev"] is not None:
            slot["ev"].synchronize()           # the launch that last read this slot is done ...
            slot["prev_losses"] = slot["losses"][:3].clone()     # ... and these are its losses (step i-2)
        off = self._zc_off
        pk = slot["packed"].numpy()
        pk[: B + 1] = indptr_np
        pk[off: off + nnz] = indices_np[:nnz]
        host_cond = bool(self.D) and not cond_on_device     # else: set_cond_rows already filled the condition buffer
        if host_cond:
            slot["cond"][:B].numpy()[:] = cond_np
        if rng_draws is not None:
            self.set_rng_draws(B, rng_draws)

        z0, z1, st = self._zc[0], self._zc[1], ptr(self.state)
        # batch in: ONE copy-engine transfer of the packed slot (a kernel reading the mapped slot over PCIe was measured
        # at ~100 MB/s: +120 us per 8 KB batch); losses out: written into the slot's pinned memory by the graph itself
        call("aae_upload_batch", ptr(slot["packed"]), ptr(slot["packed"][off:]), B, nnz, ptr(self.indptr),
             ptr(self.indices), self._stream())
        if host_cond:
            self.cond[:B].copy_(slot["cond"][:B], non_blocking=True)

        def enqueue():
            self._enqueue_step(B, injected)
            call("aae_copy_words_sel", ptr(self.losses), ptr(self.losses), ptr(z0["losses"]), ptr(z1["losses"]), 3, st, 0,
                 self._stream())
        self._run((B, bool(injected), "host"), enqueue)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        slot["ev"] = ev
        self.steps_done += 1
        self._w1_dirty = True
        self._wp_dirty = True
        return slot

    @_on_device
    def flush_w1(self):
        """Apply every pending zero-gradient Adam step to W1t (time-blocked policy): after this the weights are
        exactly those of dense Adam after ``steps_done`` steps.  Needed before reading rows outside a training
        step (predict, weight export)."""
        if self._w1_dirty:
            call("aae_w1_sweep_blocked", None, self.Vloc, self.H, ptr(self.W1t), ptr(self.W1_m1), ptr(self.W1_v1),
                 ptr(self.W1_m2), ptr(self.W1_v2), ptr(self.w1_last), ptr(self.state), ptr(self.ktab), self.w1_groups,
                 1, 0, self._stream())
            self._w1_dirty = False

    def _snapshot(self):
        names = ("W1t", "W1_m1", "W1_v1", "W1_m2", "W1_v2", "Wd3", "Wd3_m", "Wd3_v", "bd3", "bd3_m", "bd3_v",
                 "enc", "enc_m1", "enc_v1", "enc_m2", "enc_v2", "dec", "dec_m", "dec_v", "disc", "disc_m", "disc_v",
                 "state", "w1_last", "w1_claim", "ktab", "loss_sums")
        torch.cuda.synchronize(self.dev)
        return {n: getattr(self, n).clone() for n in names}

    def _restore(self, snap):
        torch.cuda.synchronize(self.dev)
        for n, v in snap.items():
            getattr(self, n).copy_(v)
        torch.cuda.synchronize(self.dev)

    # ------------------------------------------------------------------ predict
    @_on_device
    def predict_h2(self, B):
        """eval-mode encoder + condition + decoder head for the batch in the device buffers."""
        self.flush_w1()
        dims = AaeDims(B, self.H, self.C, self.D)
        if self.world == 1:
            bag = N.bag(self.indptr, self.indices, self.W1t, self.normalize, self.v_begin, self.v_end)
        else:
            bag = N.bag()
            self._gather_exchange(B, self.h1pre, 3)
        call("aae_predict_tail_bag", dims, bag, ptr(self.h1pre), ptr(self.cond), ptr(self.enc), ptr(self.dec),
             ptr(self.h2), self._stream())
        return self.h2[:B]

    @_on_device
    def scores(self, B, out, apply_sigmoid=True):
        """out[B, >=Vloc] <- sigmoid probabilities (reference predict) or logits of the local items."""
        self.predict_h2(B)
        call("aae_dec_out_scores", ptr(self.h2), B, self.H, ptr(self.Wd3), ptr(self.bd3), self.Vloc,
             1 if apply_sigmoid else 0, ptr(out), out.stride(0), self.impl_for_scores(), self._stream())
        return out

    @_on_device
    def gold_ranks(self, B, gold_indptr, gold_indices, scratch=None, mask_known=True, filt=None):
        """Ranks (1-based) of the gold items of the batch in the device buffers, in the descending order of
        remove_non_missing(predict(X), X) (known items at the bottom; ties by lower item id): int64 host array aligned
        with ``gold_indices``.  ``gold_indptr`` [B+1] / ``gold_indices``: CSR of the held-out items (global ids).
        The [B, V] score matrix lives in HBM only (never on the host).

        ``filt`` (``filters.RankFilter`` of the B rows): ranks in the full filtered ranking (``predict_topk(X, None,
        items=, exclude=)``) -- only the eligible items, never an excluded (row, item) pair.  The caller passes only returnable gold
        (eligible, not excluded for its row).  Each shard scores the compact copy of its eligible rows (``_compact``,
        the copy ``topk`` ranks) into ``scratch`` and counts with ``aae_rank_counts_filtered``; a shard whose items are
        all eligible counts on its own columns, with the exclusions only; a shard without an eligible item launches
        neither but still takes part in the encoder exchange and both all-reduces."""
        n_gold = int(gold_indptr[-1])
        if n_gold == 0:
            return np.zeros(0, dtype=np.int64)
        ids = excl = None
        if filt is not None:
            ids = filt.shard_ids(self.V, self.rank, self.world)
            excl = filt.exclude if filt.exclude is not None and filt.exclude.nnz else None   # rows without any
        gp = torch.from_numpy(np.ascontiguousarray(gold_indptr, dtype=np.int32)).to(self.dev)
        gi = torch.from_numpy(np.ascontiguousarray(gold_indices, dtype=np.int32)).to(self.dev)
        zg = torch.empty(n_gold, dtype=torch.float32, device=self.dev)
        cnt = torch.zeros(n_gold, dtype=torch.int32, device=self.dev)
        if ids is None and excl is None:        # unfiltered, or every item of this shard eligible without exclusions
            n, vb, fn, extra = self.Vloc, self.v_begin, "aae_rank_counts", ()
            if scratch is None or scratch.shape[0] < B or scratch.shape[1] < n:
                scratch = torch.empty(B, n, dtype=torch.float32, device=self.dev)
            self.scores(B, scratch, apply_sigmoid=False)
        else:
            # first, on every path: on item shards predict_h2 is a collective (the h1pre exchange)
            self.predict_h2(B)
            if ids is not None and ids.size == 0:
                n = 0
                zg.fill_(float("nan"))          # no gold of this shard: contributes 0 to the summed scores
            else:
                if ids is None:
                    W, b, n, vb, ids_dev = self.Wd3, self.bd3, self.Vloc, self.v_begin, None
                else:
                    c = self._compact(ids)
                    W, b, n, vb, ids_dev = c["Wd3c"], c["bd3c"], c["A"], 0, c["ids"]
                if scratch is None or scratch.shape[0] < B or scratch.shape[1] < n:
                    scratch = torch.empty(B, n, dtype=torch.float32, device=self.dev)
                call("aae_dec_out_scores", ptr(self.h2), B, self.H, ptr(W), ptr(b), n, 0, ptr(scratch),
                     scratch.stride(0), self.impl_for_scores(), self._stream())
                xp, xi = self._upload_exclusions(excl) if excl is not None else (None, None)
                fn, extra = "aae_rank_counts_filtered", (C.byref(N.AaeRankFilter(ptr(ids_dev), ptr(xp), ptr(xi))),)

        def run(given):
            if n == 0:
                return
            call(fn, ptr(scratch), scratch.stride(0), B, n, vb,
                 ptr(self.indptr) if (mask_known and not given) else None,
                 ptr(self.indices) if (mask_known and not given) else None, ptr(gp), ptr(gi), n_gold, ptr(zg),
                 1 if given else 0, ptr(cnt), self._stream(), *extra)
        run(False)
        if self.world > 1:
            import torch.distributed as dist
            zg.copy_(torch.nan_to_num(zg, nan=0.0))
            dist.all_reduce(zg, group=self.group)
            run(True)
            dist.all_reduce(cnt, group=self.group)
        return cnt.cpu().numpy().astype(np.int64) + 1

    def _padded_weights(self):
        """Wp = [Wd3 | bd3 | 0 0 0] as [Vloc, 104] (+ its largest row norm): the TMA-described operand of the v2 predict
        filter, rebuilt only after the weights changed (one streaming pass, amortised over all query batches)."""
        n = int(N.load().aae_pad_weights_floats(self.Vloc, self.H))
        if n == 0:
            return None, None
        if self._wp is None or self._wp.numel() < n:
            self._wp = torch.empty(n, dtype=torch.float32, device=self.dev)
            self._wp_dirty = True
        wmax = self._wp[n - 64:]
        if self._wp_dirty:
            call("aae_pad_weights", ptr(self.Wd3), ptr(self.bd3), self.Vloc, self.H, ptr(self._wp), ptr(wmax),
                 self._stream())
            self._wp_dirty = False
        return self._wp, wmax

    @_on_device
    def topk(self, B, k, scratch=None, mask_known=True, fused=None, check=True, filt=None, _out=None):
        """Masked top-k of the batch in the device buffers: returns (idx int32 [B,k] global item ids,
        val float32 [B,k] logits), descending.  Item-sharded: local top-k + all-gather + merge.

        Large shards take the fused path: candidates selected in the GEMM epilogue, no [B, Vloc] score matrix.
        ``aae_predict_topk2`` (TMA-multicast single-pass TF32 filter + exact fp32 re-scoring of the survivors) when
        the shape is inside its envelope, else ``aae_predict_topk`` (3xTF32 throughout).  The per-batch status word is
        read back (one 4-byte synchronising copy) and a batch the fused path could not rank exactly is redone through
        the dense path; ``check=False`` skips that read (the caller inspects ``topk_status()`` later -- pipelined
        callers and the device-timed benchmark loop).  ``fused=False`` forces the dense path.

        ``filt`` (``filters.RankFilter`` of the B rows): only the eligible items are ranked, excluded (row, item) pairs
        are never returned, and rows with fewer than k returnable items end in (-1, -inf) padding.  Each shard ranks the
        compact copy of its eligible rows (``_compact``) through the same paths, chosen by the number of eligible items;
        a shard whose items are all eligible, with no exclusions, runs the unfiltered path."""
        kl = min(k, self.Vloc)
        if _out is not None:        # a filtered call's shard ranked unfiltered: into that call's result buffers
            idx, val = _out
        else:
            # results land in a ring of four preallocated buffers (no allocation in the query loop); a result stays
            # valid for the next three topk calls
            if self._topk_out is None or self._topk_out[0][0].shape[0] < B or self._topk_out[0][0].shape[1] != kl:
                self._topk_out = [(torch.empty(max(B, 1), kl, dtype=torch.int32, device=self.dev),
                                   torch.empty(max(B, 1), kl, dtype=torch.float32, device=self.dev))
                                  for _ in range(4)]
                self._topk_i = 0
            self._topk_i = (self._topk_i + 1) % 4
            idx, val = self._topk_out[self._topk_i][0][:B], self._topk_out[self._topk_i][1][:B]
        if filt is not None:
            ids = filt.shard_ids(self.V, self.rank, self.world)
            excl = filt.exclude if filt.exclude is not None and filt.exclude.nnz else None   # rows without any
            if ids is not None or excl is not None:
                self._topk_filtered(B, kl, idx, val, scratch, mask_known, fused, check, ids, excl)
            else:       # every item of this shard eligible, no exclusions: the unfiltered shard ranking
                self.topk(B, kl, scratch=scratch, mask_known=mask_known, fused=fused, check=check, _out=(idx, val))
            if self.world == 1:
                return idx, val
            oi, ov = self._merge_shards(B, k, idx, val, pad=-float("inf"))
            ov.masked_fill_(oi < 0, -float("inf"))
            return oi, ov
        impl = self.impl_for_scores()
        lib = N.load()
        mode, need = None, 0
        want = os.environ.get("AAE_B200_TOPK", "")
        if fused is not False and impl in (1, 2) and want != "dense":
            if impl == 1 and want != "v1":
                need = int(lib.aae_predict_topk2_work_bytes(B, self.Vloc, kl, self.H))
                mode = "v2" if need > 0 else None
            if mode is None:
                need = int(lib.aae_predict_topk_work_bytes(B, self.Vloc, kl))
                mode = "v1" if need > 0 else None
        done = False
        if mode is not None:
            if self._topk_work is None or self._topk_work.numel() < need:
                self._topk_work = torch.empty(need, dtype=torch.uint8, device=self.dev)
            self.predict_h2(B)
            ip = ptr(self.indptr) if mask_known else None
            ii = ptr(self.indices) if mask_known else None
            if mode == "v2":
                wp, wmax = self._padded_weights()
                call("aae_predict_topk2", ptr(self.h2), B, self.H, ptr(self.Wd3), ptr(self.bd3), ptr(wp), ptr(wmax),
                     self.Vloc, self.v_begin, ip, ii, kl, ptr(self._topk_work), need, ptr(idx), ptr(val),
                     ptr(self._n_bad), self._stream())
            else:
                call("aae_predict_topk", ptr(self.h2), B, self.H, ptr(self.Wd3), ptr(self.bd3), self.Vloc, self.v_begin,
                     ip, ii, kl, impl, ptr(self._topk_work), need, ptr(idx), ptr(val), ptr(self._n_bad), self._stream())
            self.topk_mode = mode
            if check:
                done = int(self._n_bad.item()) == 0
                self.topk_fallbacks += 0 if done else 1
            else:
                done = True
        if not done:
            self.topk_mode = "dense"
            if scratch is None or scratch.shape[0] < B or scratch.shape[1] < self.Vloc:
                scratch = torch.empty(B, self.Vloc, dtype=torch.float32, device=self.dev)
            self.scores(B, scratch, apply_sigmoid=False)
            call("aae_masked_topk", ptr(scratch), scratch.stride(0), B, self.Vloc, self.v_begin,
                 ptr(self.indptr) if mask_known else None, ptr(self.indices) if mask_known else None, kl, ptr(idx),
                 ptr(val), None, self._stream())
        if _out is not None or self.world == 1:
            return idx, val
        return self._merge_shards(B, k, idx, val)

    def _compact(self, ids):
        """Compact copy of this shard's eligible rows of the output layer: Wd3c [A,H] / bd3c [A] for the ascending
        global ids ``ids`` (int32 numpy), with the device id table.  Cached: rebuilt when the eligible set or the
        weights change (the padded Wp of the compact copy follows it lazily, ``_compact_padded``)."""
        c = self._cmp
        if c is not None and c["ver"] == self._wver and np.array_equal(c["ids_host"], ids):
            return c
        A = int(ids.size)
        if c is None or c["cap"] < A:
            cap = max(A, 1)
            self._cmp = c = None    # free the old copy before the new one is allocated
            c = dict(cap=cap, Wd3c=torch.empty(cap, self.H, dtype=torch.float32, device=self.dev),
                     bd3c=torch.empty(cap, dtype=torch.float32, device=self.dev),
                     ids=torch.empty(cap, dtype=torch.int32, device=self.dev), wp=None)
        c.update(A=A, ids_host=ids.copy(), ver=self._wver, wp_ok=False)
        if A:
            c["ids"][:A].copy_(torch.from_numpy(ids))
            call("aae_gather_item_rows", ptr(self.Wd3), ptr(self.bd3), self.H, self.Vloc, self.v_begin, ptr(c["ids"]), A,
                 ptr(c["Wd3c"]), ptr(c["bd3c"]), ptr(self._n_bad), self._stream())
            bad = int(self._n_bad.item())       # once per rebuild of the copy
            if bad:
                self._cmp = None
                raise ValueError("%d of %d eligible ids are outside this shard's items [%d, %d) or not ascending"
                                 % (bad, A, self.v_begin, self.v_end))
        self._cmp = c
        return c

    def _compact_padded(self, c):
        """``_padded_weights`` of the compact copy: Wp [A,104] and its largest row norm, so that the TF32 margin of the
        v2 filter is that of exactly the rows being ranked."""
        n = int(N.load().aae_pad_weights_floats(c["A"], self.H))
        if c["wp"] is None or c["wp"].numel() < n:
            c["wp"] = torch.empty(n, dtype=torch.float32, device=self.dev)
            c["wp_ok"] = False
        wmax = c["wp"][n - 64:]
        if not c["wp_ok"]:
            call("aae_pad_weights", ptr(c["Wd3c"]), ptr(c["bd3c"]), c["A"], self.H, ptr(c["wp"]), ptr(wmax),
                 self._stream())
            c["wp_ok"] = True
        return c["wp"], wmax

    def _upload_exclusions(self, X):
        """Exclusion CSR of the batch (scipy, B rows) -> device (indptr, indices): one H2D copy from pinned staging,
        both buffers grown geometrically (no allocation per batch)."""
        B, nnz = X.shape[0], X.nnz
        n = B + 1 + nnz
        st = self._xstage
        if st is None or st["cap"] < n:
            cap = n if st is None else max(n, int(1.5 * st["cap"]))
            if st is not None and st["ev"] is not None:
                st["ev"].synchronize()
            st = self._xstage = dict(cap=cap, pin=torch.empty(cap, dtype=torch.int32).pin_memory(),
                                     dev=torch.empty(cap, dtype=torch.int32, device=self.dev), ev=None)
        if st["ev"] is not None:
            st["ev"].synchronize()      # the previous batch's copy has left the pinned buffer
        host = st["pin"].numpy()
        host[: B + 1] = X.indptr
        host[B + 1: n] = X.indices
        st["dev"][:n].copy_(st["pin"][:n], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        st["ev"] = ev
        return st["dev"][: B + 1], st["dev"][B + 1: n]

    def _topk_filtered(self, B, kl, idx, val, scratch, mask_known, fused, check, ids, exclude):
        """Local ranking of one shard under a filter (see ``topk``): ``ids`` = the shard's eligible global ids (None:
        all of them), ``exclude`` = the batch's exclusion CSR (None: none).  Same path choice as the unfiltered call,
        on the number of eligible items A: fused v2 / v1 when A is inside their envelope (A >= 32641), else the dense
        scores of the A columns + aae_masked_topk_filtered; A = 0 gives an all-padding list without a launch of the
        ranking."""
        # first, on every path: on item shards predict_h2 is a collective (the h1pre exchange), so a shard without
        # eligible items must still take part in it
        self.predict_h2(B)
        if ids is not None and ids.size == 0:
            idx.fill_(-1)
            val.fill_(-float("inf"))
            self.topk_mode = "empty"
            return
        if ids is None:
            W, b, n, vb, ids_dev = self.Wd3, self.bd3, self.Vloc, self.v_begin, None
        else:
            c = self._compact(ids)
            W, b, n, vb, ids_dev = c["Wd3c"], c["bd3c"], c["A"], 0, c["ids"]
        xp, xi = self._upload_exclusions(exclude) if exclude is not None else (None, None)
        filt = N.AaeRankFilter(ptr(ids_dev), ptr(xp), ptr(xi))
        ip = ptr(self.indptr) if mask_known else None
        ii = ptr(self.indices) if mask_known else None
        impl = self.impl_for_scores()
        lib = N.load()
        mode, need = None, 0
        want = os.environ.get("AAE_B200_TOPK", "")
        if fused is not False and impl in (1, 2) and want != "dense":
            if impl == 1 and want != "v1":
                need = int(lib.aae_predict_topk2_work_bytes(B, n, kl, self.H))
                mode = "v2" if need > 0 else None
            if mode is None:
                need = int(lib.aae_predict_topk_work_bytes(B, n, kl))
                mode = "v1" if need > 0 else None
        done = False
        if mode is not None:
            if self._topk_work is None or self._topk_work.numel() < need:
                self._topk_work = torch.empty(need, dtype=torch.uint8, device=self.dev)
            if mode == "v2":
                wp, wmax = self._padded_weights() if ids is None else self._compact_padded(c)
                call("aae_predict_topk2_filtered", ptr(self.h2), B, self.H, ptr(W), ptr(b), ptr(wp), ptr(wmax), n, vb,
                     ip, ii, kl, ptr(self._topk_work), need, ptr(idx), ptr(val), ptr(self._n_bad), self._stream(),
                     C.byref(filt))
            else:
                call("aae_predict_topk_filtered", ptr(self.h2), B, self.H, ptr(W), ptr(b), n, vb, ip, ii, kl, impl,
                     ptr(self._topk_work), need, ptr(idx), ptr(val), ptr(self._n_bad), self._stream(), C.byref(filt))
            self.topk_mode = mode
            if check:
                done = int(self._n_bad.item()) == 0
                self.topk_fallbacks += 0 if done else 1
            else:
                done = True
        if not done:
            self.topk_mode = "dense"
            if scratch is None or scratch.shape[0] < B or scratch.shape[1] < n:
                scratch = torch.empty(B, n, dtype=torch.float32, device=self.dev)
            call("aae_dec_out_scores", ptr(self.h2), B, self.H, ptr(W), ptr(b), n, 0, ptr(scratch), scratch.stride(0),
                 impl, self._stream())
            call("aae_masked_topk_filtered", ptr(scratch), scratch.stride(0), B, n, vb, ip, ii, kl, ptr(idx), ptr(val),
                 None, self._stream(), C.byref(filt))

    @_on_device
    def compact_scores(self, B, ids):
        """Logits of the batch in the device buffers for the eligible items ``ids`` only (ascending global ids, world
        1): ([B, A] scores, device id table) -- the full-ranking path under a candidate filter."""
        c = self._compact(ids)
        out = torch.empty(B, max(c["A"], 1), dtype=torch.float32, device=self.dev)
        if c["A"]:
            self.predict_h2(B)
            call("aae_dec_out_scores", ptr(self.h2), B, self.H, ptr(c["Wd3c"]), ptr(c["bd3c"]), c["A"], 0, ptr(out),
                 out.stride(0), self.impl_for_scores(), self._stream())
        return out[:, : c["A"]], c["ids"][: c["A"]]

    def _merge_shards(self, B, k, idx, val, pad=-3.0e38):
        """Item shards -> global top-k: all-gather of the [B, kpad] per-shard lists into preallocated [world, B, kpad]
        buffers, then one merge kernel that reads that layout directly (no torch repacking in the query loop)."""
        import torch.distributed as dist
        kmax = min(k, (self.V + self.world - 1) // self.world)
        kk = min(k, self.V)
        kl = idx.shape[1]
        key = (B, kmax, kk)
        mb = getattr(self, "_merge_bufs", None)
        if mb is None or mb["key"] != key:
            mb = dict(key=key,
                      pv=torch.full((B, kmax), -3.0e38, dtype=torch.float32, device=self.dev),
                      pi=torch.full((B, kmax), -1, dtype=torch.int32, device=self.dev),
                      gv=torch.empty(self.world, B, kmax, dtype=torch.float32, device=self.dev),
                      gi=torch.empty(self.world, B, kmax, dtype=torch.int32, device=self.dev),
                      out=[(torch.empty(B, kk, dtype=torch.int32, device=self.dev),
                            torch.empty(B, kk, dtype=torch.float32, device=self.dev)) for _ in range(4)], i=0)
            self._merge_bufs = mb
        if kl == kmax:
            pv, pi = val.contiguous(), idx.contiguous()
        else:                                   # a last shard smaller than k: pad its list
            mb["pv"][:, :kl].copy_(val)
            if mb.get("pad", -3.0e38) != pad:       # filtered calls pad with -inf
                mb["pv"][:, kl:].fill_(pad)
                mb["pad"] = pad
            mb["pi"][:, :kl].copy_(idx)
            pv, pi = mb["pv"], mb["pi"]
        dist.all_gather_into_tensor(mb["gv"], pv, group=self.group)
        dist.all_gather_into_tensor(mb["gi"], pi, group=self.group)
        mb["i"] = (mb["i"] + 1) % 4
        oi, ov = mb["out"][mb["i"]]
        if self.world * kmax <= 2048:
            call("aae_topk_merge_seg", ptr(mb["gv"]), ptr(mb["gi"]), self.world, B, kmax, kk, ptr(oi), ptr(ov),
                 self._stream())
        else:
            cv = mb["gv"].permute(1, 0, 2).reshape(B, -1).contiguous()
            ci = mb["gi"].permute(1, 0, 2).reshape(B, -1).contiguous()
            call("aae_topk_merge", ptr(cv), ptr(ci), B, cv.shape[1], kk, ptr(oi), ptr(ov), self._stream())
        return oi, ov

    def topk_status(self):
        """Rows the last fused ``topk(check=False)`` could not rank exactly (0 = the result is exact); synchronises."""
        return int(self._n_bad.item())
