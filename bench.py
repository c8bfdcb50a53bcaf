#!/usr/bin/env python
"""bench.py -- AAE train item-sets/s and top-100 predict sets/s (BASELINE.json metric).

A "step" is one ``partial_fit`` (reconstruction + discriminator + generator phases, all four Adam updates) over
one batch of synthetic item sets, n_hidden 100, n_code 50.  The headline workload is the MPD-shaped configuration
(BASELINE configs[3]: V = 2,000,000 items, batch 100, item-sharded over the N GPUs of the box); the PubMed-shaped
configuration (configs[1]) and the other configs are extra legs of the same JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu]
                  [--workload mpd|pubmed|econbiz] [--dump-outputs DIR]

Prints ONE JSON line.  ``value`` = sets/s with the batches already resident in HBM (device-timed with CUDA events,
exactly K steps, max over ranks); ``e2e`` = the same through the host-buffer entry ``partial_fit`` calls (pinned CSR
batch H2D + losses D2H every step inside the timed region); ``roofline`` = the dominant kernel's algorithmic bytes /
its own CUDA-event time against MEASURED_PEAKS.json; ``cpu_baseline`` = the reference's own
``AdversarialAutoEncoder.fit`` (unmodified copy under oracle/_ref, CUDA hidden, all host threads) on a bounded sample;
``gpu_baseline`` = the same unmodified reference on the B200 through stock PyTorch; ``w1_all_rows_hot`` = the headline
steps again with live Adam moments in every first-layer row (no cold row: the worst case of the time-blocked W1 sweep,
DESIGN.md 4); the predict legs carry ``cpu_baseline`` = the reference's predict + remove_non_missing + argtopk on the
host cores (internal ``--impl reference-predict``).

``--impl reference`` times the reference's CPU path alone (rank 0 only) and prints the same line with
``"impl": "reference"``.  ``--steps K`` is exactly the number of timed steps of ``--impl ours``; the reference arm runs
at most K and stops earlier once ``--budget`` seconds of timed work are spent (its CPU-port fallback without the
reference package: at most 20), and reports the steps it timed in ``steps_timed``.

``--dump-outputs DIR`` writes what the headline's last timed step computed into ``DIR/<name>.npy`` (float32): its three
losses and the weights after it, the item-indexed ones on a fixed sample of items (see ``dump_outputs``).  Inputs,
initial weights and dropout draws are seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "aae-recommender_b200"))

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (V, mean_len, min_len, max_len, data_seed, B, BASELINE.json config)
    "pubmed": (200000, 16, 2, 200, 1, 100, "configs[1]"),
    "econbiz": (4587, 5, 2, 30, 0, 100, "configs[0]"),
    "mpd": (2000000, 66, 5, 250, 3, 100, "configs[3]"),
}
H, C = 100, 50


def workload_string(name, B=None):
    """The ONE description of a training workload that both arms print (same_config)."""
    V, mean_len, lo, hi, seed, B0, cfg = WORKLOADS[name]
    return ("%s-shaped (BASELINE %s): V=%d items, batch %d sets, set sizes clip(Poisson(%d),%d,%d) with Zipf(1.0) items "
            "drawn with replacement then de-duplicated (seed %d), n_hidden %d, n_code %d, dropout (.2,.2), "
            "one partial_fit (ae+disc+gen, four Adam updates) per step"
            % (name, cfg, V, B or B0, mean_len, lo, hi, seed, H, C))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [x.strip() for x in out.stdout.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm, reasons, smax = [], set(), None
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_batches(workload, n_batches, cond_dim=0, B=None):
    from aaerec_b200.synth import synth_sets, synth_condition
    V, mean_len, lo, hi, seed, B0, _ = WORKLOADS[workload]
    B = B or B0
    X = synth_sets(n_batches * B, V, mean_len, lo, hi, seed)
    cond = synth_condition(n_batches * B, cond_dim) if cond_dim else None
    batches = []
    for i in range(n_batches):
        s, e = int(X.indptr[i * B]), int(X.indptr[(i + 1) * B])
        ip = (X.indptr[i * B:(i + 1) * B + 1] - s).astype(np.int32)
        batches.append((ip, X.indices[s:e].astype(np.int32), cond[i * B:(i + 1) * B] if cond_dim else None))
    return X, batches, V, B


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own implementation of the path (oracle/_ref = unmodified copy of aaerec/), timed
# through its public API (AdversarialAutoEncoder.fit -> partial_fit), on the CPU (CUDA hidden) or on the GPU
# ------------------------------------------------------------------------------------------------------------------
class _Enough(Exception):
    pass


def _host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def reference_fit_timed(workload, K, W, use_cuda, budget_s):
    """Run the unmodified reference's fit() on (W+K) batches of the workload; returns (steps timed, seconds, kind).
    Time runs from the entry of partial_fit number W to the end of the last timed one, so it includes the reference's
    own batch slicing + toarray() between the steps (its stock host feed), not the epoch shuffle.  Stops early (at
    least 2 timed steps) once ``budget_s`` seconds of timed work are spent."""
    import torch
    from oracle import reference_loader as RL
    V, mean_len, lo, hi, seed, B, _ = WORKLOADS[workload]
    from aaerec_b200.synth import synth_sets
    X = synth_sets((K + W) * B, V, mean_len, lo, hi, seed)
    if not RL.reference_available():
        return None
    ref = RL.load_reference()
    if use_cuda:
        # "what you get today by just having a GPU": stock PyTorch, true fp32 like the reference's CPU numerics
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    model = ref.aae.AdversarialAutoEncoder(n_hidden=H, n_code=C, n_epochs=1, batch_size=B, verbose=False)
    stamps = []
    orig = model.partial_fit

    def sync():
        if use_cuda:
            torch.cuda.synchronize()

    def timed(*a, **kw):
        sync()
        now = time.perf_counter()
        stamps.append(now)
        n_timed = len(stamps) - 1 - W
        if n_timed >= 2 and now - stamps[W] > budget_s:
            raise _Enough()
        return orig(*a, **kw)
    model.partial_fit = timed
    torch.manual_seed(42)
    np.random.seed(42)
    import contextlib
    try:
        with contextlib.redirect_stdout(sys.stderr):     # the reference prints its code size: keep stdout for the JSON line
            model.fit(X)
        sync()
        stamps.append(time.perf_counter())
    except _Enough:
        pass
    steps = len(stamps) - 1 - W
    return steps, stamps[-1] - stamps[W], "reference"


def reference_predict_timed(workload, n_query, use_cuda, k=100):
    """The unmodified reference's ranking chain on ``n_query`` query sets of the workload: model.predict (aae.py:840-870,
    dense [n,V] probabilities) -> remove_non_missing (evaluation.py:183-199, as the harness calls it, evaluation.py:375)
    -> argtopk(., k) (evaluation.py:20-58).  Returns seconds (None without oracle/_ref)."""
    import torch
    from oracle import reference_loader as RL
    from aaerec_b200.synth import synth_sets
    if not RL.reference_available():
        return None
    V, mean_len, lo, hi, seed, B, _ = WORKLOADS[workload]
    ref = RL.load_reference()
    if use_cuda:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    model = ref.aae.AdversarialAutoEncoder(n_hidden=H, n_code=C, n_epochs=1, batch_size=B, verbose=False)
    torch.manual_seed(42)
    np.random.seed(42)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):
        model.fit(synth_sets(B, V, mean_len, lo, hi, seed))      # one step: builds the modules (and warms torch up)
    if workload == "mpd":
        Xq = synth_sets(n_query, V, 25, 1, 100, seed=4321, len_choices=MPD_QUERY_LENS)
    else:
        Xq = synth_sets(n_query, V, mean_len, lo, hi, seed=1234)
    ev = ref.evaluation
    t0 = time.perf_counter()
    pred = np.asarray(model.predict(Xq))
    pred = ev.remove_non_missing(pred, Xq, copy=True)
    top = ev.argtopk(pred, k)
    dt = time.perf_counter() - t0
    assert top[1].shape == (n_query, k)
    return dt


def cpu_port_run(workload, steps, warmup, threads=None):
    """Fallback when oracle/_ref is absent: the reference's algorithm (dense, as aae.py does it) through the oracle
    port, all host threads."""
    import torch
    from oracle import aae_oracle as O
    V, mean_len, lo, hi, seed, B, _ = WORKLOADS[workload]
    _, batches, V, B = make_batches(workload, min(steps + warmup, 8))
    params = O.init_params(V, H, C, seed=42)
    model = O.OracleAAE(params, n_code=C, faithful_cost=True)
    import scipy.sparse as sp

    def dense(b):
        ip, ii, _ = b
        return sp.csr_matrix((np.ones(len(ii), dtype=np.float32), ii, ip), shape=(B, V)).toarray()
    torch.manual_seed(0)
    for i in range(warmup):
        model.partial_fit(dense(batches[i % len(batches)]), None, O.draw_step_rng(B, H, C))
    t0 = time.perf_counter()
    for i in range(steps):
        model.partial_fit(dense(batches[(warmup + i) % len(batches)]), None, O.draw_step_rng(B, H, C))
    dt = time.perf_counter() - t0
    return steps, dt, "port"


def run_reference(args, use_cuda=False):
    """--impl reference (CPU, the driver's reference arm) / --impl reference-gpu (internal: the gpu_baseline leg)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not use_cuda:
        os.environ["CUDA_VISIBLE_DEVICES"] = ""          # the reference auto-selects CUDA (aae.py:752, 794)
    import torch
    threads = _host_threads()
    torch.set_num_threads(threads)                       # torchrun exports OMP_NUM_THREADS=1: undo its effect
    V, _, _, _, _, B, _ = WORKLOADS[args.workload]
    K, W = args.steps, max(args.warmup, 3)
    if args.impl == "reference-predict":
        # internal leg: the reference's predict + remove_non_missing + argtopk on the host cores
        nq = args.predict_batch
        sec = reference_predict_timed(args.workload, nq, use_cuda)
        line = {"impl": "reference-predict", "unavailable": "oracle/_ref absent"} if sec is None else {
            "impl": "reference-predict", "metric": "top-100 predict sets/sec", "value": nq / sec, "unit": "sets/s",
            "cores": threads, "kind": "reference",
            "sample": "%d query sets through the unmodified reference's model.predict + remove_non_missing + argtopk(k=100) "
                      "(host CPU, CUDA hidden, torch %d threads; dense [n,V] float32 matrix), %.1f s" % (nq, threads, sec)}
        print(json.dumps(line), flush=True)
        return
    res = reference_fit_timed(args.workload, K, W, use_cuda, args.budget)
    if res is None:
        res = cpu_port_run(args.workload, min(K, 20), min(W, 3))
    steps, sec, kind = res
    val = B * steps / sec
    where = "B200, stock PyTorch fp32 (allow_tf32=False)" if use_cuda else "host CPU, CUDA hidden, torch %d threads" % threads
    sample = ("%d timed partial_fit steps (of the %d requested; %.0f s budget) after %d warm-up steps of the "
              "unmodified reference AdversarialAutoEncoder.fit (%s), incl. its per-batch toarray()"
              % (steps, K, args.budget, W, where)) if kind == "reference" else \
             ("%d partial_fit steps of the dense CPU port of aae.py (oracle/_ref absent), torch %d threads" % (steps, threads))
    line = {
        "impl": "reference-gpu" if use_cuda else "reference", "metric": "AAE train item-sets/sec", "value": val,
        "unit": "sets/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "steps_timed": steps,
        "ms_per_step": sec / steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": workload_string(args.workload)},
        "cpu_baseline": {"value": val, "unit": "sets/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _sub_bench(extra_args, timeout_s, env=None):
    """Run this script as a child (reference legs need their own process: CUDA hidden, or a clean torch state)."""
    try:
        e = dict(os.environ)
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS"):
            e.pop(k, None)
        if env:
            e.update(env)
        out = subprocess.run([sys.executable, os.path.abspath(__file__)] + extra_args, capture_output=True, text=True,
                             timeout=timeout_s, env=e)
        for ln in reversed(out.stdout.splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": (out.stderr or out.stdout)[-400:]}
    except Exception as ex:   # noqa: BLE001
        return {"error": repr(ex)[:400]}


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def time_kernel(fn, iters, stream):
    import torch
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        a.record(stream)
        fn()
        b.record(stream)
    torch.cuda.synchronize()
    return [a.elapsed_time(b) * 1e-3 for a, b in evs]


def _uniform_params(V, seed=42, cond_dim=0):
    """random-init weights of the reference architecture (same init law as nn.Linear), torch layout, host"""
    import torch
    g = torch.Generator().manual_seed(seed)

    def uni(shape, fan_in):
        bound = 1.0 / np.sqrt(fan_in)
        return (torch.rand(shape, generator=g) * 2 - 1) * bound
    Cp = C + cond_dim
    return {"enc.lin1.weight": uni((H, V), V), "enc.lin1.bias": uni((H,), V),
            "enc.lin2.weight": uni((H, H), H), "enc.lin2.bias": uni((H,), H),
            "enc.lin3.weight": uni((C, H), H), "enc.lin3.bias": uni((C,), H),
            "dec.lin1.weight": uni((H, Cp), Cp), "dec.lin1.bias": uni((H,), Cp),
            "dec.lin2.weight": uni((H, H), H), "dec.lin2.bias": uni((H,), H),
            "dec.lin3.weight": uni((V, H), H), "dec.lin3.bias": uni((V,), H),
            "disc.lin1.weight": uni((H, C), C), "disc.lin1.bias": uni((H,), C),
            "disc.lin2.weight": uni((H, H), H), "disc.lin2.bias": uni((H,), H),
            "disc.lin3.weight": uni((1, H), H), "disc.lin3.bias": uni((1,), H)}


class Ctx(object):
    """Per-process measurement context (rank, world, barrier, max over ranks)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.saved_stdout = None
        if self.world > 1:
            # NCCL prints its version banner on stdout at communicator creation: keep stdout for the ONE JSON line
            sys.stdout.flush()
            self.saved_stdout = os.dup(1)
            os.dup2(2, 1)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.stream = torch.cuda.current_stream()
        self.hbm_peak, self.tf_peak, self.peak_kind = peaks()

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        import torch
        if self.world == 1:
            return list(vals)
        import torch.distributed as dist
        t = torch.tensor(vals, device=torch.device("cuda", self.local), dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def engine(self, V, B, batches, cond_dim=0, world=None, rank=None, group=None):
        from aaerec_b200.engine import AAEEngine
        a = self.args
        w = self.world if world is None else world
        r = self.rank if rank is None else rank
        eng = AAEEngine(V, H, C, cond_dim=cond_dim, rank=r, world=w, group=group, impl=a.kernel, seed=1, max_batch=B,
                        max_nnz=max(len(b[1]) for b in batches) + 8, use_graph=not a.no_graph)
        if V <= 500000:
            eng.load_params(_uniform_params(V, cond_dim=cond_dim))
        else:
            eng.init_uniform(42)
        return eng


def train_leg(ctx, eng, dev_batches, B, K, W):
    """K partial_fit steps on batches already resident in HBM, after W warm-up steps; device seconds."""
    import torch
    n = len(dev_batches)
    # The time-blocked W1 Adam replays the pending zero-gradient steps of one row group per step: its cost grows for the
    # first G steps of an engine's life (1, 2, ... G replays per row) and is constant afterwards.  The timed region must
    # see the constant cost: a fresh engine first runs G + 3 untimed steps, and then come the W warm-up steps and the K
    # timed steps exactly as --warmup / --steps say.
    aged = 0
    while eng.steps_done < eng.w1_groups + 3:          # untimed: bring the sweep to its steady-state cost
        eng.set_batch_device(*dev_batches[aged % n])
        eng.train_step(B)
        aged += 1
    for i in range(W):
        eng.set_batch_device(*dev_batches[i % n])
        eng.train_step(B)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record(ctx.stream)
    for i in range(K):
        eng.set_batch_device(*dev_batches[(W + i) % n])
        eng.train_step(B)
    e1.record(ctx.stream)
    ctx.barrier()
    return e0.elapsed_time(e1) * 1e-3


def sustained_leg(ctx, eng, dev_batches, B, K, min_seconds=1.0):
    """Blocks of K steps repeated until >= min_seconds of device time: the per-step mean over a region long enough for
    the clock sampler, so that one hiccup cannot move the headline."""
    import torch
    n = len(dev_batches)
    total, steps, i = 0.0, 0, 0
    while total < min_seconds and steps < 200000:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ctx.stream)
        for _ in range(K):
            eng.set_batch_device(*dev_batches[i % n])
            eng.train_step(B)
            i += 1
        e1.record(ctx.stream)
        torch.cuda.synchronize()
        (dt,) = ctx.max_over_ranks(e0.elapsed_time(e1) * 1e-3)     # same loop count on every rank
        total += dt
        steps += K
    return total, steps


def e2e_leg(ctx, eng, batches, B, K, W, cond=None):
    """The same steps through the host-buffer entry (``AAEEngine.train_step_host``, what ``partial_fit`` calls): every
    step the CSR batch travels from pinned host memory into HBM and the three losses travel back into pinned host
    memory, inside the timed region; the host reads the losses of step i-2 when it reuses that step's slot."""
    import torch
    n = len(batches)
    for i in range(3):                       # untimed: captures the host-entry graph
        ip, ii, cc = batches[i % n]
        eng.train_step_host(ip, ii, cc)
    ctx.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h2d = 0
    seen = 0.0
    t0.record(ctx.stream)
    for i in range(K):
        ip, ii, cc = batches[(W + i) % n]
        slot = eng.train_step_host(ip, ii, cc)
        h2d += ip.nbytes + ii.nbytes + (cc.nbytes if cc is not None else 0)
        if slot["prev_losses"] is not None:
            seen += float(slot["prev_losses"][0])      # losses of step i-2, complete (its event was waited for)
    t1.record(ctx.stream)
    ctx.barrier()
    assert seen == seen
    return t0.elapsed_time(t1) * 1e-3, h2d // max(K, 1)


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the decoder-output training kernel on a whole (unsharded)
# vocabulary at batch 100, from the `ncu --set full` captures summarised in profiles/r02_k3_dec_out_train_tc2_final.txt
K3_NCU_TRAFFIC = {2000000: 2.698415e9 + 2.381553e9, 200000: 258.995968e6 + 191.858432e6}


def k3_roofline(ctx, eng, B, V, traffic=None):
    """The decoder-output kernel (K3) and the dense W1 sweep timed alone on their stream, CUDA events."""
    if traffic is None and eng.world == 1 and B == 100:
        traffic = K3_NCU_TRAFFIC.get(V)
    import torch
    from aaerec_b200._native import call, ptr
    Vl = eng.Vloc
    st = ptr(eng.state)
    torch.cuda.synchronize()

    def k3():
        call("aae_dec_out_train", ptr(eng.h2), B, H, ptr(eng.Wd3), ptr(eng.bd3), ptr(eng.Wd3_m), ptr(eng.Wd3_v),
             ptr(eng.bd3_m), ptr(eng.bd3_v), eng.v_begin, Vl, ptr(eng.indptr), ptr(eng.indices), float(B) * V, st,
             ptr(eng.dh2), ptr(eng.loss_sums), eng.impl_for(B), eng._stream())

    def sweep():
        call("aae_w1_sweep_untouched", ptr(eng.slot_of), 0, Vl, H, ptr(eng.W1t), ptr(eng.W1_m1), ptr(eng.W1_v1),
             ptr(eng.W1_m2), ptr(eng.W1_v2), st, eng._stream())
    kern = {}
    for name, fn, alg_bytes in (("dec_out_train", k3, 24.0 * (Vl * H + Vl) + 8.0 * B * H),
                                ("w1_sweep_untouched", sweep, 40.0 * Vl * H + 4.0 * Vl)):
        for _ in range(3):
            fn()
        ts = time_kernel(fn, 10, ctx.stream)
        kern[name] = {"sec": float(np.mean(ts)), "bytes": alg_bytes}
    dom = "dec_out_train"
    ach = kern[dom]["bytes"] / kern[dom]["sec"] / 1e9
    return {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": ctx.hbm_peak, "unit": "GB/s",
            "frac": ach / ctx.hbm_peak, "traffic": traffic, "peak_source": ctx.peak_kind,
            "algorithmic_bytes": kern[dom]["bytes"], "ms": kern[dom]["sec"] * 1e3,
            "kernels": {k: {"ms": v["sec"] * 1e3, "GBps": v["bytes"] / v["sec"] / 1e9,
                            "frac": v["bytes"] / v["sec"] / 1e9 / ctx.hbm_peak} for k, v in kern.items()}}


TRACE_NAMES = ["batch_prepare", "w1_sweep", "ae_fwd", "dec_out_train", "ae_bwd", "ae_wgrad", "w1_rows_update_1", "disc_phase",
               "disc_wgrad", "gen_phase", "gen_wgrad", "w1_rows_update_2", "step_finish", "bag_fwd", "w1_catchup"]


def step_timeline(eng, dev_batches, B, reps=3):
    """In-graph duration of every kernel of one training step, microseconds (median of `reps` steps): every kernel's
    first block writes %globaltimer at its start and its last block at its end into a trace buffer (aae_trace_set)."""
    import torch
    from aaerec_b200 import _native as N
    nslots = int(N.load().aae_trace_slots())
    buf = torch.zeros(nslots, dtype=torch.int64, device=eng.dev)
    pre = torch.tensor([2 ** 62, 0] * (nslots // 2), dtype=torch.int64, device=eng.dev)
    N.call("aae_trace_set", N.ptr(buf))
    rows = []
    try:
        for r in range(reps):
            buf.copy_(pre)
            torch.cuda.synchronize()
            eng.set_batch_device(*dev_batches[r % len(dev_batches)])
            eng.train_step(B)
            torch.cuda.synchronize()
            t = buf.cpu().numpy().reshape(-1, 2)
            live = [k for k in range(min(len(TRACE_NAMES), len(t))) if t[k, 1] > 0]
            d = {TRACE_NAMES[k]: (t[k, 1] - t[k, 0]) / 1e3 for k in live}
            d["first_to_last_mark"] = (max(t[k, 1] for k in live) - min(t[k, 0] for k in live)) / 1e3
            rows.append(d)
    finally:
        N.call("aae_trace_set", None)
    return {k: float(np.median([r[k] for r in rows if k in r])) for k in rows[0]}


def step_bytes(eng):
    """HBM bytes one step of the implemented policy moves (SURVEY 8(d): 'state which policy is implemented and use the
    matching figure'): dec.lin3 + its Adam state once (24 B/param), 1/G of the W1 rows with both Adam states (40/G)."""
    return (24.0 + 40.0 / eng.w1_groups) * eng.Vloc * H


MPD_QUERY_LENS = (1, 5, 10, 25, 100)     # SURVEY 8(d) C5: seed-track counts of the MPD challenge (create_dev_set.py:16-17)
COLD_M = 2.0 ** -110      # csrc/w1_blocked.cu kColdM


def w1_cold_row_frac(eng):
    """Fraction of this rank's W1 rows whose first moments (both optimizers) are all cold (|m| <= 2^-110, incl. rows
    that never were in a batch): the time-blocked sweep skips the W update of those rows (exactly)."""
    cold = (eng.W1_m1.abs().amax(1) <= COLD_M) & (eng.W1_m2.abs().amax(1) <= COLD_M)
    return float(cold.float().mean().item())


DUMP_SAMPLE_ITEMS = 32768


def dump_outputs(ctx, eng, last_batch, out_dir):
    """What the last timed step handed its caller: the step's losses (R, D, G) and the weights after it in the
    reference's names and layouts, float32.  The item-indexed tensors (enc.lin1.weight columns, dec.lin3 rows) keep the
    items of that step's batch plus a seeded draw of DUMP_SAMPLE_ITEMS items (all items when V is smaller): 800 bytes per
    kept item, about 30 MB at the MPD shape; each rank cuts its own item range on the device.  Reading W1 needs its
    pending zero-gradient Adam steps applied (flush_w1); the engine's state is restored afterwards, so the legs that
    follow start from the state the timed steps left.  Collective over the item shards; rank 0 writes."""
    import torch
    from aaerec_b200.engine import enc_block_sizes, dec_block_sizes, disc_block_sizes
    items = np.union1d(last_batch[1], np.random.RandomState(0).choice(eng.V, min(eng.V, DUMP_SAMPLE_ITEMS), replace=False))
    snap, w1_dirty = eng._snapshot(), eng._w1_dirty
    eng.flush_w1()
    loc = torch.as_tensor(items, dtype=torch.int64, device=eng.dev) - eng.v_begin
    mine = (loc >= 0) & (loc < eng.Vloc)
    loc = loc.clamp(0, max(eng.Vloc - 1, 0))

    def sampled(t):
        rows = torch.where(mine.view((-1,) + (1,) * (t.dim() - 1)), t[loc], torch.zeros((), device=eng.dev))
        if eng.world > 1:                   # every sampled item lives on exactly one rank: the sum is that rank's row
            import torch.distributed as dist
            dist.all_reduce(rows, group=eng.group)
        return rows.cpu().numpy()
    out = {"losses": eng.losses.cpu().numpy(), "enc.lin1.weight": sampled(eng.W1t).T,
           "dec.lin3.weight": sampled(eng.Wd3), "dec.lin3.bias": sampled(eng.bd3)}
    H, Cc = eng.H, eng.C
    shapes = {"enc.lin2.weight": (H, H), "enc.lin3.weight": (Cc, H), "dec.lin1.weight": (H, eng.Cp),
              "dec.lin2.weight": (H, H), "disc.lin1.weight": (H, Cc), "disc.lin2.weight": (H, H), "disc.lin3.weight": (1, H)}
    for blk, sizes in ((eng.enc, enc_block_sizes(H, Cc)), (eng.dec, dec_block_sizes(H, eng.Cp)),
                       (eng.disc, disc_block_sizes(H, Cc))):
        off = 0
        for name, sz in sizes:
            out[name] = blk[off:off + sz].cpu().numpy().reshape(shapes.get(name, (sz,)))
            off += sz
    eng._restore(snap)
    eng._w1_dirty = w1_dirty
    del snap
    if ctx.rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def train_workload(ctx, name, K, W, with_roofline=True, with_sustained=True, B=None, cond_dim=0, with_e2e=True,
                   hot_w1=False, dump_dir=None):
    """value / e2e / roofline of one training workload; returns (dict, engine, batches).  hot_w1: every W1 row starts
    with live Adam moments (as if every item had been in a recent batch): the worst case of the time-blocked sweep,
    none of its rows is cold.  dump_dir: write the outputs of the last timed step there (dump_outputs)."""
    import torch
    n_batches = min(K + W, 32 if WORKLOADS[name][0] > 500000 else 64)
    _, batches, V, B = make_batches(name, n_batches, cond_dim=cond_dim, B=B)
    eng = ctx.engine(V, B, batches, cond_dim=cond_dim)
    if hot_w1:
        g = torch.Generator(device=eng.dev).manual_seed(5)
        for m, v in ((eng.W1_m1, eng.W1_v1), (eng.W1_m2, eng.W1_v2)):
            m.normal_(0.0, 1e-3, generator=g)
            v.uniform_(1e-7, 1e-6, generator=g)
    dev_batches = [tuple(torch.as_tensor(x, device=eng.dev) for x in (ip, ii) + ((cc,) if cc is not None else ()))
                   for ip, ii, cc in batches]
    from aaerec_b200 import _native as N
    sec = train_leg(ctx, eng, dev_batches, B, K, W)
    if dump_dir is not None:
        dump_outputs(ctx, eng, batches[(W + K - 1) % len(batches)], dump_dir)
    N.reset_launch_count()
    eng.set_batch_device(*dev_batches[0])
    launches = eng.launches_per_step() * K
    out = {"metric": "AAE train item-sets/sec", "unit": "sets/s", "steps": K}
    (sec,) = ctx.max_over_ranks(sec)
    out["value"] = B * K / sec
    out["ms_per_step"] = sec / K * 1e3
    cold_roofline = None
    if with_roofline:
        # right behind the timed steps, i.e. in the same board state as `value`: the dominant kernel alone on its
        # stream, and the in-graph duration of every kernel of one step (globaltimer marks of first / last block)
        eng.set_batch_device(*dev_batches[0])
        cold_roofline = k3_roofline(ctx, eng, B, V)
        cold_roofline["step_timeline_us"] = step_timeline(eng, dev_batches, B)
    if with_e2e:
        sec_e2e, h2d = e2e_leg(ctx, eng, batches, B, K, W)
        (sec_e2e,) = ctx.max_over_ranks(sec_e2e)
        out["e2e"] = {"value": B * K / sec_e2e, "unit": "sets/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 12,
                      "ms_per_step": sec_e2e / K * 1e3}
    if with_sustained:
        # after the two K-step legs: >= 1 s of back-to-back steps (the GPU reaches its power-capped clocks here)
        tot, steps = sustained_leg(ctx, eng, dev_batches, B, K)
        out["sustained"] = {"value": B * steps / tot, "ms_per_step": tot / steps * 1e3, "steps": steps,
                            "seconds": tot}
    if eng.peer is not None and eng.peer.error():
        raise RuntimeError("peer exchange timed out (ranks diverged)")
    out["gpu_launches"] = launches
    out["decoder_kernel"] = {0: "simt-fp32", 1: "tcgen05-3xTF32", 2: "tcgen05-TF32"}.get(eng.impl_for(B), "?")
    moved = step_bytes(eng)
    ms = out["sustained"]["ms_per_step"] if with_sustained else out["ms_per_step"]
    out["step_moved_bytes_per_gpu"] = moved
    out["step_frac"] = moved / (ms * 1e-3) / 1e9 / ctx.hbm_peak
    out["tensor_frac"] = 6.0 * B * H * eng.Vloc / (ms * 1e-3) / 1e12 / ctx.tf_peak
    out["step_frac_timed"] = moved / (out["ms_per_step"] * 1e-3) / 1e9 / ctx.hbm_peak
    if with_roofline:
        out["roofline"] = cold_roofline
        if with_sustained:
            # the same kernel again after >= 1 s of back-to-back steps: the board runs at its power cap by then
            # (sw_power_cap) and the heavy kernels are ~5-10 % slower although the reported SM clock stays near its maximum
            eng.set_batch_device(*dev_batches[0])
            hot = k3_roofline(ctx, eng, B, V)
            out["roofline"]["after_sustained"] = {"ms": hot["ms"], "achieved": hot["achieved"], "frac": hot["frac"]}
    out["nnz_mean"] = float(np.mean([len(b[1]) for b in batches]))
    out["w1_cold_row_frac"] = w1_cold_row_frac(eng)
    return out, eng, batches


def predict_leg(ctx, eng, Xq, k, iters, rows_total=None):
    """top-k predict (reconstruction + known-item mask + top-k, aae.py:840-870 + evaluation.py:183-199, 20-58) of
    one query batch: device-resident and end-to-end (host CSR in, [B,k] item ids out)."""
    import torch
    Bq = Xq.shape[0]
    ip = Xq.indptr.astype(np.int32)
    ii = Xq.indices.astype(np.int32)
    eng.upload_csr(ip, ii)
    from aaerec_b200 import _native as N
    fused = int(N.load().aae_predict_topk_work_bytes(Bq, eng.Vloc, min(k, eng.Vloc))) > 0 and eng.impl_for_scores() in (1, 2)
    # the dense [B, Vloc] score matrix exists only on the dense path (small shards) -- the fused path never builds it
    scratch = None if fused else torch.empty(Bq, eng.Vloc, dtype=torch.float32, device=eng.dev)
    for _ in range(2):
        eng.topk(Bq, k, scratch=scratch)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ctx.stream)
    for _ in range(iters):
        eng.topk(Bq, k, scratch=scratch, check=False)      # status word checked once after the loop (same batch)
    e1.record(ctx.stream)
    ctx.barrier()
    if eng.topk_status() != 0:
        raise RuntimeError("fused top-k reported rows it could not rank exactly in the timed loop")
    sec = e0.elapsed_time(e1) * 1e-3 / iters
    out_pin = torch.zeros(Bq, min(k, eng.V), dtype=torch.int32).pin_memory()
    ctx.barrier()
    e0.record(ctx.stream)
    for _ in range(iters):
        eng.upload_csr(ip, ii)
        idx, _ = eng.topk(Bq, k, scratch=scratch)
        out_pin.copy_(idx, non_blocking=True)
        ctx.stream.synchronize()
    e1.record(ctx.stream)
    ctx.barrier()
    sec_e2e = e0.elapsed_time(e1) * 1e-3 / iters
    sec, sec_e2e = ctx.max_over_ranks(sec, sec_e2e)
    V = eng.V
    if rows_total is not None:          # set-sharded: this rank ranked its slice; the job's rows are rows_total
        Bq = rows_total
    return {"metric": "top-100 predict sets/sec", "value": Bq / sec, "unit": "sets/s", "ms_per_batch": sec * 1e3,
            "e2e": {"value": Bq / sec_e2e, "unit": "sets/s", "h2d_bytes_per_step": ip.nbytes + ii.nbytes,
                    "d2h_bytes_per_step": out_pin.numel() * 4},
            "roofline": {"bound": "tensor", "achieved": 2.0 * Bq * V * H / sec / 1e12 / ctx.world,
                         "peak": ctx.tf_peak, "unit": "TFLOP/s",
                         "frac": 2.0 * Bq * V * H / sec / 1e12 / ctx.tf_peak / ctx.world},
            "fallbacks": eng.topk_fallbacks, "path": getattr(eng, "topk_mode", None)}


def parity_check(ctx, name, steps=5):
    """N-GPU vs 1-GPU parity inside the driver-run record (SURVEY 8(d) gate iv): the same ``steps`` native-RNG steps
    on the item-sharded engine and on a single-rank engine (rank 0), same seed and batches; then the same top-100
    query.  Losses, every weight tensor (relative Frobenius norm) and the top-k lists are compared on rank 0."""
    import torch
    from aaerec_b200.synth import synth_sets
    _, batches, V, B = make_batches(name, steps)
    eng = ctx.engine(V, B, batches)
    losses = []
    for ip, ii, _ in batches:
        eng.train_step_host(ip, ii)
        torch.cuda.synchronize()
        losses.append(eng.losses.cpu().numpy().copy())
    sd = eng.state_dict()                                  # collective: gathers the item shards
    Xq = synth_sets(64, V, WORKLOADS[name][1], WORKLOADS[name][2], WORKLOADS[name][3], seed=99)
    eng.upload_csr(Xq.indptr.astype(np.int32), Xq.indices.astype(np.int32))
    ti, tv = eng.topk(64, 100)
    ti, tv = ti.cpu().numpy(), tv.cpu().numpy()
    eng.close()
    del eng
    torch.cuda.empty_cache()
    res = None
    if ctx.rank == 0:
        one = ctx.engine(V, B, batches, world=1, rank=0)
        l1 = []
        for ip, ii, _ in batches:
            one.train_step_host(ip, ii)
            torch.cuda.synchronize()
            l1.append(one.losses.cpu().numpy().copy())
        sd1 = one.state_dict()
        one.upload_csr(Xq.indptr.astype(np.int32), Xq.indices.astype(np.int32))
        oi, ov = one.topk(64, 100)
        oi, ov = oi.cpu().numpy(), ov.cpu().numpy()
        del one
        torch.cuda.empty_cache()
        la, lb = np.asarray(losses, dtype=np.float64), np.asarray(l1, dtype=np.float64)
        loss_rel = float(np.max(np.abs(la - lb) / np.maximum(np.abs(lb), 1e-30)))
        per = {}
        for k_, v in sd1.items():
            a, b = sd[k_].double(), v.double()
            per[k_] = float((a - b).norm() / max(float(b.norm()), 1e-30))
        big = ("enc.lin1.weight", "dec.lin3.weight", "dec.lin3.bias")      # the item-sharded tensors: 99.99 % of the parameters
        w_big = max(per[k_] for k_ in big)
        worst = max(per, key=per.get)
        mism = ti != oi
        # positions that differ although the single-GPU scores there are not tied (to 1e-6 relative)
        hard = int(np.sum(mism & (np.abs(tv - ov) > 1e-6 * np.maximum(np.abs(ov), 1e-30))))
        res = {"workload": name, "steps": steps, "loss_rel_max": loss_rel, "weights_rel_max_sharded_tensors": w_big,
               "weights_rel_max": per[worst], "weights_worst_tensor": worst,
               "topk_positions": int(ti.size), "topk_mismatch": int(mism.sum()), "topk_mismatch_outside_ties": hard,
               "tolerance": "losses and the item-sharded tensors 1e-4; the replicated small layers 5e-3: the shards sum "
                            "their [B,H] partials in rank order, a different fp32 summation order than one GPU, and "
                            "Adam's normalisation turns that rounding noise into lr-sized differences on the few "
                            "elements whose gradient is ~0 (a ReLU unit at its kink), visible on the 100-element tensors "
                            "only (DESIGN.md, 'numerical sensitivity')",
               "ok": bool(loss_rel < 1e-4 and w_big < 1e-4 and per[worst] < 5e-3 and hard == 0)}
    ctx.barrier()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    from aaerec_b200.synth import synth_sets

    ctx = Ctx(args)
    world, rank = ctx.world, ctx.rank
    K, W = args.steps, max(args.warmup, 3)
    head = args.workload
    extra = {}

    parity = parity_check(ctx, head) if world > 1 and not args.no_parity else None
    if parity is not None and rank == 0 and not parity["ok"]:
        sys.stderr.write("PARITY CHECK FAILED: %r\n" % (parity,))

    # ---------------- headline: value / e2e / roofline on the named workload ----------------
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    if sampler:
        sampler.start()
    main, eng, batches = train_workload(ctx, head, K, W, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if sampler else None
    V, B = eng.V, WORKLOADS[head][5]

    def hot_leg():
        # the same K steps with every W1 row hot (live Adam moments everywhere): the other end of the bracket
        h, e, _ = train_workload(ctx, head, K, W, with_roofline=False, with_sustained=False, with_e2e=False, hot_w1=True)
        e.close()
        del e
        torch.cuda.empty_cache()
        return {"value": h["value"], "unit": "sets/s", "ms_per_step": h["ms_per_step"], "steps": K,
                "w1_cold_row_frac": h["w1_cold_row_frac"]}
    hot = hot_leg() if (args.no_extra and world == 1) else None
    exchange, graph, groups = eng._exchange_kind, eng.use_graph, eng.w1_groups
    if args.kernel_times and world == 1:
        from aaerec_b200 import _native as N
        dev_batches = [(torch.as_tensor(ip, device=eng.dev), torch.as_tensor(ii, device=eng.dev)) for ip, ii, _ in batches]
        eng.use_graph = False
        eng.overlap_sweep = False
        N.enable_timing(True)
        for i in range(20):
            eng.set_batch_device(*dev_batches[i % len(dev_batches)])
            eng.train_step(B)
        rep = N.timing_report()
        N.enable_timing(False)
        eng.use_graph = graph
        eng.overlap_sweep = True
        tot = sum(c * us for c, us in rep.values()) / 20.0
        sys.stderr.write("per-entry-point device time per step (eager, warm): total %.1f us\n" % tot)
        for k, (c, us) in sorted(rep.items(), key=lambda kv: -kv[1][0] * kv[1][1]):
            sys.stderr.write("  %-28s x%.1f  %8.1f us each  %5.1f%%\n" % (k, c / 20.0, us, 100 * c * us / 20.0 / tot))

    if not args.no_extra:
        # ---------------- predict: reconstruction + masked top-100 (the metric's second half) ----------------
        if head == "mpd":
            sweep = {}
            for Bq in (1000, 4000, 16000, 64000):
                Xq = synth_sets(Bq, V, 25, 1, 100, seed=4321, len_choices=MPD_QUERY_LENS)
                pr = predict_leg(ctx, eng, Xq, 100, 5 if Bq <= 4000 else 2)
                pr["config"] = {"workload": "mpd-shaped (BASELINE configs[4]): V=%d items, query batch %d sets with 1/5/10/25/100 "
                                            "seed items each (uniformly; before de-duplication), k=100, known items masked, "
                                            "item-sharded x%d" % (V, Bq, world)}
                sweep["B%d" % Bq] = pr
            extra["mpd_predict"] = sweep["B1000"]
            extra["mpd_predict_sweep"] = {k: {"value": v["value"], "e2e": v["e2e"]["value"], "ms_per_batch": v["ms_per_batch"],
                                              "tensor_frac": v["roofline"]["frac"], "fallbacks": v["fallbacks"],
                                              "path": v["path"]}
                                          for k, v in sweep.items()}
            if world > 1:
                # set-sharded replicas (SURVEY 8(e)): every rank ranks its own slice of the query rows against a
                # full-weight replica -- zero communication; reported beside the item-sharded numbers above
                rep = eng.make_replica(max_batch=1024)
                ss = {}
                for Bq in (1000, 4000, 16000, 64000):
                    Xq = synth_sets(Bq, V, 25, 1, 100, seed=4321, len_choices=MPD_QUERY_LENS)
                    per = (Bq + world - 1) // world
                    Xl = Xq[rank * per:min(Bq, (rank + 1) * per)]
                    pr = predict_leg(ctx, rep, Xl, 100, 5 if Bq <= 4000 else 2, rows_total=Bq)
                    ss["B%d" % Bq] = {"value": pr["value"], "e2e": pr["e2e"]["value"], "ms_per_batch": pr["ms_per_batch"],
                                      "fallbacks": pr["fallbacks"], "path": pr["path"]}
                extra["mpd_predict_sweep_set_sharded"] = ss
                del rep
                torch.cuda.empty_cache()
        else:
            Xq = synth_sets(args.predict_batch, V, WORKLOADS[head][1], WORKLOADS[head][2], WORKLOADS[head][3], seed=1234)
            extra["predict"] = predict_leg(ctx, eng, Xq, 100, 10)
        eng.close()
        del eng
        torch.cuda.empty_cache()
        hot = hot_leg()
        # ---------------- the other BASELINE configs as extra legs ----------------
        Ke = max(10, min(K, 50))
        if head == "mpd":
            # C4 at the reference scripts' larger batches (mpd.py:75-76, aminer.py:62): the tensor-roofline configs
            for Bx, Kx in ((1000, 5), (10000, 2)):
                if args.skip_big and Bx >= 10000:
                    continue
                leg, e2, _ = train_workload(ctx, "mpd", Kx, 3, with_roofline=False, with_sustained=False, B=Bx,
                                            with_e2e=False)
                leg["config"] = {"workload": workload_string("mpd", Bx) + ", item-sharded x%d" % world}
                extra["mpd_b%d" % Bx] = leg
                e2.close()
                del e2
                torch.cuda.empty_cache()
            # PubMed-shaped: configs[1] (+ predict), configs[2] (title condition), B=500 (main.py:76)
            leg, e2, _ = train_workload(ctx, "pubmed", Ke, 3)
            leg["config"] = {"workload": workload_string("pubmed") + (", item-sharded x%d" % world if world > 1 else "")}
            Xq = synth_sets(args.predict_batch, 200000, 16, 2, 200, seed=1234)
            leg["predict"] = predict_leg(ctx, e2, Xq, 100, 10)
            extra["pubmed"] = leg
            e2.close()
            del e2
            torch.cuda.empty_cache()
            leg, e2, _ = train_workload(ctx, "pubmed", Ke, 3, with_roofline=False, with_sustained=False, B=500)
            leg["config"] = {"workload": workload_string("pubmed", 500)}
            extra["pubmed_b500"] = leg
            e2.close()
            del e2
            leg, e2, _ = train_workload(ctx, "pubmed", Ke, 3, with_roofline=False, with_sustained=False, cond_dim=300)
            leg["config"] = {"workload": workload_string("pubmed") + " + 300-d title condition (BASELINE configs[2]: "
                                         "concatenation-based conditioning on the code, decoder lin1 350 -> 100)"}
            extra["pubmed_cond"] = leg
            e2.close()
            del e2
            torch.cuda.empty_cache()
            if world == 1:
                leg, e2, _ = train_workload(ctx, "econbiz", Ke, 3, with_roofline=False, with_sustained=False)
                leg["config"] = {"workload": workload_string("econbiz")}
                extra["econbiz"] = leg
                del e2
                extra["fit_epoch"] = fit_epoch_leg(ctx)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu = gpu_ref = None
    if world == 1 and not args.no_cpu:
        r = _sub_bench(["--impl", "reference", "--workload", head, "--steps", "6", "--warmup", "3", "--budget", "25"], 900)
        cpu = r.get("cpu_baseline", r)
        g = _sub_bench(["--impl", "reference-gpu", "--workload", head, "--steps", "20", "--warmup", "5", "--budget", "20"], 600)
        gpu_ref = {"value": g["value"], "unit": "sets/s", "ms_per_step": g["ms_per_step"],
                   "what": g["cpu_baseline"]["sample"]} if "value" in g else g
        if not args.no_extra:
            # the reference's ranking chain on the host cores, bounded samples (V=2M: 200 sets = two dense 800 MB batches)
            if "mpd_predict" in extra:
                extra["mpd_predict"]["cpu_baseline"] = _sub_bench(
                    ["--impl", "reference-predict", "--workload", "mpd", "--predict-batch", "200"], 600)
            if "pubmed" in extra and "predict" in extra["pubmed"]:
                extra["pubmed"]["predict"]["cpu_baseline"] = _sub_bench(
                    ["--impl", "reference-predict", "--workload", "pubmed", "--predict-batch", "1000"], 600)
    line = {
        "metric": "AAE train item-sets/sec", "value": main["value"], "unit": "sets/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(head),
                   "parallelism": ("item-sharded x%d (Wd3/bd3/W1t by item range; exchange: %s)" % (world, exchange))
                   if world > 1 else "single GPU",
                   "decoder_kernel": main["decoder_kernel"], "cuda_graph": graph,
                   "rng": "in-kernel Philox (native)",
                   "w1_policy": "dense-Adam-equivalent, time-blocked in %d groups (exact)" % groups,
                   "w1_cold_rows": {"frac": main["w1_cold_row_frac"],
                                    "note": "the sweep skips the W update of elements whose first moments are <= 2^-110 "
                                            "(it cannot change W: bit-identical, tests/test_gpu_parity.py) -- rows that "
                                            "never were in a batch or not for ~650 steps.  This run starts from fresh "
                                            "moments and cycles through %d batches, so nearly every row outside them is "
                                            "cold; `w1_all_rows_hot` is the same measurement with live moments in EVERY "
                                            "row (no cold row at all), a long training run lies between the two "
                                            "(DESIGN.md 4: ~65 %% of the rows cold under this Zipf law, more on real "
                                            "long-tail catalogues)" % len(batches)},
                   "pre_aging_steps": groups + 3,
                   "pre_aging_note": "the time-blocked sweep replays 1..G pending steps per row during an engine's first G "
                                     "steps and G afterwards: a fresh engine runs G + 3 untimed steps before the W warm-up "
                                     "and K timed steps, so that the timed steps pay the constant (steady-state) cost",
                   "board_state": "the K timed steps follow ~60 ms of untimed steps; `sustained` (>= 1 s of back-to-back "
                                  "steps, board at its power cap) is 5-8 % slower, roofline.after_sustained is the dominant "
                                  "kernel in that state",
                   "mean_items_per_set": main["nnz_mean"] / B,
                   "l2": "per-step working set %.2f GB per GPU >> 126 MB L2 (no flush needed)"
                         % (main["step_moved_bytes_per_gpu"] / 1e9)},
        "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "sustained": main.get("sustained"),
        "roofline": dict(main["roofline"], step_moved_bytes=main["step_moved_bytes_per_gpu"],
                         step_frac=main["step_frac_timed"], step_frac_sustained=main["step_frac"]),
        "tensor_frac": main["tensor_frac"],
        "w1_all_rows_hot": hot,
        "cpu_baseline": cpu, "gpu_baseline": gpu_ref, "clocks": clocks,
    }
    if parity is not None:
        line["parity_check"] = parity
    line.update(extra)
    if ctx.saved_stdout is not None:
        sys.stdout.flush()
        os.dup2(ctx.saved_stdout, 1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def fit_epoch_leg(ctx, n=50000):
    """Epochs of ``AdversarialAutoEncoder.fit`` (the public call) on PubMed-shaped n=50k: wall-clock per epoch
    (shuffle + device-side batching + all steps, SURVEY 8(f)-4) against n/B x the device step time."""
    from aaerec_b200.aae import AdversarialAutoEncoder
    from aaerec_b200.synth import synth_sets
    import contextlib
    import io
    V, mean_len, lo, hi, seed, B, _ = WORKLOADS["pubmed"]
    X = synth_sets(n, V, mean_len, lo, hi, seed)
    np.random.seed(0)
    model = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=B, n_epochs=3, verbose=False)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        model.fit(X)
    total = time.perf_counter() - t0
    steps = (n + B - 1) // B
    ep = min(model.epoch_seconds[1:])        # epoch 1 also captures the step's CUDA graph
    model.engine.close()
    return {"n_sets": n, "batch": B, "steps_per_epoch": steps, "epoch_wall_s": ep, "ms_per_step_wall": ep / steps * 1e3,
            "sets_per_s": n / ep, "first_epoch_wall_s": model.epoch_seconds[0], "fit_total_wall_s": total,
            "note": "AdversarialAutoEncoder.fit, 3 epochs; epoch wall-clock = host permutation + upload + "
                    "aae_batch_gather + train step per batch, synchronised once per epoch"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu", "reference-predict"])
    ap.add_argument("--workload", default="mpd", choices=sorted(WORKLOADS))
    ap.add_argument("--kernel", default="auto", help="decoder-output kernel: auto|simt|tc|tf32")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU / stock-PyTorch-GPU reference baselines")
    ap.add_argument("--no-parity", action="store_true", help="skip the N-GPU vs 1-GPU parity check (world > 1)")
    ap.add_argument("--kernel-times", action="store_true", help="print warm per-kernel device times to stderr")
    ap.add_argument("--no-extra", action="store_true", help="headline workload only")
    ap.add_argument("--skip-big", action="store_true", help="skip the B=10000 leg")
    ap.add_argument("--predict-batch", type=int, default=1000)
    ap.add_argument("--budget", type=float, default=120.0, help="reference arm: seconds of timed work before it stops")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the losses and (sampled) weights of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl in ("reference", "reference-predict"):
        run_reference(args, use_cuda=False)
    elif args.impl == "reference-gpu":
        run_reference(args, use_cuda=True)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
