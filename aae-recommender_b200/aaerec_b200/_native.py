"""ctypes binding of ``libaae_b200.so`` (the C ABI declared in ``include/aae_b200.h``).

There is no fallback: if the library is missing, or the device is not sm_100, every entry
point raises.  Pointers are passed as plain integers (``tensor.data_ptr()``), the stream as
``torch.cuda.current_stream().cuda_stream``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AAE_B200_LIB") or os.path.join(_HERE, "libaae_b200.so")   # override: kernel A/B experiments

P = C.c_void_p
I = C.c_int
I64 = C.c_int64
F = C.c_float
D = C.c_double


class AaeDims(C.Structure):
    _fields_ = [("B", I), ("H", I), ("C", I), ("D", I)]


class AaeDrop(C.Structure):
    _fields_ = [("mask", P), ("p", F), ("stream_id", C.c_uint32)]


class AaeBag(C.Structure):
    """Mirror of ``aae_bag``: the batch's CSR rows + W1t for the in-kernel gather (indptr NULL: read h1pre)."""
    _fields_ = [("indptr", P), ("indices", P), ("W1t", P), ("normalize", I), ("v_begin", I), ("v_end", I)]


class AdamBlock(C.Structure):
    """Mirror of ``aae_adam_block``: a packed parameter block with its Adam moments (p NULL: gradient only)."""
    _fields_ = [("p", P), ("m", P), ("v", P), ("which", I)]


class AaePeers(C.Structure):
    """Mirror of ``aae_peers``: every rank's exchange buffer as mapped in this process."""
    _fields_ = [("base", P * 8), ("rank", I), ("world", I)]


class AaeRankFilter(C.Structure):
    """Mirror of ``aae_rank_filter``: column -> global id table and per-row exclusion CSR of a filtered ranking."""
    _fields_ = [("item_ids", P), ("excl_indptr", P), ("excl_indices", P)]


class StepState(C.Structure):
    """Mirror of ``aae_step_state`` (device resident; used for size and for debugging reads)."""
    _fields_ = [("t", C.c_int32), ("rng_step", C.c_uint32), ("step_size_gen", F), ("step_size_reg", F),
                ("bc2_sqrt", F), ("beta1", F), ("beta2", F), ("eps", F), ("gen_lr", F), ("reg_lr", F),
                ("seed", C.c_uint64)]


_SIGS = {
    "aae_version": (I, []),
    "aae_last_error": (C.c_char_p, []),
    "aae_device_check": (I, [I]),
    "aae_step_state_init": (I, [P, F, F, C.c_uint64, P]),
    "aae_step_tick": (I, [P, P]),
    "aae_bag_fwd": (I, [P, P, I, P, P, I, I, I, I, I, P, P]),
    "aae_w1_sweep_untouched": (I, [P, I, I, I, P, P, P, P, P, P, P]),
    "aae_ae_bwd": (I, [AaeDims, P, P, P, AaeDrop, AaeDrop, AaeDrop, AaeDrop, P, P, P, P, P, P, P, P, P, P, P]),
    "aae_ae_fwd_bag": (I, [AaeDims, AaeBag, P, P, P, P, AaeDrop, AaeDrop, AaeDrop, AaeDrop, P, P, P, P, P, P, P, P]),
    "aae_disc_phase_bag": (I, [AaeDims, AaeBag, P, P, F, P, P, AaeDrop, AaeDrop, AaeDrop, AaeDrop, P, P, P, P, P]),
    "aae_gen_phase_bag": (I, [AaeDims, AaeBag, P, P, P, AaeDrop, AaeDrop, AaeDrop, AaeDrop, P, P, P, P, P, P, P, P]),
    "aae_predict_tail_bag": (I, [AaeDims, AaeBag, P, P, P, P, P, P]),
    "aae_batch_prepare": (I, [P, P, I, I, I, P, P, P, P, P, P, P, I, P]),
    "aae_w1_rows_update": (I, [P, P, I, P, P, P, I, P, P, P, P, I, P, I, P, P]),
    "aae_step_finish": (I, [P, P, P, I, P, I, D, I, P, P, P, P]),
    "aae_ktab_write": (I, [P, P, P]),
    "aae_w1_catchup": (I, [P, P, I, I, I, P, P, P, P, P, P, P, I, P, P, P]),
    "aae_w1_sweep_blocked": (I, [P, I, I, P, P, P, P, P, P, P, P, I, I, I, P]),
    "aae_ae_wgrad": (I, [AaeDims, P, P, P, P, P, P, P, P, P, P, P, AdamBlock, AdamBlock, P, P]),
    "aae_disc_wgrad": (I, [AaeDims, P, P, P, AdamBlock, P, P]),
    "aae_gen_wgrad": (I, [AaeDims, P, P, P, P, P, P, AdamBlock, P, P]),
    "aae_dec_out_train": (I, [P, I, I, P, P, P, P, P, P, I, I, P, P, D, P, P, P, I, P]),
    "aae_dec_out_train_ws": (I, [P, I, I, P, P, P, P, P, P, I, I, P, P, D, P, P, P, I, P, I64, P]),
    "aae_dec_out_train_work_floats": (I64, [I, I, I, I]),
    "aae_dec_out_scores": (I, [P, I, I, P, P, I, I, P, I64, I, P]),
    "aae_masked_topk": (I, [P, I64, I, I, I, P, P, I, P, P, P, P]),
    "aae_topk_merge": (I, [P, P, I, I, I, P, P, P]),
    "aae_topk_merge_seg": (I, [P, P, I, I, I, I, P, P, P]),
    "aae_rank_counts": (I, [P, I64, I, I, I, P, P, P, P, I, P, I, P, P]),
    "aae_rank_counts_filtered": (I, [P, I64, I, I, I, P, P, P, P, I, P, I, P, P, C.POINTER(AaeRankFilter)]),
    "aae_predict_topk_work_bytes": (I64, [I, I, I]),
    "aae_predict_topk": (I, [P, I, I, P, P, I, I, P, P, I, I, P, I64, P, P, P, P]),
    "aae_pad_weights_floats": (I64, [I, I]),
    "aae_pad_weights": (I, [P, P, I, I, P, P, P]),
    "aae_predict_topk2_work_bytes": (I64, [I, I, I, I]),
    "aae_predict_topk2": (I, [P, I, I, P, P, P, P, I, I, P, P, I, P, I64, P, P, P, P]),
    "aae_gather_item_rows": (I, [P, P, I, I, I, P, I, P, P, P, P]),
    "aae_masked_topk_filtered": (I, [P, I64, I, I, I, P, P, I, P, P, P, P, C.POINTER(AaeRankFilter)]),
    "aae_predict_topk_filtered": (I, [P, I, I, P, P, I, I, P, P, I, I, P, I64, P, P, P, P,
                                      C.POINTER(AaeRankFilter)]),
    "aae_predict_topk2_filtered": (I, [P, I, I, P, P, P, P, I, I, P, P, I, P, I64, P, P, P, P,
                                       C.POINTER(AaeRankFilter)]),
    "aae_tc_selftest": (I, [I, P, P, P, I, P]),
    "aae_upload_batch": (I, [P, P, I, I, P, P, P]),
    "aae_batch_gather": (I, [P, P, P, I64, I, P, P, P, I, P, P]),
    "aae_batch_corrupt": (I, [P, P, I, I, F, P, P, P, P, P]),
    "aae_copy_words_sel": (I, [P, P, P, P, I64, P, I, P]),
    "aae_peer_buffer_bytes": (I64, [I64]),
    "aae_peer_alloc": (I, [I64, C.POINTER(P), C.c_char_p]),
    "aae_peer_open": (I, [C.c_char_p, C.POINTER(P)]),
    "aae_peer_close": (I, [P]),
    "aae_peer_free": (I, [P]),
    "aae_peer_allreduce": (I, [AaePeers, I, P, I, P, I, I64, P]),
    "aae_peer_error": (I, [P, C.POINTER(I)]),
    "aae_peer_bag_allreduce": (I, [AaePeers, I, P, P, I, P, P, I, I, I, I, P, I64, P]),
    "aae_decoder_fwd": (I, [AaeDims, P, P, AaeDrop, AaeDrop, P, P, P, P, I, P]),
    "aae_decoder_bwd": (I, [AaeDims, P, P, AaeDrop, AaeDrop, P, P, P, P, P, P]),
    "aae_decoder_wgrad": (I, [AaeDims, P, P, P, P, P, AdamBlock, P, P]),
    "aae_vae_fwd": (I, [AaeDims, AaeBag, P, P, P, P, P, P, P, P, P, P, P, P, P, P]),
    "aae_vae_bwd": (I, [AaeDims, P, P, P, P, P, P, P, P, P, P, P]),
    "aae_vae_wgrad": (I, [AaeDims, P, P, P, P, P, P, P, AdamBlock, AdamBlock, P, P]),
    "aae_trace_set": (I, [P]),
    "aae_trace_slots": (I, []),
}

EXPORTS = tuple(sorted(_SIGS))

_lib = None


class NativeError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises NativeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "libaae_b200.so is not built (expected at %s); run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C aae-recommender_b200/csrc`.  There is no CPU/PyTorch fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)       # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().aae_last_error().decode("utf-8", "replace")


# kernels launched per entry point (for the bench's gpu_launches claim); memcpy-only calls count 0
KERNELS = {"aae_upload_batch": 0, "aae_w1_sweep_blocked": 2, "aae_batch_gather": 2, "aae_batch_corrupt": 2, "aae_rank_counts": 3, "aae_rank_counts_filtered": 4, "aae_masked_topk": 2, "aae_predict_topk": 6, "aae_predict_topk2": 8, "aae_masked_topk_filtered": 3, "aae_predict_topk_filtered": 6,
           "aae_predict_topk2_filtered": 8, "aae_trace_set": 0, "aae_trace_slots": 0,
           "aae_peer_alloc": 0, "aae_peer_open": 0, "aae_peer_close": 0, "aae_peer_free": 0, "aae_peer_error": 0}
TRACE_NAMES = ("batch_prepare", "w1_sweep_untouched", "ae_fwd", "dec_out_train", "ae_bwd", "ae_wgrad", "w1_rows_update_1",
               "disc_phase", "disc_wgrad", "gen_phase", "gen_wgrad", "w1_rows_update_2", "step_finish", "bag_fwd", "w1_catchup")
_launches = 0


def reset_launch_count():
    global _launches
    _launches = 0


def launch_count():
    return _launches


def count_launch(n=1):
    """Account for kernels launched outside ``call`` (the peer-exchange kernel)."""
    global _launches
    _launches += n


_timing = None   # list of (name, start_event, end_event) while timing is enabled


def enable_timing(on=True):
    """Per-entry-point device timing (CUDA events on the current stream) for eager, non-graph runs."""
    global _timing
    _timing = [] if on else None


def timing_report():
    """{entry point: (calls, mean microseconds)} since enable_timing(); synchronises."""
    import torch
    torch.cuda.synchronize()
    agg = {}
    for name, e0, e1 in _timing or []:
        agg.setdefault(name, []).append(e0.elapsed_time(e1) * 1e3)
    return {k: (len(v), sum(v) / len(v)) for k, v in agg.items()}


def call(name, *args):
    """Invoke an int-returning entry point; non-zero status raises with the library's message."""
    global _launches
    lib = load()
    if _timing is not None:
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(lib, name)(*args)
        e1.record()
        _timing.append((name, e0, e1))
    else:
        rc = getattr(lib, name)(*args)
    _launches += KERNELS.get(name, 1)
    if rc != 0:
        raise NativeError("%s failed (%d): %s" % (name, rc, last_error()))
    return rc


def require_device(dev=0):
    import torch
    if not torch.cuda.is_available():
        raise NativeError("no CUDA device: aaerec_b200 runs only on sm_100 (B200); there is no CPU fallback")
    call("aae_device_check", int(dev))


def drop(mask=None, p=0.0, stream_id=0):
    return AaeDrop(P(mask.data_ptr()) if mask is not None else None, float(p), int(stream_id))


def bag(indptr=None, indices=None, W1t=None, normalize=1, v_begin=0, v_end=0):
    if indptr is None:
        return AaeBag(None, None, None, 0, 0, 0)
    return AaeBag(P(indptr.data_ptr()), P(indices.data_ptr()), P(W1t.data_ptr()), int(normalize), int(v_begin),
                  int(v_end))


def adam_block(p=None, m=None, v=None, which=0):
    if p is None:
        return AdamBlock(None, None, None, 0)
    return AdamBlock(P(p.data_ptr()), P(m.data_ptr()), P(v.data_ptr()), int(which))


def ptr(t):
    return P(t.data_ptr()) if t is not None else None
