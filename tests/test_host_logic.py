"""Host-side logic that needs no GPU: API surface, error conventions, condition protocol, batching."""
import numpy as np
import pytest
import scipy.sparse as sp


def test_constructor_defaults_and_str_match_reference():
    # aae.py:592-606 defaults; __str__ is printed into logs (evaluation.py:355)
    from aaerec_b200.aae import AdversarialAutoEncoder, AAERecommender
    m = AdversarialAutoEncoder()
    assert (m.n_hidden, m.n_code, m.gen_lr, m.reg_lr, m.batch_size, m.n_epochs) == (100, 50, 0.001, 0.001, 100, 500)
    assert m.prior == "gauss" and m.optimizer == "adam" and m.dropout == (.2, .2) and m.normalize_inputs
    s = str(m)
    assert s.startswith("Adversarial Autoencoder (100, 100, 50, 100, 100) optimized by adam")
    assert "Matching the gauss distribution by linear activation." in s
    r = AAERecommender(n_hidden=7, verbose=False)
    assert "Adversarial Autoencoder" in str(r) and "'n_hidden': 7" in str(r)
    assert r.model_params == {"n_hidden": 7, "verbose": False} and r.adversarial


def test_error_conventions():
    from aaerec_b200.aae import AdversarialAutoEncoder
    with pytest.raises(KeyError):          # unknown prior -> KeyError from the table lookup (aae.py:612-613)
        AdversarialAutoEncoder(prior="nope")
    with pytest.raises(KeyError):          # unknown optimizer (aae.py:798)
        AdversarialAutoEncoder(optimizer="rmsprop")
    with pytest.raises(NotImplementedError):
        AdversarialAutoEncoder(activation="SELU")
    m = AdversarialAutoEncoder(verbose=False)
    X = sp.csr_matrix(np.eye(3, dtype=np.float32))
    with pytest.raises(NotImplementedError):   # aae.py:748-749, 770-771
        m.partial_fit(X, y=np.zeros(3))
    with pytest.raises(NotImplementedError):
        m.fit(X, y=np.zeros(3))
    with pytest.raises(AssertionError):        # condition mismatch, condition.py:53-55
        m.fit(X, condition_data=[np.zeros((3, 2))])
    X2 = sp.csr_matrix(np.array([[2.0, 0], [0, 1]]))
    with pytest.raises(RuntimeError):          # non-binary targets (torch BCE's error in the reference)
        m._csr_batch(X2)


def test_csr_batch_from_dense_and_unsorted():
    from aaerec_b200.aae import AdversarialAutoEncoder
    dense = np.array([[0, 1, 1, 0], [0, 0, 0, 0], [1, 0, 0, 1]], dtype=np.float64)
    ip, ii = AdversarialAutoEncoder._csr_batch(dense)
    assert ip.tolist() == [0, 2, 2, 4] and ii.tolist() == [1, 2, 0, 3] and ip.dtype == np.int32
    X = sp.csr_matrix((np.ones(3), np.array([3, 0, 1]), np.array([0, 2, 3])), shape=(2, 4))
    ip, ii = AdversarialAutoEncoder._csr_batch(X)
    assert ii.tolist() == [0, 3, 1]


def test_condition_protocol_shape_contract():
    # reference tests/test_condition.py:28-78: conditioned.size(1) == code.size(1) + size_increment()
    from aaerec_b200.condition import (ConditionList, PrecomputedEmbeddingCondition, ConcatenationBasedConditioning,
                                       ConditionBase, _check_conditions)
    c = PrecomputedEmbeddingCondition(5)
    assert isinstance(c, ConcatenationBasedConditioning) and isinstance(c, ConditionBase)
    code = np.zeros((4, 3), dtype=np.float32)
    rows = np.ones((4, 5))
    out = c.encode_impose(code, rows)
    assert out.shape == (4, 3 + c.size_increment())
    cl = ConditionList([("title", c), ("abstract", PrecomputedEmbeddingCondition(2))])
    assert list(cl.keys()) == ["title", "abstract"] and cl.size_increment() == 7
    out = cl.encode_impose(code, [rows, np.ones((4, 2))])
    assert out.shape == (4, 10)
    from aaerec_b200.condition import CondAdapter
    ad = CondAdapter(cl)
    assert ad.all_rows and ad.size == 7 and ad.kinds == ["rows", "rows"]
    assert ad.encode_all_rows([rows, 2 * np.ones((4, 2))]).shape == (4, 7)
    assert cl.zero_grad() is cl and cl.step() is cl
    assert _check_conditions(None, None) is False
    assert _check_conditions(cl, [rows, rows]) is True
    with pytest.raises(AssertionError):
        _check_conditions(cl, [rows])
    with pytest.raises(AssertionError):
        _check_conditions([("x", c)], [rows])


def test_generic_and_non_concatenating_conditions():
    """A concatenation condition that is not a float-row lookup goes through the generic (Python protocol) path; a
    condition that does not concatenate is outside the envelope and raises."""
    import torch
    from aaerec_b200.condition import ConditionList, ConcatenationBasedConditioning, ConditionBase, CondAdapter

    class Trainable(ConcatenationBasedConditioning):
        def __init__(self):
            self.emb = torch.nn.Embedding(5, 2)
            self.opt = torch.optim.SGD(self.emb.parameters(), lr=1.0)

        def encode(self, inputs):
            return self.emb(torch.as_tensor(inputs))

        def size_increment(self):
            return 2

        def zero_grad(self):
            self.opt.zero_grad()

        def step(self):
            self.opt.step()
    t = Trainable()
    cl = ConditionList([("t", t)])
    ad = CondAdapter(cl)
    assert ad.kinds == ["generic"] and not ad.all_rows
    before = t.emb.weight.detach().clone()
    cl.zero_grad()
    rows, leaves = ad.encode_batch([[1, 3, 3]], torch.device("cpu"), want_grad=True)
    assert rows.shape == (3, 2) and not rows.requires_grad and len(leaves) == 1
    ad.backward_and_step(leaves, torch.ones(3, 2))          # dL/drows = 1 -> SGD moves row 1 by -1, row 3 by -2
    after = t.emb.weight.detach()
    assert torch.allclose(after[1], before[1] - 1) and torch.allclose(after[3], before[3] - 2)
    assert torch.equal(after[0], before[0])
    assert ad.take([10, 11, 12, 13], np.array([2, 0])) == [12, 10]

    class Biasing(ConditionBase):
        def impose(self, inputs, encoded_condition, dim=None):
            return inputs + encoded_condition

        def size_increment(self):
            return 0
    with pytest.raises(NotImplementedError):
        CondAdapter(ConditionList([("b", Biasing())]))


def test_reference_condition_list_is_accepted_by_duck_typing():
    """main.py:103-110 builds aaerec.condition.ConditionList([...PretrainedWordEmbeddingCondition...]); the B200
    classes must take that object as it is (here: the real reference classes when oracle/_ref or /root/reference is
    present, with the vectoriser bypassed as SURVEY 8(c) notes its constructor is broken on this sklearn)."""
    from oracle import reference_loader as RL
    if not RL.reference_available():
        pytest.skip("reference package not present")
    ref = RL.load_reference()
    from aaerec_b200.condition import _check_conditions, CondAdapter
    RC = ref.condition
    pw = RC.PretrainedWordEmbeddingCondition.__new__(RC.PretrainedWordEmbeddingCondition)   # skip the broken ctor
    pw.dim = 1
    import torch
    pw.device = torch.device("cpu")

    class _V(object):
        embedding = np.zeros((10, 6), dtype=np.float32)
    pw.vect = _V()
    cat = RC.CategoricalCondition(embedding_dim=4, reduce="sum", sparse=False, use_cuda=False)
    cat.fit([["a", "b"], ["b"], ["c", "a"]])
    cl = RC.ConditionList([("title", pw), ("journal", cat)])
    data = [np.ones((3, 6)), cat.transform([["a", "b"], ["b"], ["c", "a"]])]
    assert _check_conditions(cl, data) is True
    ad = CondAdapter(cl)
    assert ad.kinds == ["rows", "generic"] and ad.size == 10
    rows, leaves = ad.encode_batch([ad.take(d, np.array([2, 0])) for d in data], torch.device("cpu"), want_grad=True)
    assert rows.shape == (2, 10) and len(leaves) == 1 and leaves[0][1:] == (6, 10)


def test_shard_ranges_cover_vocabulary():
    from aaerec_b200.engine import shard_range
    for V in (1, 7, 100, 200000, 2000001):
        for world in (1, 2, 3, 4, 8):
            parts = [shard_range(V, r, world) for r in range(world)]
            assert parts[0][0] == 0 and parts[-1][1] == V
            for a, b in zip(parts, parts[1:]):
                assert a[1] == b[0]
            assert all(lo <= hi for lo, hi in parts)


def test_synth_sets_are_binary_sorted_unique():
    from aaerec_b200.synth import synth_sets
    X = synth_sets(200, 1000, 8, seed=0)
    assert X.shape == (200, 1000) and X.data.min() == 1 and X.data.max() == 1
    for r in range(200):
        row = X.indices[X.indptr[r]:X.indptr[r + 1]]
        assert np.all(np.diff(row) > 0)
    assert (np.diff(X.indptr) >= 1).all()


def test_plain_autoencoder_api_surface():
    # aae.py:221-247 constructor (lr instead of gen_lr/reg_lr), :321-322 ValueError on y, AAERecommender(adversarial=False)
    from aaerec_b200.aae import AutoEncoder, AAERecommender
    m = AutoEncoder(n_hidden=7, lr=0.01, verbose=False)
    assert (m.n_hidden, m.n_code, m.lr, m.batch_size, m.n_epochs) == (7, 50, 0.01, 100, 500)
    assert m.gen_lr == 0.01 and m.reg_lr == 0.0 and not m.adversarial and m.disc is None
    X = sp.csr_matrix(np.eye(3, dtype=np.float32))
    with pytest.raises(ValueError):
        m.partial_fit(X, y=np.zeros(3))
    with pytest.raises(NotImplementedError):
        m.fit(X, y=np.zeros(3))
    r = AAERecommender(adversarial=False, lr=0.01, verbose=False)
    assert str(r).startswith("Autoencoder") and not r.adversarial


def test_peer_exchange_buffer_layout():
    # the exchange buffer holds a header (flags of 4 exchanges x 32 blocks x 8 ranks, counters) and 2 slots per
    # exchange, each n_max floats + 4 doubles, 256-byte aligned
    from aaerec_b200 import _native as N
    lib = N.load()
    n = 12800
    slot = (n * 4 + 32 + 255) // 256 * 256
    header = (4 * 32 * 8 * 4 + 4 * 4 + 4 * 4 + 32 + 255) // 256 * 256
    assert lib.aae_peer_buffer_bytes(n) == header + 8 * slot
    assert lib.aae_peer_buffer_bytes(0) == 0


def test_fused_topk_envelope_and_workspace():
    # aae_predict_topk_work_bytes is a pure host function: 0 outside the fused envelope (small shards, huge k),
    # positive and growing with the batch inside it
    from aaerec_b200 import _native as N
    lib = N.load()
    assert lib.aae_predict_topk_work_bytes(100, 20000, 100) == 0          # shard below 32,768 items: dense path
    assert lib.aae_predict_topk_work_bytes(100, 200000, 2000) == 0        # k above 1024
    assert lib.aae_predict_topk_work_bytes(0, 200000, 100) == 0
    a = lib.aae_predict_topk_work_bytes(100, 200000, 100)
    b = lib.aae_predict_topk_work_bytes(1000, 200000, 100)
    c = lib.aae_predict_topk_work_bytes(1000, 2000000, 100)
    assert 0 < a < b <= c
    # the score matrix the fused path avoids would be far larger than its whole workspace
    assert c < 1000 * 2000000 * 4 / 8


def test_reference_arm_prints_contract_line():
    # bench.py --impl reference runs the reference's own CPU implementation (oracle/_ref when present, else the CPU
    # port of its algorithm; no GPU needed) and prints ONE JSON line with the contract's keys
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "econbiz",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "sets/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_predict_leg_and_query_set_lengths():
    # the predict legs' host baseline: the reference's own model.predict + remove_non_missing + argtopk (no GPU needed)
    import json
    import os
    import subprocess
    import sys
    import numpy as np
    from aaerec_b200.synth import synth_sets
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference-predict", "--workload",
                          "econbiz", "--predict-batch", "150"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["impl"] == "reference-predict"
    if "unavailable" not in d:            # oracle/_ref (or /root/reference) present
        assert d["kind"] == "reference" and d["value"] > 0 and d["unit"] == "sets/s" and d["cores"] >= 1
    # the MPD challenge's query lengths (create_dev_set.py:16-17): 1 / 5 / 10 / 25 / 100 seed items, before de-duplication
    X = synth_sets(400, 50000, 25, 1, 100, seed=3, len_choices=(1, 5, 10, 25, 100))
    lens = np.diff(X.indptr)
    assert set(np.unique(lens)) <= set(range(1, 101)) and lens.max() > 60 and (lens == 1).sum() > 30
    assert (X.data == 1).all() and all(np.all(np.diff(X.indices[X.indptr[r]:X.indptr[r + 1]]) > 0) for r in range(400))
    # the named shapes of SURVEY 8(d)
    from aaerec_b200.synth import synth_named, SHAPES
    E = synth_named("econbiz", 300)
    assert E.shape == (300, SHAPES["econbiz"][1]) and np.diff(E.indptr).min() >= 1 and np.diff(E.indptr).max() <= 30


def test_peer_struct_layout():
    import ctypes
    from aaerec_b200 import _native as N
    assert ctypes.sizeof(N.AaePeers) == 8 * 8 + 8      # void* base[8]; int rank, world


def test_w1_cold_element_bound_holds_in_float32():
    """The arithmetic behind the cold-row shortcut of the time-blocked W1 sweep (csrc/w1_blocked.cu cold4): with
    |m| <= 2^-110, denom >= eps = 1e-8, step <= 2^10 and |W| >= 2^-40 the zero-gradient Adam update
    W' = fma(-step, m' / denom, W) returns W bit for bit (float32, round to nearest), so skipping it is exact; the moments
    keep decaying through the unchanged operations.  (The kernel itself is checked bit for bit against the full replay
    on the GPU: test_w1_sweep_cold_rows_bit_identical_to_full_replay.)"""
    import numpy as np
    rs = np.random.RandomState(0)
    n = 200000
    f32 = np.float32
    m = (rs.uniform(-1, 1, n) * 2.0 ** -110).astype(f32)
    m[::7] = f32(2.0 ** -110)                                     # the threshold itself
    m[1::7] = f32(-(2.0 ** -110))
    v = (rs.uniform(0, 1, n) ** 8).astype(f32)                    # second moments from 0 to 1
    v[::5] = 0
    w_mag = 2.0 ** rs.uniform(-40, 2, n)
    w = (np.where(rs.rand(n) < 0.5, -1, 1) * w_mag).astype(f32)
    w[::11] = f32(2.0 ** -40)                                     # the smallest admitted magnitude, a power of two
    step = (2.0 ** rs.uniform(-20, 10, n)).astype(f32)
    inv_bc2_sqrt = (1.0 / np.sqrt(1.0 - 0.999 ** rs.randint(1, 5000, n))).astype(f32)
    eps = f32(1e-8)
    m1 = (m - f32(0.1) * m).astype(f32)                          # fma(w1, -m, m) up to one rounding: magnitude only shrinks
    assert np.all(np.abs(m1) <= np.abs(m))
    denom = (np.sqrt(v).astype(f32) * inv_bc2_sqrt + eps).astype(f32)
    assert np.all(denom >= eps)
    q = (m1 / denom).astype(f32)
    # the fma is exact in float64 here (24-bit x 24-bit product, then one addition), rounded once to float32
    w_new = (w.astype(np.float64) - step.astype(np.float64) * q.astype(np.float64)).astype(f32)
    assert np.array_equal(w_new.view(np.int32), w.view(np.int32))
    # m == +0: the increment is -0 and W' == W for EVERY W, also tiny and zero weights
    w_any = np.concatenate([w, f32([0.0, 1e-44, -1e-44, 1e-30])])
    w_any_new = (w_any.astype(np.float64) - np.float64(1024.0) * np.float64(0.0)).astype(f32)
    assert np.array_equal(w_any_new.view(np.int32), w_any.view(np.int32))


def test_overlay_resolves_the_import_block_of_main_py(tmp_path):
    """The zero-edit path of INTEGRATION.md A, on the CPU: with aae-recommender_b200/ in front of the reference on the
    module path, the imports of main.py:11-20 resolve -- recommenders of aaerec.aae / .vae / .dae to the B200 classes,
    everything else to the reference's own modules (runs in a child process: it rebinds the ``aaerec`` package).  The
    reference tree is a stand-in with the reference's module layout (helpers.write_reference_standin), and the real
    reference too when its package is present."""
    import os
    import subprocess
    import sys
    from helpers import write_reference_standin
    from oracle import reference_loader as RL
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    trees = [(write_reference_standin(tmp_path), "")]
    if RL.reference_available():
        trees.append((RL.REFERENCE_ROOT, r'''
from oracle import reference_loader as RL
RL.load_reference()                      # gensim / docutils stubs for the real reference's imports
for k in [k for k in sys.modules if k == "aaerec" or k.startswith("aaerec.")]:
    del sys.modules[k]'''))
    for reference_root, prelude in trees:
        code = r'''
import sys
sys.path.insert(0, %r)%s
sys.path.insert(0, %r)
from aaerec.datasets import Bags
from aaerec.evaluation import Evaluation
from aaerec.aae import AAERecommender, DecodingRecommender
from aaerec.baselines import RandomBaseline, Countbased, MostPopular
from aaerec.svd import SVDRecommender
from aaerec.vae import VAERecommender
from aaerec.dae import DAERecommender
from aaerec.condition import ConditionList, PretrainedWordEmbeddingCondition, CategoricalCondition
mods = [c.__module__ for c in (AAERecommender, DecodingRecommender, VAERecommender, DAERecommender)]
assert mods == ["aaerec_b200.aae", "aaerec_b200.decoding", "aaerec_b200.vae", "aaerec_b200.dae"], mods
for c in (Bags, Evaluation, Countbased, SVDRecommender, ConditionList, CategoricalCondition):
    assert c.__module__.startswith("aaerec.") and "b200" not in c.__module__, c
print("OVERLAY_OK")
''' % (root, prelude, os.path.join(root, "aae-recommender_b200"))
        env = dict(os.environ, AAEREC_REFERENCE=reference_root)
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=env)
        assert out.returncode == 0 and "OVERLAY_OK" in out.stdout, (reference_root, out.stderr[-2000:])


def test_reference_arm_under_torchrun_uses_all_host_threads():
    """The driver launches the reference arm like ours: ``torchrun --nproc-per-node N bench.py --impl reference --gpus N``.
    Rank 0 alone runs and prints ONE line; the other ranks exit 0 without work; torchrun's OMP_NUM_THREADS=1 must not
    cripple the baseline (round-1 verdict: the N>1 ratios were inflated 8x by a 1-thread reference)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    try:
        cores = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        cores = os.cpu_count() or 1
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload",
           "econbiz", "--steps", "2", "--warmup", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
    assert d["cpu_baseline"]["cores"] == cores, (d["cpu_baseline"], cores)
