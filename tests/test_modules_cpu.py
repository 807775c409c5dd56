"""Host-side logic of the module mirror: construction, state_dict contract, init parity, error paths.
No compute (there is no CPU path to compute with)."""
import copy
import ctypes
import io
import os
import re
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import ROOT, build_module, golden_index, load_golden, quiet, state_dict_from_golden

CASES = golden_index()


@pytest.mark.parametrize("case", CASES[:11], ids=[c["name"] for c in CASES[:11]])
def test_state_dict_keys_shapes_and_init_stream_match_reference(case):
    """Same seed -> bit-identical parameters (same RNG consumption order, same distribution)."""
    g = load_golden(case["name"])
    ref_sd = state_dict_from_golden(g)
    torch.manual_seed(case["seed"])
    m = build_module(case)
    sd = m.state_dict()
    assert list(sd.keys()) == list(ref_sd.keys())
    for k in sd:
        assert tuple(sd[k].shape) == tuple(ref_sd[k].shape), k
        assert torch.equal(sd[k], ref_sd[k]), k
    m.load_state_dict(ref_sd)            # reference checkpoints load


def test_param_count_and_attributes():
    m = quiet(tr.TTLSTM, 40, 256, 3, torch.device("cpu"), n_cores=3, tt_rank=8)
    assert m.param_count() == 35840                       # SURVEY.md section 8a-9, cfg3
    g = quiet(tr.TTGRU, 1, 256, 1, torch.device("cpu"), n_cores=2, tt_rank=4)
    assert g.param_count() == 5344                        # cfg2
    for attr in ("input_size", "hidden_size", "num_layers", "bias", "device", "log_grads", "n_cores",
                 "tt_rank", "is_naive", "new_core", "_all_layers"):
        assert hasattr(m, attr), attr
    assert m._all_layers[1] is m.cell1
    lin = m.cell0.input_weights
    assert lin.shape == [[2, 4, 5], [8, 8, 16]]
    assert lin.weight_t.raw_shape == [[8, 8, 16], [2, 4, 5]]
    assert lin.weight_t.shape == [1024, 40]
    assert lin.weight_t.ranks == [1, 8, 8, 1]
    assert lin.weight_t.ndims == 3
    assert callable(lin.parameters) and len(list(lin.parameters())) == 4
    h, c = m.init_hidden(5)
    assert h.shape == (5, 256) and c.shape == (5, 256) and float(h.abs().sum()) == 0.0


def test_cores_shared_between_weight_t_and_parameter_list():
    m = quiet(tr.TTGRU, 12, 24, 2, torch.device("cpu"), n_cores=2, tt_rank=2)
    for mod in (m, copy.deepcopy(m), copy.deepcopy(m).double()):
        lin = mod.cell1.hidden_weights
        plist = lin._modules["parameters"]
        for a, b in zip(lin.weight_t.tt_cores, plist):
            assert a is b
    assert all(getattr(p, "is_tt", False) for p in m.cell1.hidden_weights._modules["parameters"])


def test_bias_false_drops_bias_keys():
    m = quiet(tr.TTGRU, 28, 64, 2, torch.device("cpu"), n_cores=3, tt_rank=3, bias=False)
    assert not any(k.endswith(".bias") for k in m.state_dict())
    assert m.cell0.input_weights.bias is None


def test_new_core_variants_build_with_reference_shapes():
    m = quiet(tr.TTLSTM, 40, 64, 1, torch.device("cpu"), n_cores=2, tt_rank=2, new_core="last")
    shapes = [tuple(p.shape) for p in m.cell0.input_weights.weight_t.tt_cores]
    assert shapes == [(1, 8, 5, 2), (2, 8, 8, 2), (2, 4, 1, 1)]
    m = quiet(tr.TTGRU, 40, 64, 1, torch.device("cpu"), n_cores=2, tt_rank=2, new_core="first")
    assert tuple(m.cell0.hidden_weights.weight_t.tt_cores[0].shape) == (1, 3, 1, 2)


def test_invalid_options_fail_loudly():
    with pytest.raises(AssertionError):
        quiet(tr.TTGRU, 4, 8, 1, torch.device("cpu"), n_cores=2, tt_rank=2, new_core="middle")


def test_no_cpu_fallback():
    m = quiet(tr.TTLSTM, 4, 8, 1, torch.device("cpu"), n_cores=2, tt_rank=2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(2, 3, 4))
    lin = quiet(tr.TTLinear, in_features=16, out_features=8, d=2, tt_rank=2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        lin(torch.zeros(2, 16))
    with pytest.raises(NameError):
        m(torch.zeros(2, 0, 4))


def test_ttlinear_prints_like_reference_and_matches_init():
    buf = io.StringIO()
    torch.manual_seed(2000)
    with redirect_stdout(buf):
        lin = tr.TTLinear(in_features=256, out_features=10, bias=True, auto_shapes=True, d=2, tt_rank=4)
    assert "Created TTLinear layer with input shape: [16, 16]. output shape: [2, 5]" in buf.getvalue()
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "ttlinear_0.npz")))
    for k, v in lin.state_dict().items():
        assert torch.equal(v, torch.from_numpy(g["param:" + k])), k


def test_tensor_train_full_matches_oracle_dense():
    from helpers import oracle
    lin = quiet(tr.TTLinear, in_features=40, out_features=64, d=3, tt_rank=4)
    w = lin.weight_t.full()
    assert w.shape == (64, 40)
    assert torch.allclose(w, oracle.tt_dense([c.detach() for c in lin.weight_t.tt_cores]), atol=1e-6)


# ---- the C-ABI library: loads on a CPU-only box and exports what the header declares ----------
def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    declared = set(re.findall(r"\b(ttrnn_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found"
    lib = ctypes.CDLL(_lib.lib_path())
    for name in declared:
        assert hasattr(lib, name), "library does not export %s" % name
    assert declared == set(_lib.SYMBOLS), "python binding and header disagree: %s" % (declared ^ set(_lib.SYMBOLS))
    assert _lib.load().ttrnn_abi_version() == _lib.ABI_VERSION == 4


def test_struct_layout_matches_header():
    # sizes implied by include/ttrnn_b200.h
    assert ctypes.sizeof(_lib.TTShape) == 4 * (1 + 6 + 6 + 7)
    assert ctypes.sizeof(_lib.RnnDesc) == 4 * 6 + 8 + 2 * 8 * ctypes.sizeof(_lib.TTShape)
    assert ctypes.sizeof(_lib.RnnWorkspace) == 8 * (3 + _lib.PLAN_WORDS)


def test_descriptor_validation_without_gpu():
    lib = _lib.load()
    m = quiet(tr.TTLSTM, 40, 256, 3, torch.device("cpu"), n_cores=3, tt_rank=8)
    d = m.spec().desc(8, 5)
    assert lib.ttrnn_rnn_param_count(ctypes.byref(d)) == 35840
    d2 = quiet(tr.TTGRU, 1, 256, 1, torch.device("cpu"), n_cores=2, tt_rank=4).spec().desc(4, 4)
    assert lib.ttrnn_rnn_param_count(ctypes.byref(d2)) == 5344
    bad = m.spec().desc(8, 5)
    bad.hidden_size = 128
    assert lib.ttrnn_rnn_param_count(ctypes.byref(bad)) == -1
    assert b"expected" in lib.ttrnn_last_error()
    bad.hidden_size = 256


def test_every_registered_static_kernel_fits_shared_memory():
    """The registry silently skips a static kernel whose shared-memory footprint exceeds the 227 KB opt-in limit
    (the shape then runs on the slow runtime-shape kernels).  Every kernel compiled into the library must fit."""
    import ctypes
    from tensorized_rnn_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(1 << 16)
    n = lib.ttrnn_static_kernel_table(buf, len(buf))
    assert n > 0
    rows = [ln.split("|") for ln in buf.value.decode().strip().splitlines()]
    assert len(rows) >= 30
    too_big = [r for r in rows if r[4] != "1"]
    assert not too_big, too_big
    assert {r[0] for r in rows} == {"rnn_fwd", "rnn_bwd", "ttl_fwd", "ttl_bwd"}


# A stand-in for the reference's import layout: the module names compat.patch_reference() rewrites, and a caller that,
# like the reference's experiments/digit_classification/mnist_classifier.py, imports the classes by name at import time
# and picks them at construction time.  The stand-in classes only need to be distinct from the B200 ones.
_STANDIN_REFERENCE = {
    "tensorized_rnn/__init__.py": "",
    "tensorized_rnn/rnn_utils.py": "class ActivGradLogger(object):\n    pass\n",
    "tensorized_rnn/tt_lstm.py": "import torch\n\nclass TTLSTMCell(torch.nn.Module):\n    pass\n\n"
                                 "class TTLSTM(torch.nn.Module):\n    def __init__(self, *args, **kwargs):\n"
                                 "        super().__init__()\n",
    "tensorized_rnn/gru.py": "import torch\nfrom tensorized_rnn.rnn_utils import ActivGradLogger\n\n"
                             "class GRUCell(torch.nn.Module):\n    pass\n\nclass GRU(torch.nn.Module):\n    pass\n\n"
                             "class TTGRUCell(torch.nn.Module):\n    pass\n\n"
                             "class TTGRU(torch.nn.Module):\n    def __init__(self, *args, **kwargs):\n"
                             "        super().__init__()\n",
    "tensorized_rnn/lstm.py": "import torch\nfrom tensorized_rnn.rnn_utils import ActivGradLogger\n\n"
                              "class LSTMCell(torch.nn.Module):\n    pass\n\nclass LSTM(torch.nn.Module):\n    pass\n",
    "tensorized_rnn/tt_linearset.py": "import torch\n\nclass TTLinearSet(torch.nn.Module):\n    pass\n",
    "t3nsor/__init__.py": "from t3nsor.layers import TTLinear\n",
    "t3nsor/layers.py": "import torch\n\nclass TTLinear(torch.nn.Module):\n    def __init__(self, *args, **kwargs):\n"
                        "        super().__init__()\n",
    "mnist_classifier.py": "import torch\nfrom tensorized_rnn.tt_lstm import TTLSTM\nfrom tensorized_rnn.gru import TTGRU\n"
                           "from t3nsor.layers import TTLinear\n\n"
                           "class MNIST_Classifier(torch.nn.Module):\n"
                           "    def __init__(self, in_size, emb_size, hidden, n_layers, device, tt, gru, n_cores, tt_rank):\n"
                           "        super().__init__()\n"
                           "        cls = TTGRU if gru else TTLSTM\n"
                           "        self.rnn = cls(in_size, hidden, n_layers, device, n_cores=n_cores, tt_rank=tt_rank)\n"
                           "        self.linear = TTLinear(in_features=hidden, out_features=emb_size, bias=True,\n"
                           "                               auto_shapes=True, d=n_cores, tt_rank=tt_rank)\n",
}


def test_patch_reference_switches_the_callers_over(tmp_path):
    """compat.patch_reference(): a caller of the reference's modules then builds the B200 modules, with the
    reference's own state_dict layout and, from the same seed, the reference's own parameters (the stored
    parameters of the reference TTLSTM of the golden case lstm_d2r2_L2_small); unpatch_reference() restores the
    reference's classes."""
    import sys
    import tensorized_rnn_b200.compat as compat
    for rel, text in _STANDIN_REFERENCE.items():
        path = tmp_path / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(text)
    case = next(c for c in golden_index() if c["name"] == "lstm_d2r2_L2_small")
    g = load_golden(case["name"])
    args = (case["input_size"], 10, case["hidden_size"], case["num_layers"], torch.device("cpu"))
    kw = dict(tt=True, gru=False, n_cores=case["n_cores"], tt_rank=case["tt_rank"])
    standin = ("tensorized_rnn", "t3nsor", "mnist_classifier")
    sys.path.insert(0, str(tmp_path))
    try:
        import mnist_classifier as mc
        import tensorized_rnn.tt_lstm as ref_tt
        ref_cls = ref_tt.TTLSTM
        ref = mc.MNIST_Classifier(*args, **kw)
        with redirect_stdout(io.StringIO()):
            n = compat.patch_reference()
            assert n >= 4
            torch.manual_seed(case["seed"])
            ours = mc.MNIST_Classifier(*args, **kw)
        assert isinstance(ours.rnn, tr.TTLSTM) and not isinstance(ref.rnn, tr.TTLSTM)
        assert isinstance(ours.linear, tr.TTLinear) and not isinstance(ref.linear, tr.TTLinear)
        sd = ours.state_dict()
        ref_rnn = {"rnn." + k: v for k, v in state_dict_from_golden(g).items()}
        # state_dict layout of the reference's TTLinear (d = 2, with bias), from its stored fixture
        ref_linear = ["linear." + k for k in state_dict_from_golden(load_golden("ttlinear_0"))]
        assert case["n_cores"] == 2
        assert list(sd.keys()) == list(ref_rnn.keys()) + ref_linear
        for k, v in ref_rnn.items():
            assert tuple(sd[k].shape) == tuple(v.shape), k
            assert torch.equal(sd[k], v), k                                  # same RNG stream -> identical parameters
        ours.rnn.load_state_dict(state_dict_from_golden(g))                  # reference checkpoints load
        compat.unpatch_reference()
        assert ref_tt.TTLSTM is ref_cls and mc.TTLSTM is ref_cls
    finally:
        compat.unpatch_reference()
        sys.path.remove(str(tmp_path))
        for name in list(sys.modules):
            if name.split(".")[0] in standin:
                del sys.modules[name]


def test_ih_route_selection_is_host_logic():
    """Contraction order of the batched ih projection per layer (ttrnn_rnn_ih_route): rank-one for I = 1, dense where
    I*G*H is at most 1.3x the chain's multiply-adds (4x when no static chain kernel exists), else the TT chain.
    Pure host logic: runs without a GPU."""
    import ctypes
    from tensorized_rnn_b200 import _lib
    lib = _lib.load()

    def routes(cls, I, H, L, d, r):
        m = quiet(cls, I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r)
        desc = m.spec().desc(8, 16)
        out = []
        for l in range(L):
            cm, dm = ctypes.c_int64(0), ctypes.c_int64(0)
            out.append((lib.ttrnn_rnn_ih_route(ctypes.byref(desc), l, ctypes.byref(cm), ctypes.byref(dm)), cm.value, dm.value))
        return out

    assert [r[0] for r in routes(tr.TTGRU, 1, 256, 1, 2, 4)] == [2]                       # cfg2: rank-one input
    r3 = routes(tr.TTLSTM, 40, 256, 3, 3, 8)                                              # cfg3
    assert [r[0] for r in r3] == [1, 1, 1]
    assert r3[0][1:] == (87040, 40960) and r3[1][1:] == (327680, 262144)                  # SURVEY 8a-5 / DESIGN 4.5
    r4 = routes(tr.TTLSTM, 40, 256, 3, 4, 16)                                             # cfg4
    assert [r[0] for r in r4] == [1, 1, 1] and r4[1][1:] == (2195456, 262144)
    r5 = routes(tr.TTLSTM, 256, 1024, 1, 4, 8)                                            # cfg5
    assert r5 == [(1, 933888, 1048576)]
    assert [r[0] for r in routes(tr.TTLSTM, 30, 50, 1, 3, 4)] == [0]                      # G*H = 200: not a multiple of 128
    lib.ttrnn_set_option(b"dense_ih", 0)
    try:
        assert [r[0] for r in routes(tr.TTLSTM, 40, 256, 3, 3, 8)] == [0, 0, 0]
    finally:
        lib.ttrnn_set_option(b"dense_ih", 1)
    assert lib.ttrnn_set_option(b"no_such_option", 1) != 0
    assert lib.ttrnn_set_option(b"save_bytes", 1) != 0


def test_header_is_valid_c_and_matches_the_binding():
    """include/ttrnn_b200.h must compile as plain C99 (it is the drop-in boundary for non-C++ hosts) and declare
    exactly the functions the ctypes binding knows."""
    import shutil
    import subprocess
    import tempfile
    from tensorized_rnn_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = os.path.join(root, "include", "ttrnn_b200.h")
    gcc = shutil.which("gcc")
    if gcc:
        with tempfile.TemporaryDirectory() as td:
            src = os.path.join(td, "t.c")
            with open(src, "w") as f:
                f.write('#include "ttrnn_b200.h"\nint main(void) { ttrnn_rnn_desc d; (void)d; return TTRNN_ABI_VERSION == 4 ? 0 : 1; }\n')
            res = subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.dirname(hdr), src],
                                 capture_output=True, text=True)
            assert res.returncode == 0, res.stderr
    text = open(hdr).read()
    declared = set(re.findall(r"\b(ttrnn_[a-z0-9_]+)\s*\(", text))
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
