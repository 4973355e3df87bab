"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol that
include/ds2_b200.h declares; host-only entry points are exact; the shell keeps the reference's
state_dict surface.  No GPU compute here."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, golden_names, Golden

import deepspeech_pytorch_b200 as ds
from deepspeech_pytorch_b200 import _lib


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "ds2_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(ds2_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    syms = header_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/ds2_b200.h but not exported"
    assert set(syms) == set(_lib.PROTOTYPES), "ctypes prototypes out of sync with the header"


def test_version_and_error_string():
    lib = ds.get_lib()
    assert b"sm_100a" in lib.ds2_version()
    assert lib.ds2_set_precision(7) != 0
    assert b"precision" in lib.ds2_last_error()


def test_seq_lens_host_bit_exact():
    # reference model.py:299-310 == ((L + 2*5 - 10 - 1)//2 + 1, then //1 + 1)
    L = np.arange(0, 5000, dtype=np.int32)
    out = np.empty_like(L)
    assert ds.get_lib().ds2_seq_lens_host(L.ctypes.data, L.size, out.ctypes.data) == 0
    ref = (L.astype(np.int64) + 10 - 10 - 1) // 2 + 1
    ref = (ref + 10 - 10 - 1) // 1 + 1
    assert np.array_equal(out, ref.astype(np.int32))
    from oracle import ds2_oracle as O
    assert O.get_seq_lens(torch.from_numpy(L)).tolist() == out.tolist()


def test_missing_gpu_fails_loudly():
    m = ds.DeepSpeech(ds.LABELS, ds.BiDirectionalConfig(hidden_size=8, hidden_layers=1), 32, ds.AdamConfig(),
                      ds.SpectConfig())
    with pytest.raises(ds.Ds2Error):
        m(torch.zeros(1, 1, 161, 20), torch.tensor([20]))
    if not torch.cuda.is_available():
        assert ds.get_lib().ds2_device_check(None, None, None) != 0


@pytest.mark.parametrize("name", golden_names())
def test_state_dict_surface_matches_reference(name):
    g = Golden(name)
    m = g.meta
    rt = getattr(ds.RNNType, m["rnn_type"])
    if m["bidirectional"]:
        cfg = ds.BiDirectionalConfig(rnn_type=rt, hidden_size=m["hidden_size"], hidden_layers=m["hidden_layers"])
    else:
        cfg = ds.UniDirectionalConfig(rnn_type=rt, hidden_size=m["hidden_size"], hidden_layers=m["hidden_layers"],
                                      lookahead_context=m["lookahead_context"])
    model = ds.DeepSpeech(ds.LABELS, cfg, 32, ds.AdamConfig(), ds.SpectConfig())
    sd = model.state_dict()
    assert list(sd.keys()) == [k for k, _, _ in g.param_spec]
    for k, shape, _ in g.param_spec:
        assert list(sd[k].shape) == shape, k
    model.load_state_dict(g.params)  # strict


@pytest.mark.parametrize("name", golden_names())
def test_default_init_is_bit_identical_to_the_reference(name):
    """The fixtures hold digests of the state_dict the REFERENCE's own constructor produced under
    torch.manual_seed(123456) (oracle/make_golden.py; only the BatchNorm affine parameters / running statistics were
    overwritten afterwards).
    The shell keeps its parameters in the same torch container classes, created in the same order, so the same seed
    must give bit-identical conv / recurrent / lookahead / fc weights: a drop-in replacement starts training from
    the same point as the reference."""
    g = Golden(name)
    m = g.meta
    rt = getattr(ds.RNNType, m["rnn_type"])
    if m["bidirectional"]:
        cfg = ds.BiDirectionalConfig(rnn_type=rt, hidden_size=m["hidden_size"], hidden_layers=m["hidden_layers"])
    else:
        cfg = ds.UniDirectionalConfig(rnn_type=rt, hidden_size=m["hidden_size"], hidden_layers=m["hidden_layers"],
                                      lookahead_context=m["lookahead_context"])
    from oracle.golden_format import digest
    reference = {k: d for k, _, d in g.param_spec}
    torch.manual_seed(123456)
    model = ds.DeepSpeech(ds.LABELS, cfg, 32, ds.AdamConfig(), ds.SpectConfig())
    checked = 0
    for k, v in model.state_dict().items():
        is_bn = ("batch_norm" in k or "seq_module.1." in k or "seq_module.4." in k or "module.0." in k)
        if is_bn:
            continue
        assert digest(v) == reference[k], k
        checked += 1
    assert checked >= 4 + 4 * m["hidden_layers"]


def test_configs_mirror_reference_defaults():
    assert ds.BiDirectionalConfig().hidden_size == 1024 and ds.BiDirectionalConfig().hidden_layers == 5
    assert ds.UniDirectionalConfig().lookahead_context == 20
    a = ds.AdamConfig()
    assert (a.learning_rate, a.learning_anneal, a.weight_decay, a.eps, a.betas) == (1.5e-4, 0.99, 1e-5, 1e-8, (0.9, 0.999))
    assert ds.SGDConfig().momentum == 0.9
    assert ds.SpectConfig().sample_rate == 16000 and ds.LABELS[0] == "_" and len(ds.LABELS) == 29
