import glob
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


class Sampled:
    """A reference array stored as a seeded sample (oracle/golden_format.py): its values at fixed flat positions and
    the max |value| of the whole array."""

    def __init__(self, z, key):
        self.shape = tuple(int(n) for n in z[key + "@shape"])
        self.idx = torch.from_numpy(z[key + "@idx"].astype(np.int64))
        self.val = torch.from_numpy(z[key + "@val"])
        self.absmax = float(z[key + "@absmax"])

    def rel(self, a):
        """max |a - ref| / max |ref| over the sampled positions, with the whole array's max |ref|"""
        a = torch.as_tensor(a).detach().cpu()
        assert tuple(a.shape) == self.shape, (tuple(a.shape), self.shape)
        d = (a.reshape(-1)[self.idx].double() - self.val.double()).abs().max()
        return float(d) / (self.absmax if self.absmax > 0 else 1.0)


def _load_entries(z, prefix):
    out = {}
    for k in z.files:
        if k.startswith(prefix) and "@" not in k:
            out[k[len(prefix):]] = torch.from_numpy(z[k])
        elif k.startswith(prefix) and k.endswith("@idx"):
            out[k[len(prefix):-4]] = Sampled(z, k[:-4])
    return out


def reference_initial_state(meta):
    """the initial state_dict of a fixture: default initialisation under INIT_SEED, then the BatchNorm perturbation;
    the generator is returned to draw the inputs from"""
    import deepspeech_pytorch_b200 as ds
    from oracle import golden_format as GF
    rt = getattr(ds.RNNType, meta["rnn_type"])
    if meta["bidirectional"]:
        cfg = ds.BiDirectionalConfig(rnn_type=rt, hidden_size=meta["hidden_size"], hidden_layers=meta["hidden_layers"])
    else:
        cfg = ds.UniDirectionalConfig(rnn_type=rt, hidden_size=meta["hidden_size"],
                                      hidden_layers=meta["hidden_layers"], lookahead_context=meta["lookahead_context"])
    torch.manual_seed(GF.INIT_SEED)
    model = ds.DeepSpeech(ds.LABELS, cfg, 32, ds.AdamConfig(), ds.SpectConfig())
    g = torch.Generator().manual_seed(GF.DATA_SEED)
    GF.perturb_batchnorm(model, g)
    return {k: v.detach().clone() for k, v in model.state_dict().items()}, g


class Golden:
    """One fixture written by oracle/make_golden.py (outputs of the reference itself).  The initial parameters and
    the input are recomputed from their seeds and must match the reference's digests bit for bit."""

    def __init__(self, name):
        from oracle import golden_format as GF
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
        self.name = name
        self.meta = json.loads(str(z["meta"]))
        self.z = z
        self.param_spec = self.meta["params"]          # [key, shape, sha256] in the reference's state_dict order
        self.params, g = reference_initial_state(self.meta)
        assert [[k, list(v.shape), GF.digest(v)] for k, v in self.params.items()] == self.param_spec, \
            f"{name}: the recomputed initial parameters differ from the reference's"
        self.x = GF.spectrograms(g, self.meta["B"], self.meta["T"], self.meta["lengths"])
        assert GF.digest(self.x) == self.meta["x"], f"{name}: the recomputed input differs from the reference's"
        self.grads = _load_entries(z, "g/")
        self.buffers_after = _load_entries(z, "b1/")
        self.taps = _load_entries(z, "tap/")
        self.targets = torch.from_numpy(z["targets"])
        self.input_percentages = torch.from_numpy(z["input_percentages"])
        self.target_sizes = torch.from_numpy(z["target_sizes"])
        self.input_sizes = torch.from_numpy(z["input_sizes"])
        self.output_sizes = torch.from_numpy(z["output_sizes"])
        self.logits = torch.from_numpy(z["logits"])
        self.loss = float(z["loss"])
        self.eval_out = torch.from_numpy(z["eval_out"])

    def oracle_cfg(self):
        from oracle.ds2_oracle import OracleConfig
        m = self.meta
        return OracleConfig(rnn_type=m["rnn_type"], hidden_size=m["hidden_size"], hidden_layers=m["hidden_layers"],
                            bidirectional=m["bidirectional"], lookahead_context=m["lookahead_context"] or 20)


@pytest.fixture(params=golden_names())
def golden(request):
    return Golden(request.param)


def rel_err(a, b):
    """max |a-b| / max |b|  — the 'rel' of the north_star tolerance (1e-3 rel, fp32)."""
    if isinstance(b, Sampled):
        return b.rel(a)
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    denom = float(b.abs().max())
    return float((a - b).abs().max()) / (denom if denom > 0 else 1.0)
