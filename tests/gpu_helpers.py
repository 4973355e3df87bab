"""Shared by the -m gpu tests: build the shell from a fixture / oracle params, error metrics."""
import torch

import deepspeech_pytorch_b200 as ds
from conftest import Sampled
from oracle import ds2_oracle as O


def make_model(rnn_type, bidirectional, H, layers, ctx=20, params=None, device="cuda"):
    rt = getattr(ds.RNNType, rnn_type)
    if bidirectional:
        cfg = ds.BiDirectionalConfig(rnn_type=rt, hidden_size=H, hidden_layers=layers)
    else:
        cfg = ds.UniDirectionalConfig(rnn_type=rt, hidden_size=H, hidden_layers=layers, lookahead_context=ctx)
    m = ds.DeepSpeech(ds.LABELS, cfg, 32, ds.AdamConfig(), ds.SpectConfig())
    if params is not None:
        m.load_state_dict(params)
    return m.to(device)


def model_from_golden(g, device="cuda"):
    m = g.meta
    return make_model(m["rnn_type"], m["bidirectional"], m["hidden_size"], m["hidden_layers"],
                      m["lookahead_context"] or 20, g.params, device)


def rel(a, b):
    if isinstance(b, Sampled):
        return b.rel(a)
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    d = float(b.abs().max())
    return float((a - b).abs().max()) / (d if d > 0 else 1.0)


def oracle_cfg(rnn_type, bidirectional, H, layers, ctx=20):
    return O.OracleConfig(rnn_type=rnn_type, hidden_size=H, hidden_layers=layers, bidirectional=bidirectional,
                          lookahead_context=ctx)


def rel_l2(a, b):
    """||a-b||_2 / ||b||_2 — the noise-robust companion of `rel` for reduced-precision paths"""
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    d = float(b.norm())
    return float((a - b).norm()) / (d if d > 0 else 1.0)
