"""TEST INFRASTRUCTURE — layout of tests/golden/*.npz, shared by the writer (oracle/make_golden.py, which runs the
reference) and the reader (tests/conftest.py).

What a fixture needs but can be recomputed from a seed is not stored: the initial state_dict (the model's default
initialisation under INIT_SEED, then the BatchNorm perturbation below) and the input spectrograms.  The file holds
their SHA-256 digests instead, and the reader recomputes them and checks them bit for bit.  Outputs with more than
FULL_MAX elements (the conv weight gradients, the input-projection gradients of the first recurrent layer, the conv
activations) are stored as SAMPLE values at fixed, seeded flat positions plus the max |value| of the whole array,
so that a relative error against the sample has the same denominator as against the whole array.  Everything else
is stored whole.
"""
import hashlib
import zlib

import numpy as np
import torch

INIT_SEED = 123456   # reference train_config.py:90
DATA_SEED = 7
FULL_MAX = 4096
SAMPLE = 4096


def digest(t) -> str:
    a = np.ascontiguousarray(torch.as_tensor(t).detach().cpu().numpy())
    return hashlib.sha256(a.dtype.str.encode() + str(a.shape).encode() + a.tobytes()).hexdigest()


def perturb_batchnorm(model, g):
    """non-trivial BatchNorm affine parameters and running statistics, so that parity exercises them"""
    with torch.no_grad():
        for k, v in model.state_dict().items():
            if k.endswith("running_mean"):
                v.copy_(0.05 * torch.randn(v.shape, generator=g))
            elif k.endswith("running_var"):
                v.copy_(1.0 + 0.2 * torch.rand(v.shape, generator=g))
            elif "batch_norm" in k or "seq_module.1" in k or "seq_module.4" in k or "module.0" in k:
                if k.endswith(".weight"):
                    v.copy_(1.0 + 0.2 * torch.randn(v.shape, generator=g))
                elif k.endswith(".bias"):
                    v.copy_(0.1 * torch.randn(v.shape, generator=g))


def spectrograms(g, B, T, lengths):
    """N(0, 1) input of shape (B, 1, 161, T), zero beyond each utterance's length"""
    x = torch.randn(B, 1, 161, T, generator=g)
    for b, n in enumerate(lengths):
        x[b, :, :, n:] = 0
    return x


def store(blob, key, a):
    """blob[key] = a, or a seeded sample of it when a is large"""
    a = np.asarray(a)
    if a.size <= FULL_MAX:
        blob[key] = a
        return
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    idx = np.sort(rng.choice(a.size, SAMPLE, replace=False)).astype(np.int32)
    blob[key + "@shape"] = np.array(a.shape, np.int64)
    blob[key + "@idx"] = idx
    blob[key + "@val"] = a.reshape(-1)[idx]
    blob[key + "@absmax"] = np.array(np.abs(a).max(), np.float64)
