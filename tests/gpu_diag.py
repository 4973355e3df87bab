"""Not a test: one-shot diagnostic run on the GPU box (every check reports, nothing stops early).
    python tests/gpu_diag.py > gpurun_out/diag.txt
"""
import os
import sys
import time
import traceback

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import deepspeech_pytorch_b200 as ds  # noqa: E402
from conftest import Golden, golden_names  # noqa: E402
from gpu_helpers import make_model, model_from_golden, oracle_cfg, rel  # noqa: E402
from oracle import ds2_oracle as O  # noqa: E402


def section(name):
    print(f"\n=== {name}", flush=True)


def run(name, fn):
    try:
        fn()
    except Exception:
        print(f"[EXC] {name}\n{traceback.format_exc()}", flush=True)


def golden_case(name):
    g = Golden(name)
    model = model_from_golden(g).train()
    taps = {}
    # block-level taps through the ops, replaying the model's forward by hand
    out, out_lens, hs = model(g.x.cuda(), g.input_sizes)
    print(f"{name}: out_lens ok={out_lens.tolist() == g.output_sizes.tolist()} logits rel={rel(out, g.logits):.3e}")
    sd = model.state_dict()
    for k, v in g.buffers_after.items():
        if "num_batches" not in k:
            print(f"   buf {k}: {rel(sd[k], v):.3e}")
    model = model_from_golden(g).train()
    loss = model.training_step((g.x.cuda(), g.targets, g.input_percentages.clone(), g.target_sizes), 0)
    loss.backward()
    print(f"   loss {float(loss):.6f} vs {g.loss:.6f}")
    for k, p in model.named_parameters():
        print(f"   grad {k}: {rel(p.grad, g.grads[k]) if p.grad is not None else 'NONE'}")


def conv_block():
    g = Golden("bilstm_h24_l2")
    model = model_from_golden(g).train()
    sm = model.conv.seq_module
    ol = model.get_seq_lens(g.input_sizes).cuda()
    y = ds.ops.ConvFrontend.apply(g.x.cuda(), ol, sm[0].weight, sm[0].bias, sm[1].weight, sm[1].bias,
                                  sm[1].running_mean, sm[1].running_var, sm[3].weight, sm[3].bias, sm[4].weight,
                                  sm[4].bias, sm[4].running_mean, sm[4].running_var, True, 0.1, 1e-5)
    tap = g.taps["conv"]  # (B,32,41,T'), stored as a seeded sample
    B, C, D, T = tap.shape
    got = y.detach().permute(1, 2, 0).reshape(B, C, D, T)
    print(f"conv tap rel={rel(got, tap):.3e}")


def main():
    print(torch.cuda.get_device_name(0), ds.get_lib().ds2_version())
    ds.set_precision("fp32")
    section("conv block vs reference tap")
    run("conv", conv_block)
    section("golden fixtures (fp32)")
    for n in golden_names():
        run(n, lambda n=n: golden_case(n))
    section("timing: cfg-L-like forward/backward (fp32 FFMA path), B=8 T=400 H=256 x3")
    def timing():
        ocfg = oracle_cfg("lstm", True, 256, 3)
        P = O.init_params(ocfg, seed=1)
        model = make_model("lstm", True, 256, 3, params=P).train()
        x, targets, pct, tsz = O.synth_batch(8, 400, seed=3, ragged=False, lmin=50, lmax=60)
        xc = x.cuda()
        for it in range(3):
            torch.cuda.synchronize(); t0 = time.time()
            model.zero_grad()
            loss = model.training_step((xc, targets, pct.clone(), tsz), 0)
            loss.backward()
            torch.cuda.synchronize()
            print(f"   iter {it}: {1e3 * (time.time() - t0):.1f} ms loss={float(loss):.4f} launches={ds.get_lib().ds2_launch_count(1)}")
    run("timing", timing)


if __name__ == "__main__":
    main()
