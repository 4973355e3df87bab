"""TEST INFRASTRUCTURE — generates tests/golden/*.npz by EXECUTING THE REFERENCE.

Runs only in the dev container (needs /root/reference).  For each small configuration it builds the
reference's own `DeepSpeech` (unmodified deepspeech_pytorch/model.py, imported through
oracle/ref_shim.py), runs `training_step` + `loss.backward()` on seeded synthetic input and stores
digests of the inputs and of the initial state_dict, logits, loss, every parameter gradient, the
post-step BatchNorm buffers, per-block activations (forward hooks) and an eval-mode forward (softmax +
final RNN states), in the layout of oracle/golden_format.py.  These fixtures are what pins
oracle/ds2_oracle.py and the CUDA path to the reference.

    python oracle/make_golden.py            # rewrites tests/golden/*.npz
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import golden_format as GF  # noqa: E402
import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

CASES = {
    # name: (rnn_type, bidirectional, H, layers, ctx, B, T, lengths, target_lengths)
    "bilstm_h24_l2": ("lstm", True, 24, 2, 0, 3, 73, [73, 60, 41], [9, 7, 5]),
    # longest utterance shorter than the padded tensor: T_out = max(output_lengths) < T'
    "bigru_h20_l2": ("gru", True, 20, 2, 0, 4, 64, [57, 57, 40, 23], [8, 11, 6, 4]),
    "unigru_h16_l2_la5": ("gru", False, 16, 2, 5, 3, 50, [50, 33, 20], [6, 5, 10]),  # last one infeasible? (T'=10,L=10 ok)
    "birnn_h12_l3": ("rnn", True, 12, 3, 0, 2, 40, [40, 31], [5, 3]),
    # CTC edge cases: repeated labels, infeasible alignment (zero_infinity), length-1 target
    "bilstm_h8_l1_ctcedge": ("lstm", True, 8, 1, 0, 4, 30, [30, 28, 20, 12], [7, 14, 1, 6]),
}


def build(ns, rnn_type, bidir, H, layers, ctx):
    labels = json.load(open(os.path.join(ref_shim.REFERENCE_ROOT, "labels.json")))
    rt = getattr(ns.RNNType, rnn_type)
    if bidir:
        cfg = ns.BiDirectionalConfig(rnn_type=rt, hidden_size=H, hidden_layers=layers)
    else:
        cfg = ns.UniDirectionalConfig(rnn_type=rt, hidden_size=H, hidden_layers=layers, lookahead_context=ctx)
    return ns.DeepSpeech(labels=labels, model_cfg=cfg, precision=32, optim_cfg=ns.AdamConfig(),
                         spect_cfg=ns.SpectConfig())


def main():
    ns = ref_shim.load_reference()
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)  # deterministic reductions
    for name, (rnn_type, bidir, H, layers, ctx, B, T, lens, tlens) in CASES.items():
        torch.manual_seed(GF.INIT_SEED)
        model = build(ns, rnn_type, bidir, H, layers, ctx)
        g = torch.Generator().manual_seed(GF.DATA_SEED)
        GF.perturb_batchnorm(model, g)
        sd0 = {k: v.detach().clone() for k, v in model.state_dict().items()}

        x = GF.spectrograms(g, B, T, lens)
        pct = torch.tensor([l / float(T) for l in lens], dtype=torch.float32)
        tsz = torch.tensor(tlens, dtype=torch.int32)
        targets = torch.randint(1, 29, (sum(tlens),), generator=g, dtype=torch.int64)
        if name.endswith("ctcedge"):
            targets[0:7] = torch.tensor([3, 3, 3, 5, 5, 1, 1])        # repeats need blanks between
            # utterance 1: L=14 with T'=14 and a repeat -> infeasible -> zero_infinity path
            targets[7:21] = torch.tensor([2, 2, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15])

        taps = {}
        hooks = [model.conv.register_forward_hook(lambda m, i, o: taps.__setitem__("conv", o[0].detach().clone()))]
        for i, r in enumerate(model.rnns):
            hooks.append(r.register_forward_hook(
                lambda m, inp, o, i=i: taps.__setitem__(f"rnn{i}", o[0].detach().clone())))
        if model.lookahead is not None:
            hooks.append(model.lookahead.register_forward_hook(
                lambda m, i, o: taps.__setitem__("lookahead", o.detach().clone())))

        model.train()
        # training_step mutates input_percentages in place (model.py:243) -> hand it a clone
        batch = (x.clone(), targets.clone(), pct.clone(), tsz.clone())
        inputs, tg, ip, ts = batch
        input_sizes = ip.clone().mul_(int(inputs.size(3))).int()
        out, output_sizes, _ = model(inputs, input_sizes)             # for logits capture
        logits = out.detach().clone()
        model.load_state_dict(sd0)                                    # undo the running-stat update
        model.zero_grad()
        loss = model.training_step(batch, 0)
        loss.backward()
        for h in hooks:
            h.remove()
        grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
        sd1 = {k: v.detach().clone() for k, v in model.state_dict().items()}

        model.eval()
        with torch.no_grad():
            eout, eos, ehs = model(x.clone(), input_sizes)
        dec = ns.GreedyDecoder(model.labels)
        _, offsets = dec.decode(eout, eos)
        am = eout.argmax(2)

        params = [[k, list(v.shape), GF.digest(v)] for k, v in sd0.items()]
        blob = {"meta": np.array(json.dumps(dict(rnn_type=rnn_type, bidirectional=bidir, hidden_size=H,
                                                  hidden_layers=layers, lookahead_context=ctx, B=B, T=T,
                                                  lengths=lens, x=GF.digest(x), params=params,
                                                  torch=torch.__version__)))}
        blob["targets"] = targets.numpy()
        blob["input_percentages"] = pct.numpy()
        blob["target_sizes"] = tsz.numpy()
        blob["input_sizes"] = input_sizes.numpy()
        blob["output_sizes"] = output_sizes.numpy()
        blob["logits"] = logits.numpy()
        blob["loss"] = np.array(float(loss.detach()), np.float64)
        for k, v in grads.items():
            GF.store(blob, "g/" + k, v.numpy())
        for k, v in sd1.items():
            if "running_" in k or "num_batches" in k:
                blob["b1/" + k] = v.numpy()
        for k, v in taps.items():
            GF.store(blob, "tap/" + k, v.numpy())
        blob["eval_out"] = eout.numpy()
        blob["eval_argmax"] = am.numpy().astype(np.int64)
        for b in range(B):
            blob[f"eval_offsets/{b}"] = offsets[b][0].numpy().astype(np.int32)
        for i, h in enumerate(ehs):
            if isinstance(h, tuple):
                blob[f"eval_hn/{i}"] = h[0].numpy()
                blob[f"eval_cn/{i}"] = h[1].numpy()
            else:
                blob[f"eval_hn/{i}"] = h.numpy()
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **blob)
        print(f"{name}: loss={float(loss):.6f} out={tuple(logits.shape)} out_sizes={output_sizes.tolist()} "
              f"-> {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
