#!/usr/bin/env python
"""Benchmark of the DeepSpeech2 train step (BASELINE.json metric: utterances/sec, 161x1000 synthetic
spectrograms).  One JSON line on stdout (rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = forward + CTC + backward (+ one gradient all-reduce for N>1) + fused clip/AdamW step on one
batch of B=32 utterances per GPU (weak scaling).  `value` is timed with the batch resident in HBM;
`e2e` repeats the same steps through the public API with pinned-host inputs copied H2D and the loss
read back D2H inside the timed region.  `--impl reference` times the reference's own CPU path (the
oracle port issuing the same ATen calls: oneDNN conv, packed `_VF.lstm`, `ctc_loss`, autograd) on the
host cores of the box, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: rnn_type, bidirectional, H, layers, ctx, B/GPU, T, target_len     (BASELINE.json configs)
    "librispeech": ("lstm", True, 1024, 5, 20, 32, 1000, 200),      # configs[1] / [2]: the headline
    "an4": ("gru", True, 256, 2, 20, 4, 1000, 200),                 # configs[0]
    "unigru_lookahead": ("gru", False, 1024, 5, 20, 32, 1000, 200),  # configs[3]
    "stress": ("lstm", True, 1536, 7, 20, 8, 4000, 400),            # configs[4]
}


T0 = time.time()


def synth_batch(B, T, L, seed):
    """SURVEY.md §8d throughput inputs: N(0,1) spectrograms (B,1,161,T), every utterance T frames long
    (percentages 1.0), every target L labels drawn from 1..28 (0 is the CTC blank); flat int64 targets and int32
    target sizes exactly as the reference's _collate_fn emits them (data_loader.py:247-270)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 1, 161, T, generator=g)
    pct = torch.ones(B, dtype=torch.float32)
    tsz = torch.full((B,), L, dtype=torch.int32)
    targets = torch.randint(1, 29, (B * L,), generator=g, dtype=torch.int64)
    return x, targets, pct, tsz


DUMP_MAX_ELEMS = 1 << 17


def dump_outputs(path, loss, state, grads):
    """--dump-outputs: what the last timed step hands its caller, as <path>/<name>.npy: `loss`, the model's state_dict
    after the optimizer step (parameters and BatchNorm running statistics, under their state_dict keys) and every
    parameter's gradient of that step (`grad.<key>`).  float32, integer buffers as float64.  A tensor of more than
    DUMP_MAX_ELEMS elements is stored as that many values at fixed positions (numpy default_rng(0), sorted flat
    indices), which keeps the largest workload (stress) below 64 MB in all.  At the default precision the librispeech
    step sums its gradients in a fixed order: two runs with the same arguments write identical values.  Other
    workloads and --precision fp32 can reach kernels that still add with float atomics (the lookahead weight
    gradient, the FFMA conv weight / bias gradients, column sums where the recurrent sweep does not produce the bias
    gradients), so their dumps may differ in the last bits from run to run.  The conv biases feed BatchNorm: their
    true gradient is zero and what is dumped for them is rounding noise, not meaningful across builds."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {"loss": np.array([loss], np.float64)}
    for prefix, tensors in (("", state), ("grad.", grads)):
        for k, v in tensors.items():
            a = v.detach().cpu().numpy()
            a = a.astype(np.float32 if v.is_floating_point() else np.float64)
            if a.size > DUMP_MAX_ELEMS:
                a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
            arrays[prefix + k] = a
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    log(f"dumped {len(arrays)} arrays ({sum(a.nbytes for a in arrays.values()) / 2**20:.1f} MiB) to {path}")


def log(msg):
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench +{time.time() - T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


def host_cores():
    """usable host cores: min(affinity mask, cgroup cpu quota) — the GPU boxes expose 128 logical CPUs but the
    container is limited to a quota (cpu.max), and oversubscribing torch's thread pool makes the CPU path crawl"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port, ATen ops) on the host."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import ds2_oracle as O
    rnn, bidir, H, layers, ctx, B, T, L = WORKLOADS[args.workload]
    cores = host_cores()
    torch.set_num_threads(cores)
    Bs = args.cpu_batch
    ocfg = O.OracleConfig(rnn_type=rnn, hidden_size=H, hidden_layers=layers, bidirectional=bidir,
                          lookahead_context=ctx)
    P = O.init_params(ocfg, seed=123456)
    x, targets, pct, tsz = O.synth_batch(Bs, T, seed=1234, ragged=False, lmin=L, lmax=L)

    def step():
        O.train_step(x, targets, pct.clone(), tsz, P, ocfg, use_aten_rnn=True, use_aten_ctc=True)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    v = Bs / dt
    line = {"impl": "reference", "metric": "utterances/sec (train step, 161x1000 spectrogram)", "value": v,
            "unit": "utt/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "rnn": f"{layers}x{'bi' if bidir else 'uni'}-{rnn}-{H}",
                       "frames": T, "target_len": L, "batch_per_step": Bs},
            "cpu_baseline": {"value": v, "unit": "utt/s", "cores": cores, "kind": "port",
                             "sample": f"{args.steps} steps of B={Bs} utterances (fwd+CTC+bwd, torch CPU ATen ops, "
                                       f"{cores} threads)"},
            "e2e": {"value": v, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
def cpu_baseline(workload, timeout_s=150):
    """reference CPU path (oracle port) on a bounded sample, in a subprocess so that a slow host cannot stall
    the bench: 1 warm-up + 2 timed steps of B=2 utterances of the same workload."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload, "--steps", "2",
           "--warmup", "1", "--cpu-batch", "2"]
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env).stdout.strip().splitlines()
        d = json.loads(out[-1])["cpu_baseline"]
        return d
    except subprocess.TimeoutExpired:
        return {"value": None, "unit": "utt/s", "cores": host_cores(), "kind": "port",
                "sample": f"did not finish 3 steps of B=2 within {timeout_s} s"}
    except Exception as e:  # pragma: no cover
        return {"value": None, "unit": "utt/s", "cores": host_cores(), "kind": "port", "sample": f"failed: {e!r}"}


def _oracle_cfg(workload):
    from oracle import ds2_oracle as O
    rnn, bidir, H, layers, ctx, B, T, L = WORKLOADS[workload]
    return O.OracleConfig(rnn_type=rnn, hidden_size=H, hidden_layers=layers, bidirectional=bidir,
                          lookahead_context=ctx)


def stock_cuda_baseline(workload, P0, batch, steps=10, warmup=3):
    """north_star's denominator: the reference's stock PyTorch CUDA path — the ATen calls of reference model.py
    (cuDNN conv / packed cuDNN RNN, ATen CTC, clip_grad_norm_, torch AdamW) issued by the oracle port on the GPU,
    starting from the SAME weights and the SAME batch as the B200 arm.  Three variants so that the comparison is
    not against a handicapped baseline (SURVEY.md §8d):
      default      torch's default flags (cudnn.allow_tf32=True, matmul.allow_tf32=False, cudnn.benchmark=False —
                   reference lightning_config.py:59), fp32
      cudnn_bench  same with cudnn.benchmark=True
      amp_fp16     torch.autocast(float16) + GradScaler: the reference's shipped `precision: 16`
                   (configs/librispeech.yaml:12)"""
    import torch
    import torch.nn.functional as F
    from oracle import ds2_oracle as O
    rnn, bidir, H, layers, ctx, B, T, L = WORKLOADS[workload]
    ocfg = _oracle_cfg(workload)
    x, targets, pct, tsz = batch
    dev = x.device
    res = {}
    saved = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    for name, bench_flag, amp in (("default", False, False), ("cudnn_bench", True, False), ("amp_fp16", False, True)):
        try:
            torch.backends.cudnn.benchmark = bench_flag
            torch.backends.cudnn.allow_tf32 = True
            torch.backends.cuda.matmul.allow_tf32 = False
            P = {k: v.detach().clone() for k, v in P0.items()}
            leaves = {k: v.requires_grad_(True) for k, v in P.items()
                      if v.dtype.is_floating_point and "running_" not in k}
            opt = torch.optim.AdamW(list(leaves.values()), lr=1.5e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-5)
            scaler = torch.amp.GradScaler("cuda", enabled=amp)
            sizes = O.input_sizes_from_percentages(pct.clone(), T)

            def step():
                with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                    out, osz, _, nb = O.forward(x, sizes, P, ocfg, training=True, use_aten_rnn=True)
                    loss = F.ctc_loss(out.transpose(0, 1).float().log_softmax(-1), targets, osz, tsz, blank=0,
                                      reduction="sum", zero_infinity=True)
                for k, v in nb.items():          # running statistics advance like nn.BatchNorm's buffers
                    P[k] = v.detach()
                opt.zero_grad(set_to_none=True)
                scaler.scale(loss).backward()
                scaler.unscale_(opt)
                torch.nn.utils.clip_grad_norm_(list(leaves.values()), 400.0)
                scaler.step(opt)
                scaler.update()
                return loss

            first = None
            for i in range(warmup):
                l = step()
                if i == 0:
                    first = float(l.detach())
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            res[name] = {"value": B / (ms * 1e-3), "unit": "utt/s", "ms_per_step": ms, "steps": steps,
                         "first_step_loss": first}
        except Exception as e:  # pragma: no cover
            res[name] = {"error": repr(e)[:300]}
        finally:
            (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
             torch.backends.cuda.matmul.allow_tf32) = saved
        torch.cuda.empty_cache()
    res["kind"] = ("stock torch CUDA ops (cuDNN conv/RNN, ATen CTC, clip_grad_norm_, torch AdamW) issued by the "
                   "oracle port; same initial weights and batch as the B200 arm")
    return res


def _group_of(name):
    if name.startswith("conv."):
        return "conv"
    if name.startswith("rnns."):
        i = name.split(".")[1]
        kind = ("bn" if "batch_norm" in name else "w_ih" if "weight_ih" in name else
                "w_hh" if "weight_hh" in name else "bias")
        return f"rnn{i}.{kind}"
    if name.startswith("lookahead"):
        return "lookahead"
    return "fc.bn" if "module.0" in name else "fc.w"


def parity_fullsize(workload, model, flat, P0, batch):
    """The benchmarked configuration against the fp32 reference arithmetic, at full size and with the same weights:
    the B200 arm (current precision mode) vs the reference's own ATen calls on the GPU with every TF32 switch OFF
    (cuDNN fp32 conv/RNN, fp32 matmul) and the CTC lattice in float64.  `oracle/` is the checker here, nothing of
    it is timed.  Reports logits / loss / per-parameter-group gradient errors (rel = max|a-b| / max|b|,
    rel_l2 = ||a-b|| / ||b||)."""
    import torch
    import torch.nn.functional as F
    from oracle import ds2_oracle as O
    rnn, bidir, H, layers, ctx, B, T, L = WORKLOADS[workload]
    ocfg = _oracle_cfg(workload)
    x, targets, pct, tsz = batch
    sizes = O.input_sizes_from_percentages(pct.clone(), T)

    def rel(a, b):
        d = float(b.abs().max())
        return float((a - b).abs().max()) / (d if d > 0 else 1.0)

    def rel_l2(a, b):
        d = float(b.double().norm())
        return float((a.double() - b.double()).norm()) / (d if d > 0 else 1.0)

    # ---- reference arithmetic (fp32 everywhere, CTC in fp64)
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = False
    def reference_arm():
        P = {k: v.detach().clone() for k, v in P0.items()}
        leaves = {k: v.requires_grad_(True) for k, v in P.items() if v.dtype.is_floating_point and "running_" not in k}
        out, osz, _, _ = O.forward(x, sizes, P, ocfg, training=True, use_aten_rnn=True)
        loss = F.ctc_loss(out.transpose(0, 1).double().log_softmax(-1), targets, osz, tsz, blank=0, reduction="sum",
                          zero_infinity=True)
        loss.backward()
        return out.detach(), float(loss.detach()), {k: v.grad.detach() for k, v in leaves.items()}

    def grad_groups(grads):
        groups = {}
        for k, g in grads.items():
            a, b = g.reshape(-1), ref_grads[k].reshape(-1)
            acc = groups.setdefault(_group_of(k), [0.0, 0.0, 0.0, 0.0])
            acc[0] += float((a.double() - b.double()).pow(2).sum())
            acc[1] += float(b.double().pow(2).sum())
            acc[2] = max(acc[2], float((a - b).abs().max()))
            acc[3] = max(acc[3], float(b.abs().max()))
        return ({g: (v[0] / v[1]) ** 0.5 if v[1] > 0 else 0.0 for g, v in sorted(groups.items())},
                {g: v[2] / v[3] if v[3] > 0 else 0.0 for g, v in sorted(groups.items())})

    try:
        ref_logits, ref_loss, ref_grads = reference_arm()
        # yardstick: the reference's own default CUDA path (cuDNN TF32 allowed) against the same fp32 arithmetic,
        # logits and gradients (the Hardtanh clips of the front-end are not smooth: a 1e-3 forward deviation flips a
        # few clip masks, which is what the conv-gradient figure of either arm shows)
        torch.backends.cudnn.allow_tf32 = True
        stock_logits, _, stock_grads = reference_arm()
        stock_rel, stock_rel_l2 = rel(stock_logits, ref_logits), rel_l2(stock_logits, ref_logits)
        stock_grad_l2, _ = grad_groups(stock_grads)
        del stock_logits, stock_grads
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    # ---- B200 arm, same weights
    model.load_state_dict(P0)
    flat.zero_grad()
    got_logits, _, _ = model(x, sizes)
    got_logits = got_logits.detach().clone()
    model.load_state_dict(P0)                       # undo the running-statistics update of that forward
    flat.zero_grad()
    loss = model.training_step((x, targets, pct.clone(), tsz), 0)
    loss.backward()
    torch.cuda.synchronize()
    got_loss = float(loss.detach())
    got_l2, got_max = grad_groups({k: p.grad.detach() for k, p in model.named_parameters()})
    res = {
        "reference": "reference ATen ops on the GPU, cudnn.allow_tf32=False, matmul.allow_tf32=False, CTC in float64; "
                     "same weights, same batch",
        "logits_rel": rel(got_logits, ref_logits), "logits_rel_l2": rel_l2(got_logits, ref_logits),
        "stock_default_tf32_logits_rel": stock_rel, "stock_default_tf32_logits_rel_l2": stock_rel_l2,
        "loss": got_loss, "loss_reference": ref_loss, "loss_rel": abs(got_loss - ref_loss) / max(1.0, abs(ref_loss)),
        "grad_rel_l2": got_l2, "grad_rel_max": got_max, "stock_default_tf32_grad_rel_l2": stock_grad_l2,
        "finite": bool(all(torch.isfinite(p.grad).all() for p in model.parameters())),
    }
    model.load_state_dict(P0)
    flat.zero_grad()
    del ref_grads, ref_logits, got_logits
    torch.cuda.empty_cache()
    return res


def run_b200(args):
    import torch
    import deepspeech_pytorch_b200 as ds
    from deepspeech_pytorch_b200 import dist as D
    from deepspeech_pytorch_b200.optim import FlatParams, FusedOptimizer

    # NCCL prints its version banner on stdout: keep fd 1 clean for the single JSON line
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = D.init_from_env()
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = ds.get_lib()
    ds.set_precision(args.precision)
    rnn, bidir, H, layers, ctx, B, T, L = WORKLOADS[args.workload]
    if args.batch:
        B = args.batch
    rt = getattr(ds.RNNType, rnn)
    mcfg = (ds.BiDirectionalConfig(rnn_type=rt, hidden_size=H, hidden_layers=layers) if bidir else
            ds.UniDirectionalConfig(rnn_type=rt, hidden_size=H, hidden_layers=layers, lookahead_context=ctx))
    torch.manual_seed(123456)
    model = ds.DeepSpeech(ds.LABELS, mcfg, 32, ds.AdamConfig(), ds.SpectConfig()).to(dev).train()
    flat = FlatParams(model, direct_grads=True)   # backward kernels write straight into the flat gradient buffer
    if not args.no_defer:
        # the step runs on a high-priority stream; the weight-gradient GEMMs of each recurrent layer are queued on a
        # normal-priority side stream and fill the SMs / pipes the next layer's latency-bound sweep leaves idle
        main_stream = torch.cuda.Stream(device=dev, priority=-1)
        main_stream.wait_stream(torch.cuda.current_stream(dev))
        torch.cuda.set_stream(main_stream)
        ds.ops.enable_deferred_weight_grads(dev)
    opt = FusedOptimizer(flat, model.optim_cfg, max_norm=400.0)
    n_params = sum(p.numel() for p in model.parameters())

    # the weights every arm of this run starts from (B200 timing, full-size parity check, stock CUDA baseline)
    P0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
    x, targets, pct, tsz = synth_batch(B, T, L, seed=1234 + rank)
    x_pinned = x.pin_memory()
    x_dev = x.to(dev)
    targets_pinned = targets.pin_memory()

    # one all-reduce of the flat gradient buffer, its (99.7 %) recurrent + fc part started as soon as those
    # gradients are final so that it overlaps the conv backward
    exchange = D.OverlappedGradAllReduce(flat, model)

    def train_step(inputs):
        loss = model.training_step((inputs, targets_pinned, pct.clone(), tsz), 0)
        loss.backward()
        exchange.finish()
        opt.step(grad_scale=1.0 / world)
        flat.zero_grad()
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    def timed(n, e2e):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lib.ds2_launch_count(1)
        e0.record()
        last = None
        for _ in range(n):
            if e2e:
                last = float(train_step(x_pinned.to(dev, non_blocking=True)).item())   # H2D + D2H every step
            else:
                last = train_step(x_dev)
        e1.record()
        barrier()
        launches = int(lib.ds2_launch_count(0))
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)   # max over ranks
            ms = float(t)
        return ms / n, launches, (last if e2e else float(last.detach()))

    parity = None
    if world == 1 and not args.no_parity:
        log("full-size parity check against the fp32 reference arithmetic (same weights, same batch)")
        try:
            parity = parity_fullsize(args.workload, model, flat, P0, (x_dev, targets, pct, tsz))
            log("parity_fullsize: " + json.dumps(parity))
        except Exception as e:  # pragma: no cover
            parity = {"error": repr(e)[:300]}
            log(f"parity_fullsize failed: {e!r}")
        model.load_state_dict(P0)
        flat.zero_grad()
    lib.ds2_fallback_count(1)
    log(f"model built ({n_params} params), warming up")
    for _ in range(max(3, args.warmup)):
        train_step(x_dev)
    torch.cuda.synchronize()
    log("warm-up done")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, launches, loss_val = timed(args.steps, e2e=False)
    log(f"device-resident: {ms_dev:.2f} ms/step")
    if args.dump_outputs and rank == 0:      # device copies now, written out once the timed windows are over
        dump = (loss_val, {k: v.detach().clone() for k, v in model.state_dict().items()},
                {k: p.grad.detach().clone() for k, p in model.named_parameters()})
    ms_e2e, _, _ = timed(args.steps, e2e=True)
    log(f"e2e: {ms_e2e:.2f} ms/step")
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *dump)
        del dump

    # ---- per-block device times (cudaEvent ranges inside the library) for the roofline of the dominant kernel
    prof = {}
    if rank == 0:
        lib.ds2_prof_enable(1)
    for _ in range(2):          # every rank runs the steps (they contain the all-reduce); rank 0 records ranges
        train_step(x_dev)
    if rank == 0:
        buf = (__import__("ctypes").c_char * 8192)()
        lib.ds2_prof_report(buf, 8192)
        lib.ds2_prof_enable(0)
        for item in buf.value.decode().split(";"):
            if item:
                tag, ms, cnt = item.split(":")
                prof[tag] = {"ms_per_step": float(ms) / 2, "ranges_per_step": int(cnt) // 2}
    barrier()

    if rank != 0:
        return
    hbm_peak, tf_peak, which = load_peaks()
    Tp = (T - 1) // 2 + 1
    D_ = 2 if bidir else 1
    G = {"lstm": 4, "gru": 3, "rnn": 1}[rnn]
    # SURVEY.md §8d algorithmic bytes of the recurrent sweep, per layer and direction:
    #   fwd: read G_x (T'*B*G*H) + W_hh once (G*H*H) + write h (+ c for LSTM)
    #   bwd: read dY + h,c (3*T'BH) + gates (T'B*GH) + W_hh once + write dG (T'B*GH)
    tbh = Tp * B * H * 4
    fwd_bytes = (G * tbh + G * H * H * 4 + tbh * (2 if rnn == "lstm" else 1)) * D_ * layers
    bwd_bytes = ((2 * G + 3) * tbh + G * H * H * 4) * D_ * layers
    roofs = {}
    traffic_db = {}
    try:   # DRAM bytes per launch from the committed ncu --set full captures (librispeech workload only)
        if args.workload == "librispeech" and B == 32:
            traffic_db = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
    except Exception:
        traffic_db = {}
    for tag, nbytes in (("rnn_fwd_sweep", fwd_bytes), ("rnn_bwd_sweep", bwd_bytes)):
        if tag in prof and prof[tag]["ms_per_step"] > 0:
            nl = max(1, prof[tag]["ranges_per_step"])          # launches per step (one per layer)
            ms_launch = prof[tag]["ms_per_step"] / nl
            ach = (nbytes / nl) / (ms_launch * 1e-3) / 1e9
            roofs[tag] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                          "traffic": traffic_db.get(tag, {}).get("dram_bytes_per_launch"), "peak_source": which,
                          "algorithmic_bytes_per_launch": nbytes / nl, "launches_per_step": nl,
                          "ms_per_launch": ms_launch, "ms_per_step": prof[tag]["ms_per_step"],
                          "note": "latency-bound: T' serial steps of (grid barrier + MMA issue chain + epilogue); "
                                  "see DESIGN.md 5.1"}
    if "ctc" in prof and prof["ctc"]["ms_per_step"] > 0:
        # SURVEY.md §8d: read logits (T'*B*C*4) + write grad (same) + targets / lengths; the alpha/beta tables the
        # kernel keeps (or spills) are overhead, not credit
        Cn = 29
        ctc_bytes = 2 * Tp * B * Cn * 4 + B * L * 8 + 2 * B * 4
        ach = ctc_bytes / (prof["ctc"]["ms_per_step"] * 1e-3) / 1e9
        roofs["ctc"] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                        "traffic": traffic_db.get("ctc", {}).get("dram_bytes_per_launch"), "peak_source": which,
                        "algorithmic_bytes_per_launch": ctc_bytes, "launches_per_step": 1,
                        "ms_per_launch": prof["ctc"]["ms_per_step"], "ms_per_step": prof["ctc"]["ms_per_step"],
                        "note": "latency-bound: T' dependent lattice steps per utterance, B*2 CTAs; the HBM fraction "
                                "is not the binding limit (DESIGN.md 5.4)"}
    dominant = max(prof, key=lambda k: prof[k]["ms_per_step"]) if prof else None
    roofline = roofs.get(dominant) or (roofs.get("rnn_bwd_sweep") if roofs else None)
    if roofline is not None:
        roofline = dict(roofline, kernel=dominant if dominant in roofs else "rnn_bwd_sweep")

    value = B * world / (ms_dev * 1e-3)
    e2e = B * world / (ms_e2e * 1e-3)
    h2d = x.numel() * 4 + targets.numel() * 8 + B * 4 * 2
    line = {
        "metric": "utterances/sec (train step, 161x1000 spectrogram)", "value": value, "unit": "utt/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_dev,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"tf32": "tf32+fp16-recurrent", "fp16": "fp16-operands(rnn)+tf32(conv/fc)", "fp32": "f32"}[args.precision],
        "data": "synthetic",
        "dtype_note": ("dense GEMMs / conv2: TF32 operands (TMA rounds to nearest); recurrent products: fp16 operands "
                       "(10-bit mantissa like TF32; backward gate gradients scaled per step by a power of two); fp32 "
                       "accumulation in TMEM, fp32 state / activations / gradients / optimizer"
                       if args.precision == "tf32" else
                       "the reference's `precision: 16`: recurrent-stack GEMMs (input projection, dW_ih, dW_hh, dX) on "
                       "fp16 operand copies (gradients scaled by a power of two per tensor), recurrent products fp16, "
                       "conv2 / fc head TF32, fp32 accumulation, fp32 state / activations / gradients / optimizer"
                       if args.precision == "fp16" else "fp32 FFMA everywhere"),
        "config": {"workload": args.workload, "rnn": f"{layers}x{'bi' if bidir else 'uni'}-{rnn}-{H}",
                   "batch_per_gpu": B, "global_batch": B * world, "frames": T, "target_len": L, "params": n_params,
                   "parallelism": f"dp{world}", "optimizer": "fused clip(400)+AdamW inside the step",
                   "l2": "per-step working set (activations 3+ GB) exceeds the 126 MB L2; no explicit flush"},
        "e2e": {"value": e2e, "unit": "utt/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4},
        "gpu_launches": launches, "ffma_fallback_sweeps": int(lib.ds2_fallback_count(0)), "clocks": clocks,
        "loss": loss_val, "parity_fullsize": parity,
        "roofline": roofline, "roofline_all": roofs, "blocks_ms_per_step": {k: v["ms_per_step"] for k, v in prof.items()},
    }
    log("profile ranges: " + json.dumps(line["blocks_ms_per_step"]))
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args.workload)
        log("cpu baseline done")
    if world == 1 and not args.no_stock_cuda:
        log("stock torch CUDA baseline (north_star denominator), same weights")
        try:
            torch.cuda.empty_cache()
            sc = stock_cuda_baseline(args.workload, P0, (x_dev, targets, pct, tsz))
            line["stock_cuda_baseline"] = sc
            line["vs_stock_cuda"] = {k: (value / v["value"]) for k, v in sc.items()
                                     if isinstance(v, dict) and v.get("value")}
            line["vs_stock_cuda_e2e"] = {k: (e2e / v["value"]) for k, v in sc.items()
                                         if isinstance(v, dict) and v.get("value")}
        except Exception as e:  # pragma: no cover
            line["stock_cuda_baseline"] = {"error": repr(e)[:300]}
        log("stock baseline done: " + json.dumps(line.get("vs_stock_cuda")))
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="librispeech", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override utterances per GPU")
    ap.add_argument("--precision", default="fp16", choices=["tf32", "fp32", "fp16"],
                    help="fp16 (default) = the reference's `precision: 16`, what configs/librispeech.yaml ships: fp16 "
                         "operand copies (10-bit mantissa like TF32) for the recurrent stack's GEMMs, fp32 accumulation; "
                         "tf32 = TF32 operands for those GEMMs; fp32 = FFMA everywhere")
    ap.add_argument("--cpu-batch", type=int, default=2, help="--impl reference: utterances per CPU step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stock-cuda", action="store_true", help="(default on at N=1; kept for compatibility)")
    ap.add_argument("--no-stock-cuda", action="store_true", help="skip the stock torch CUDA baseline legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-size parity check against fp32 ATen")
    ap.add_argument("--no-defer", action="store_true", help="weight-gradient GEMMs on the compute stream (no side stream)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss, parameters, running statistics and gradients of the "
                         "last device-resident timed step to DIR/<name>.npy (same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path's timed steps; --impl reference has none")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
        if int(os.environ.get("WORLD_SIZE", "1")) > 1 and int(os.environ.get("RANK", "0")) != 0:
            try:
                import torch
                if torch.distributed.is_initialized():
                    torch.distributed.destroy_process_group()
            except Exception:
                pass


if __name__ == "__main__":
    main()
