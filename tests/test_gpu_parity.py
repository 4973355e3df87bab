"""-m gpu: the CUDA path (through the C-ABI) against (1) the committed outputs of the reference
itself (tests/golden) and (2) the oracle on seeded inputs.  fp32 mode tolerance: 1e-3 rel (the
north_star bound; measured errors are ~1e-5); integers bit-exact."""
import numpy as np
import pytest
import torch

from conftest import Golden, golden_names
from gpu_helpers import make_model, model_from_golden, oracle_cfg, rel, rel_l2
from oracle import ds2_oracle as O

import deepspeech_pytorch_b200 as ds

pytestmark = pytest.mark.gpu
TOL = 1e-3        # north_star: logits within 1e-3 rel fp32
TOL_GRAD = 2e-3


@pytest.fixture(autouse=True)
def _fp32():
    ds.set_precision("fp32")
    yield


@pytest.mark.parametrize("name", golden_names())
def test_golden_forward_and_buffers(name):
    g = Golden(name)
    model = model_from_golden(g).train()
    out, out_lens, hs = model(g.x.cuda(), g.input_sizes)
    assert out_lens.dtype == torch.int32 and out_lens.device.type == "cpu"
    assert out_lens.tolist() == g.output_sizes.tolist()              # integers: bit-exact
    assert tuple(out.shape) == tuple(g.logits.shape)
    assert rel(out, g.logits) < TOL
    sd = model.state_dict()
    for k, v in g.buffers_after.items():
        if "num_batches" in k:
            assert int(sd[k]) == int(v), k
        else:
            assert rel(sd[k], v) < TOL, k


@pytest.mark.parametrize("name", golden_names())
def test_golden_train_step_loss_and_every_gradient(name):
    g = Golden(name)
    model = model_from_golden(g).train()
    pct = g.input_percentages.clone()
    loss = model.training_step((g.x.cuda(), g.targets, pct, g.target_sizes), 0)
    # model.py:243 mutates the caller's tensor in place: afterwards it holds percentage * T (fp32), and its
    # truncation is the reference's input_sizes (bit-exact, including the frames the fp32 product loses)
    assert torch.equal(pct, g.input_percentages.clone().mul_(int(g.x.size(3))))
    assert torch.equal(pct.int(), g.input_sizes)
    loss.backward()
    assert abs(float(loss) - g.loss) <= 1e-4 * max(1.0, abs(g.loss))
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert set(grads) == set(g.grads)
    for k, ref in g.grads.items():
        assert grads[k] is not None, k
        assert rel(grads[k], ref) < TOL_GRAD, k


@pytest.mark.parametrize("name", golden_names())
def test_golden_eval_forward_states_and_greedy_decode(name):
    g = Golden(name)
    P = dict(g.params)
    P.update(g.buffers_after)
    model = model_from_golden(g)
    model.load_state_dict(P)
    model.eval()
    with torch.no_grad():
        out, out_lens, hs = model(g.x.cuda(), g.input_sizes)
    assert rel(out, g.eval_out) < TOL
    for i, h in enumerate(hs):
        hn = h[0] if isinstance(h, tuple) else h
        assert rel(hn, g.z[f"eval_hn/{i}"]) < TOL
        if isinstance(h, tuple):
            assert rel(h[1], g.z[f"eval_cn/{i}"]) < TOL
    # integer outputs, bit-exact: decode the reference's own probabilities on the GPU
    labels, offsets, counts = model.evaluation_decoder.decode_indices(g.eval_out.cuda(), out_lens)
    ref = O.greedy_path(g.eval_out, g.output_sizes)
    for b, (lab, offs) in enumerate(ref):
        n = int(counts[b])
        assert labels[b, :n].tolist() == lab
        assert offsets[b, :n].tolist() == offs == g.z[f"eval_offsets/{b}"].tolist()


def test_unsorted_or_empty_lengths_raise_like_pack_padded_sequence():
    model = make_model("gru", True, 8, 1).train()
    x = torch.randn(2, 1, 161, 40, device="cuda")
    with pytest.raises(RuntimeError, match="sorted"):
        model(x, torch.tensor([20, 40]))
    with pytest.raises(RuntimeError, match="greater than 0"):
        model(x, torch.tensor([40, 0]))


CASES = [  # rnn_type, bidirectional, H, layers, B, T   (sizes the oracle finishes in seconds)
    ("lstm", True, 40, 3, 5, 157),
    ("gru", True, 36, 2, 3, 101),
    ("gru", False, 32, 2, 4, 90),
    ("lstm", False, 24, 2, 2, 64),
    ("rnn", True, 16, 2, 3, 75),
    ("lstm", True, 64, 2, 33, 80),      # batch > 32 exercises the batch-tile loop
]


@pytest.mark.parametrize("rnn_type,bidir,H,layers,B,T", CASES)
def test_train_step_vs_oracle(rnn_type, bidir, H, layers, B, T):
    ocfg = oracle_cfg(rnn_type, bidir, H, layers, ctx=7)
    P = O.init_params(ocfg, seed=11)
    x, targets, pct, tsz = O.synth_batch(B, T, seed=3, lmin=4, lmax=15)
    ref = O.train_step(x, targets, pct.clone(), tsz, P, ocfg)
    model = make_model(rnn_type, bidir, H, layers, ctx=7, params=P).train()
    loss = model.training_step((x.cuda(), targets, pct.clone(), tsz), 0)
    loss.backward()
    assert abs(float(loss) - ref["loss"]) <= 1e-4 * max(1.0, abs(ref["loss"]))
    for k, r in ref["grads"].items():
        got = dict(model.named_parameters())[k].grad
        assert rel(got, r) < TOL_GRAD, k
    sd = model.state_dict()
    for k, v in ref["new_buffers"].items():
        assert rel(sd[k], v) < TOL, k


def test_hidden_state_carry_matches_oracle_chunked_inference():
    # reference inference.py:86-97: chunked transcribe carries `hs`; exact for unidirectional models
    ocfg = oracle_cfg("gru", False, 24, 2, ctx=5)
    P = O.init_params(ocfg, seed=2)
    model = make_model("gru", False, 24, 2, ctx=5, params=P).eval()
    x = torch.randn(1, 1, 161, 80)
    hs_o = hs_m = None
    for c in range(2):
        chunk = x[:, :, :, c * 40:(c + 1) * 40].contiguous()
        lens = torch.tensor([40])
        out_o, _, hs_o, _ = O.forward(chunk, lens, P, ocfg, training=False, hs=hs_o)
        with torch.no_grad():
            out_m, _, hs_m = model(chunk.cuda(), lens, hs_m)
        assert rel(out_m, out_o) < TOL
        for a, b in zip(hs_m, hs_o):
            assert rel(a, b) < TOL


@pytest.mark.parametrize("T,B,L", [(50, 4, 12), (500, 8, 200), (33, 3, 1)])
def test_ctc_kernel_vs_oracle(T, B, L):
    g = torch.Generator().manual_seed(T)
    logits = torch.randn(T, B, 29, generator=g) * 2
    in_len = torch.tensor(sorted([max(1, T - 7 * i) for i in range(B)], reverse=True), dtype=torch.int32)
    tgt_len = torch.tensor([max(1, L - i) for i in range(B)], dtype=torch.int32)
    targets = torch.randint(1, 29, (int(tgt_len.sum()),), generator=g)
    nll, grad = O.ctc_loss_and_grad(logits.numpy(), targets.numpy(), in_len.numpy(), tgt_len.numpy())
    lg = logits.cuda().requires_grad_(True)
    loss = ds.ops.CtcLoss.apply(lg, targets.cuda(), in_len.cuda(), tgt_len.cuda(), int(tgt_len.max()), 0)
    loss.backward()
    assert abs(float(loss) - nll.sum()) <= 1e-5 * max(1.0, abs(nll.sum()))
    assert float((lg.grad.cpu().double() - torch.from_numpy(grad)).abs().max()) < 1e-4
    for b in range(B):                                   # exact zeros beyond the input length
        assert float(lg.grad[int(in_len[b]):, b].abs().max() if int(in_len[b]) < T else 0.0) == 0.0


def test_ctc_infeasible_and_repeats_zero_infinity():
    T, B, C = 12, 3, 29
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(T, B, C, generator=g)
    in_len = torch.tensor([12, 9, 5], dtype=torch.int32)
    tgt_len = torch.tensor([6, 5, 5], dtype=torch.int32)
    targets = torch.tensor([4, 4, 4, 4, 4, 4, 1, 2, 3, 4, 5, 7, 7, 8, 9, 10])   # utt0: 6 repeats need 11 frames
    nll, grad = O.ctc_loss_and_grad(logits.numpy(), targets.numpy(), in_len.numpy(), tgt_len.numpy())
    assert nll[2] == 0.0                                                        # 5 labels + repeat in 5 frames
    lg = logits.cuda().requires_grad_(True)
    loss = ds.ops.CtcLoss.apply(lg, targets.cuda(), in_len.cuda(), tgt_len.cuda(), 6, 0)
    loss.backward()
    assert abs(float(loss) - nll.sum()) <= 1e-5 * max(1.0, abs(nll.sum()))
    assert float(lg.grad[:, 2].abs().max()) == 0.0
    assert float((lg.grad.cpu().double() - torch.from_numpy(grad)).abs().max()) < 1e-4


@pytest.mark.parametrize("tA,tB,M,N,K", [(0, 1, 300, 96, 200), (1, 0, 29, 130, 4100), (0, 0, 257, 129, 65),
                                           (1, 1, 64, 64, 64)])
def test_gemm_fp32_vs_torch(tA, tB, M, N, K):
    g = torch.Generator().manual_seed(M + N)
    a = torch.randn((K, M) if tA else (M, K), generator=g).cuda()
    b = torch.randn((N, K) if tB else (K, N), generator=g).cuda()
    c = ds.ops.gemm(a, b, bool(tA), bool(tB))
    ref = (a.t() if tA else a).double() @ (b.t() if tB else b).double()
    assert rel(c, ref) < 1e-5


def test_adamw_and_sgd_step_match_torch_optim():
    import ctypes as C
    lib = ds.get_lib()
    n = 100003
    g0 = torch.Generator().manual_seed(1)
    p0 = torch.randn(n, generator=g0)
    grads = [torch.randn(n, generator=g0) * s for s in (1.0, 30.0, 0.1)]
    ws = torch.zeros(64, device="cuda")
    norm = torch.zeros(1, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    # AdamW + clip 400 (configs/librispeech.yaml:12, model.py:283-289)
    ref = torch.nn.Parameter(p0.clone().cuda())
    opt = torch.optim.AdamW([ref], lr=1.5e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-5)
    p = p0.clone().cuda(); m = torch.zeros_like(p); v = torch.zeros_like(p)
    for step, gr in enumerate(grads, 1):
        ref.grad = gr.clone().cuda()
        tn = torch.nn.utils.clip_grad_norm_([ref], 400.0)
        opt.step()
        gg = gr.cuda()
        assert lib.ds2_adamw_step(n, p.data_ptr(), gg.data_ptr(), m.data_ptr(), v.data_ptr(), 1.5e-4, 0.9, 0.999, 1e-8,
                                  1e-5, step, 1.0, 400.0, norm.data_ptr(), ws.data_ptr(), st) == 0
        assert abs(float(norm) - float(tn)) <= 1e-4 * float(tn)
        assert rel(p, ref.data) < 1e-5
    # SGD Nesterov (model.py:275-281)
    ref = torch.nn.Parameter(p0.clone().cuda())
    opt = torch.optim.SGD([ref], lr=1e-3, momentum=0.9, nesterov=True, weight_decay=1e-5)
    p = p0.clone().cuda(); buf = torch.zeros_like(p)
    for step, gr in enumerate(grads, 1):
        ref.grad = gr.clone().cuda()
        torch.nn.utils.clip_grad_norm_([ref], 400.0)
        opt.step()
        gg = gr.cuda()
        assert lib.ds2_sgd_nesterov_step(n, p.data_ptr(), gg.data_ptr(), buf.data_ptr(), 1e-3, 0.9, 1e-5,
                                         int(step == 1), 1.0, 400.0, norm.data_ptr(), ws.data_ptr(), st) == 0
        assert rel(p, ref.data) < 1e-5


# ---- tensor-core (TF32) mode: tcgen05 GEMMs + persistent recurrent sweeps --------------------------
# Same arithmetic class as the reference's stock CUDA path (cuDNN allow_tf32): 10-bit operand
# mantissas, fp32 accumulation.  Tolerances against the fp32 oracle: logits 3e-3 rel (measured ~5e-4);
# gradients 3e-2 in relative L2 norm and 1e-1 in max-norm (measured ~3e-3 typical; the worst max-norm case,
# 5.8e-2, is the n-gate bias gradient of a 2-layer uni-GRU — a long signed sum that amplifies operand rounding).
TC_CASES = [("lstm", True, 64, 2, 6, 90), ("gru", True, 96, 2, 33, 70), ("gru", False, 64, 2, 5, 81),
            ("rnn", True, 32, 2, 4, 60), ("lstm", True, 128, 3, 16, 120)]


@pytest.mark.parametrize("rnn_type,bidir,H,layers,B,T", TC_CASES)
def test_tf32_train_step_vs_oracle(rnn_type, bidir, H, layers, B, T):
    ds.set_precision("tf32")
    ocfg = oracle_cfg(rnn_type, bidir, H, layers, ctx=7)
    P = O.init_params(ocfg, seed=5)
    x, targets, pct, tsz = O.synth_batch(B, T, seed=8, lmin=4, lmax=12)
    ref = O.train_step(x, targets, pct.clone(), tsz, P, ocfg)
    model = make_model(rnn_type, bidir, H, layers, ctx=7, params=P).train()
    out, _, _ = model(x.cuda(), O.input_sizes_from_percentages(pct, T))
    assert rel(out, ref["logits"]) < 3e-3
    model = make_model(rnn_type, bidir, H, layers, ctx=7, params=P).train()
    loss = model.training_step((x.cuda(), targets, pct.clone(), tsz), 0)
    loss.backward()
    assert abs(float(loss) - ref["loss"]) <= 2e-3 * max(1.0, abs(ref["loss"]))
    for k, r in ref["grads"].items():
        got = dict(model.named_parameters())[k].grad
        assert rel_l2(got, r) < 3e-2, k
        assert rel(got, r) < 1e-1, k


def test_tf32_full_size_properties_librispeech_layer():
    """BASELINE size (T'=500, B=32, H=1024): size-independent properties of one bi-LSTM layer on the tensor-core
    path: masked frames exactly zero, h_n equals the output at the last valid frame, agreement with the FFMA path."""
    from deepspeech_pytorch_b200 import _lib
    T, B, In, H = 500, 32, 1024, 1024
    g = torch.Generator().manual_seed(4)
    x = torch.randn(T, B, In, generator=g).cuda()
    lens = torch.tensor(sorted([500 - 9 * i for i in range(B)], reverse=True), dtype=torch.int32)
    for b in range(B):
        x[int(lens[b]):, b] = 0
    k = 1.0 / H ** 0.5
    ws = [((torch.rand(s, generator=g) * 2 - 1) * k).cuda() for s in
          [(4 * H, In), (4 * H, H), (4 * H,), (4 * H,)] * 2]
    outs = {}
    for prec in ("tf32", "fp32"):
        ds.set_precision(prec)
        y, hn, cn = ds.ops.RnnLayer.apply(x, lens.cuda(), _lib.RNN_LSTM, True, False, 0.1, 1e-5, None, None, None,
                                          None, None, None, *ws)
        outs[prec] = (y, hn)
    y, hn = outs["tf32"]
    for b in range(B):
        L = int(lens[b])
        if L < T:
            assert float(y[L:, b].abs().max()) == 0.0
    assert rel(y, outs["fp32"][0]) < 5e-3 and rel(hn, outs["fp32"][1]) < 5e-3


def test_tf32_stress_shape_h1536_one_launch_per_direction():
    """BASELINE configs[4] layer shape (H=1536, B=8): 2 x 96 CTAs do not fit on 148 SMs, so the persistent sweeps are
    launched one direction at a time; result must agree with the FFMA step kernels, masked frames stay exactly 0."""
    from deepspeech_pytorch_b200 import _lib
    T, B, In, H = 40, 8, 1536, 1536
    g = torch.Generator().manual_seed(6)
    x = torch.randn(T, B, In, generator=g).cuda()
    lens = torch.tensor([40, 40, 37, 33, 30, 22, 15, 9], dtype=torch.int32)
    for b in range(B):
        x[int(lens[b]):, b] = 0
    k = 1.0 / H ** 0.5
    ws = [((torch.rand(s, generator=g) * 2 - 1) * k).cuda().requires_grad_(True) for s in
          [(4 * H, In), (4 * H, H), (4 * H,), (4 * H,)] * 2]
    dy = torch.randn(T, B, H, generator=g).cuda()
    res = {}
    for prec in ("tf32", "fp32"):
        ds.set_precision(prec)
        for w in ws:
            w.grad = None
        xx = x.clone().requires_grad_(True)
        y, hn, cn = ds.ops.RnnLayer.apply(xx, lens.cuda(), _lib.RNN_LSTM, True, True, 0.1, 1e-5, None, None, None,
                                          None, None, None, *ws)
        y.backward(dy)
        res[prec] = (y.detach(), hn.detach(), xx.grad.clone(), [w.grad.clone() for w in ws])
    a, b_ = res["tf32"], res["fp32"]
    for bb in range(B):
        L = int(lens[bb])
        if L < T:
            assert float(a[0][L:, bb].abs().max()) == 0.0
    assert rel(a[0], b_[0]) < 5e-3 and rel(a[1], b_[1]) < 5e-3 and rel_l2(a[2], b_[2]) < 1e-2
    for ga, gb in zip(a[3], b_[3]):
        assert rel_l2(ga, gb) < 1e-2


# ---- kernel variants behind the tensor-core mode: every selectable path must give the same answer ----------
def _one_layer(rnn, T, B, In, H, seed):
    from deepspeech_pytorch_b200 import _lib
    G = {"lstm": 4, "gru": 3}[rnn]
    code = {"lstm": _lib.RNN_LSTM, "gru": _lib.RNN_GRU}[rnn]
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(T, B, In, generator=g).cuda()
    lens = torch.tensor(sorted([max(1, T - 2 * i) for i in range(B)], reverse=True), dtype=torch.int32)
    for b in range(B):
        x[int(lens[b]):, b] = 0
    k = 1.0 / H ** 0.5
    ws = [((torch.rand(s, generator=g) * 2 - 1) * k).cuda().requires_grad_(True) for s in
          [(G * H, In), (G * H, H), (G * H,), (G * H,)] * 2]
    dy = torch.randn(T, B, H, generator=g).cuda()
    for b in range(B):
        dy[int(lens[b]):, b] = 0

    def run():
        for w in ws:
            w.grad = None
        xx = x.clone().requires_grad_(True)
        y, hn, cn = ds.ops.RnnLayer.apply(xx, lens.cuda(), code, True, True, 0.1, 1e-5, None, None, None, None, None,
                                          None, *ws)
        y.backward(dy)
        torch.cuda.synchronize()
        return [y.detach(), hn.detach(), xx.grad.clone()] + [w.grad.clone() for w in ws]
    return run


@pytest.mark.parametrize("rnn,B", [("lstm", 32), ("lstm", 20), ("gru", 20), ("lstm", 40), ("gru", 48)])
def test_tf32_sweep_variants_agree_with_the_fp32_path(rnn, B, monkeypatch):
    """forward: 2-CTA split-K clusters vs 16-unit CTAs; backward: 8- vs 4-CTA clusters (LSTM, B = 32); grid barrier + TMA
    (default) vs the flag-in-data exchange (DS2_FWD_LL / DS2_BWD_LL = 1); stores deferred past the barrier or not.  H = 256 takes every variant; B = 20 exercises the N padding (24 / 32 columns),
    B > 32 the second pass of the epilogues over the batch columns."""
    run = _one_layer(rnn, T=33, B=B, In=192, H=256, seed=11)
    ds.set_precision("fp32")
    ref = run()
    ds.set_precision("tf32")
    variants = [{}, {"DS2_FWD_SPLITK": "0"}, {"DS2_SPLITK_CL": "4"}, {"DS2_SWEEP_DEFER": "0"},
                {"DS2_FWD_LL": "1"}, {"DS2_BWD_LL": "1"}, {"DS2_FWD_LL": "1", "DS2_BWD_LL": "1", "DS2_SPLITK_CL": "4"},
                {"DS2_FWD_SPLITK": "0", "DS2_SPLITK_CL": "4", "DS2_SWEEP_DEFER": "0"}]
    for env in variants:
        for k_, v in env.items():
            monkeypatch.setenv(k_, v)
        got = run()
        for k_ in env:
            monkeypatch.delenv(k_)
        assert rel(got[0], ref[0]) < 5e-3 and rel(got[1], ref[1]) < 5e-3, env
        for a, b in zip(got[2:], ref[2:]):
            assert rel_l2(a, b) < 1e-2, env


@pytest.mark.parametrize("cfg", ["1", "2", "3"])
def test_gemm_tile_configurations_vs_fp64(cfg, monkeypatch):
    """128x256x4 stages, 256x256x3 stages (two TMEM accumulators), 128x256x2 stages with two CTAs per SM; K-major and
    MN-major operands (3-D boxes when the extent is a multiple of 32, 2-D boxes otherwise); TF32 error level."""
    monkeypatch.setenv("DS2_GEMM_CFG", cfg)
    ds.set_precision("tf32")
    g = torch.Generator(device="cuda").manual_seed(3)
    for tA, tB, M, N, K in [(0, 1, 600, 520, 300), (1, 0, 512, 320, 2000), (0, 0, 640, 1312, 512),
                            (1, 1, 424, 96, 100), (1, 0, 500, 260, 1000)]:
        a = torch.randn((K, M) if tA else (M, K), generator=g, device="cuda")
        b = torch.randn((N, K) if tB else (K, N), generator=g, device="cuda")
        ref = (a.t() if tA else a).double() @ (b.t() if tB else b).double()
        c = ds.ops.gemm(a, b, bool(tA), bool(tB))
        assert rel_l2(c, ref) < 1e-3, (cfg, tA, tB, M, N, K)


def test_gemm_split_k_accumulates_into_c():
    """weight-gradient shape class (64 tiles of 256x256): 2-way split-K with vector atomics, beta = 0 and beta = 1"""
    ds.set_precision("tf32")
    g = torch.Generator(device="cuda").manual_seed(5)
    M, N, K = 4096, 1024, 2304
    a = torch.randn(K, M, generator=g, device="cuda")
    b = torch.randn(K, N, generator=g, device="cuda")
    ref = a.t().double() @ b.double()
    c = ds.ops.gemm(a, b, True, False)
    assert rel_l2(c, ref) < 1e-3
    c0 = torch.randn(M, N, generator=g, device="cuda")
    c1 = ds.ops.gemm(a, b, True, False, out=c0.clone(), alpha=0.5, beta=1.0)
    assert rel_l2(c1, 0.5 * ref + c0.double()) < 1e-3


@pytest.mark.parametrize("rnn_type,bidir", [("lstm", True), ("gru", False)])
def test_direct_gradient_sinks_equal_autograd_accumulation(rnn_type, bidir):
    """FlatParams(direct_grads=True): every backward kernel writes its parameter gradients straight into the flat
    buffer (no AccumulateGrad adds).  Must be bit-identical to the autograd route, also on a second step (gradients
    are overwritten, not accumulated), and a model without sinks must be unaffected by a registry entry whose owner
    is gone."""
    from deepspeech_pytorch_b200.optim import FlatParams
    ocfg = oracle_cfg(rnn_type, bidir, 32, 2, ctx=5)
    P = O.init_params(ocfg, seed=4)
    batches = [O.synth_batch(3, 70, seed=s, lmin=3, lmax=8) for s in (1, 2)]
    grads = {}
    for direct in (False, True):
        model = make_model(rnn_type, bidir, 32, 2, ctx=5, params=P).train()
        flat = FlatParams(model, direct_grads=direct)
        snaps = []
        for x, targets, pct, tsz in batches:
            flat.zero_grad()
            model.training_step((x.cuda(), targets, pct.clone(), tsz), 0).backward()
            torch.cuda.synchronize()
            snaps.append(flat.grad.clone())
        grads[direct] = snaps
        del model, flat
    # (not bit-equal: the fp32-mode column sums / BatchNorm reductions use float atomics, whose order varies run to run)
    for a, b in zip(grads[False], grads[True]):
        assert rel(a, b) < 1e-5 and rel_l2(a, b) < 1e-6
    assert rel(grads[True][0], grads[True][1]) > 1e-2          # the second step really overwrote the first
    model = make_model(rnn_type, bidir, 32, 2, ctx=5, params=P).train()       # no FlatParams: plain autograd grads
    x, targets, pct, tsz = batches[0]
    model.training_step((x.cuda(), targets, pct.clone(), tsz), 0).backward()
    assert all(p.grad is not None for p in model.parameters())


def test_deferred_weight_gradient_gemms_give_the_same_gradients():
    """precision-16 mode with gradient sinks: dW_ih / dW_hh of every recurrent layer queued on the side stream (two
    alternating operand workspaces, join before the gradients are read) vs everything on the compute stream.  The
    GEMMs are the same kernels on the same operands: the flat gradient buffer must agree to the level of the float
    atomics' run-to-run noise, on the first backward and on a second one from the same parameters (workspace slots
    reused, gradients overwritten)."""
    from deepspeech_pytorch_b200.optim import FlatParams, FusedOptimizer
    ds.set_precision("fp16")
    ocfg = oracle_cfg("lstm", True, 128, 3)
    P = O.init_params(ocfg, seed=13)
    batches = [O.synth_batch(8, 200, seed=s_, lmin=5, lmax=20) for s_ in (3, 4)]
    out = {}
    try:
        for defer in (False, True):
            model = make_model("lstm", True, 128, 3, params=P).train()
            flat = FlatParams(model, direct_grads=True)
            opt = FusedOptimizer(flat, model.optim_cfg)
            main = torch.cuda.Stream(priority=-1)
            main.wait_stream(torch.cuda.current_stream())
            gs = []
            with torch.cuda.stream(main):
                ds.ops.enable_deferred_weight_grads(enable=defer)
                for x, targets, pct, tsz in batches:         # same parameters for both backwards
                    model.load_state_dict(P)                 # (undo the running-statistics update)
                    model.training_step((x.cuda(), targets, pct.clone(), tsz), 0).backward()
                    ds.ops.join_deferred()
                    gs.append(flat.grad.clone())
                before = flat.data.clone()
                opt.step()                                   # joins by itself
            torch.cuda.synchronize()
            assert not torch.equal(before, flat.data)
            out[defer] = gs
            del model, flat, opt
    finally:
        ds.ops.enable_deferred_weight_grads(enable=False)
        ds.set_precision("fp32")
    # (the BatchNorm / column-sum reductions use float atomics: run-to-run differences in the last bits are expected; a
    # missing dependency would show up as stale or partial gradients, orders of magnitude above this bound)
    for a, b in zip(out[True], out[False]):
        assert rel(a, b) < 1e-5 and rel_l2(a, b) < 1e-6
    assert rel(out[True][0], out[True][1]) > 1e-2


def test_precision_16_train_step_is_bit_repeatable():
    """the benchmarked mode (precision 16, tensor-core front-end incl. both conv weight gradients, gradient sinks): train
    steps from the same parameters on the same batch give bit-identical loss and gradients, so that repeated runs of a
    training job or of the benchmark compute the same thing.  T' = 300 is eligible for the tensor-core weight gradients,
    and T' * B = 2400 rows make the fc head's weight gradient a split-K product"""
    from deepspeech_pytorch_b200.optim import FlatParams
    ds.set_precision("fp16")
    ocfg = oracle_cfg("lstm", True, 128, 3)
    P = O.init_params(ocfg, seed=13)
    x, targets, pct, tsz = O.synth_batch(8, 600, seed=3, lmin=5, lmax=20)
    model = make_model("lstm", True, 128, 3, params=P).train()
    flat = FlatParams(model, direct_grads=True)
    runs = []
    for _ in range(3):
        model.load_state_dict(P)
        loss = model.training_step((x.cuda(), targets, pct.clone(), tsz), 0)
        loss.backward()
        torch.cuda.synchronize()
        runs.append((float(loss), flat.grad.clone()))
    for loss, grad in runs[1:]:
        assert loss == runs[0][0]
        assert torch.equal(grad, runs[0][1]), float((grad - runs[0][1]).abs().max())


@pytest.mark.parametrize("cfg", ["1", "2", "3"])
def test_gemm_f16_tile_configurations_vs_fp64(cfg, monkeypatch):
    """the precision-16 mode's GEMM (fp16 K-major operands, fp32 accumulation) in every tile configuration, incl. the
    2-CTAs-per-SM one the short-K projection shape selects, a K tail (K % 64 != 0), split-K and alpha / beta"""
    import ctypes as C
    monkeypatch.setenv("DS2_GEMM16_CFG", cfg)
    lib = ds.get_lib()
    g = torch.Generator(device="cuda").manual_seed(7)
    for M, N, K, alpha, beta in [(640, 520, 1000, 1.0, 0.0), (4096, 1024, 4104, 0.5, 1.0), (300, 96, 72, 1.0, 0.0)]:
        a = (torch.randn(M, K, generator=g, device="cuda")).half()
        b = (torch.randn(N, K, generator=g, device="cuda")).half()
        c0 = torch.randn(M, N, generator=g, device="cuda")
        out = c0.clone()
        rc = lib.ds2_gemm_f16(M, N, K, alpha, C.c_void_p(a.data_ptr()), K, C.c_void_p(b.data_ptr()), K, beta,
                              C.c_void_p(out.data_ptr()), N, C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, lib.ds2_last_error()
        ref = alpha * (a.double() @ b.double().t()) + beta * c0.double()
        assert rel_l2(out, ref) < 1e-5, (cfg, M, N, K)


@pytest.mark.parametrize("T,B", [(301, 5), (1000, 3), (301, 4), (640, 6)])
def test_conv_frontend_tensor_core_paths_vs_fp32(T, B):
    """tensor-core front-end (conv2 forward / data gradient / weight gradient on tcgen05, TF32) against the FFMA
    front-end on a ragged batch: several 128-position tiles per row, a partially filled last tile, fully masked tiles,
    BatchNorm batch statistics (running stats) from the fused partial sums; masked frames exactly zero.  Odd batches
    run one CTA per tile, even ones the 2-CTA clusters that share the tap matrices by multicast."""
    g = torch.Generator().manual_seed(T)
    x = torch.randn(B, 1, 161, T, generator=g)
    lens = sorted([max(40, T - (T // 4) * i) for i in range(B)], reverse=True)
    for b, l in enumerate(lens):
        x[b, :, :, l:] = 0
    outs = {}
    for prec in ("fp32", "tf32"):
        ds.set_precision(prec)
        model = make_model("gru", True, 8, 1).train()
        torch.manual_seed(1)
        sm = model.conv.seq_module
        with torch.no_grad():
            for m in (sm[0], sm[3]):
                m.weight.copy_(torch.randn(m.weight.shape, generator=torch.Generator().manual_seed(5)).cuda() * 0.05)
                m.bias.copy_(torch.randn(m.bias.shape, generator=torch.Generator().manual_seed(6)).cuda() * 0.1)
        out_len = model.get_seq_lens(torch.tensor(lens)).cuda()
        y = ds.ops.ConvFrontend.apply(x.cuda(), out_len, sm[0].weight, sm[0].bias, sm[1].weight, sm[1].bias,
                                      sm[1].running_mean, sm[1].running_var, sm[3].weight, sm[3].bias, sm[4].weight,
                                      sm[4].bias, sm[4].running_mean, sm[4].running_var, True, 0.1, 1e-5)
        dy = torch.randn(y.shape, generator=torch.Generator().manual_seed(9)).cuda()
        for m in (sm[0], sm[1], sm[3], sm[4]):
            m.weight.grad = m.bias.grad = None
        (y * dy).sum().backward()
        torch.cuda.synchronize()
        outs[prec] = (y.detach().clone(), sm[1].running_mean.clone(), sm[1].running_var.clone(),
                      sm[4].running_mean.clone(), sm[4].running_var.clone(), out_len.cpu(),
                      [m.weight.grad.clone() for m in (sm[0], sm[1], sm[3], sm[4])])
    a, r = outs["tf32"], outs["fp32"]
    assert rel(a[0], r[0]) < 3e-3 and rel_l2(a[0], r[0]) < 1e-3
    for i in range(1, 5):
        assert rel(a[i], r[i]) < 1e-3, i
    # gradients: conv1 weight (through the conv2 data gradient), BN1, conv2 weight, BN2.  The Hardtanh clips are not
    # smooth, so a TF32 forward deviation flips a few clip masks: percent-level bound, not 1e-3
    for i, (ga, gr) in enumerate(zip(a[6], r[6])):
        assert torch.isfinite(ga).all() and rel_l2(ga, gr) < 3e-2, (i, rel_l2(ga, gr))
    ol = a[5]
    for b in range(B):
        if int(ol[b]) < a[0].shape[0]:
            assert float(a[0][int(ol[b]):, b].abs().max()) == 0.0
