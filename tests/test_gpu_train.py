"""Train-mode forward + backward (SURVEY.md section 8f-1) against the reference's own autograd.

* unit level: each autograd stage of fastspeech2_b200/train.py against the same torch op's autograd in float64;
* model level: `model.train(); loss, report = model(...); loss.backward()` against the UNMODIFIED reference class (CPU,
  fp32; its results stored in tests/golden by make_golden.py) with identical weights, inputs and dropout masks --
  `torch.nn.functional.dropout` was patched in the reference run to draw masks from a seeded generator; the same masks
  are redrawn and injected into our path (`model.dropout_masks`).  Compared: the loss, the seven report values, the
  gradient of every parameter, BatchNorm's updated running statistics.
Stated tolerance: fp32 arithmetic with different summation orders (weight gradients are sums over thousands of frames,
split-K with atomics here, one long chain in the reference) -- loss rel 1e-4; gradients max-abs <= 1e-2 * max|g_ref| + 1e-6
(observed: worst 5.3e-3 on a decoder conv-FFN weight, typically 1e-4).
Needs a B200: run with `-m gpu`."""
import math

import pytest
import torch

from fastspeech2_b200 import FeedForwardTransformer
from fastspeech2_b200 import train as T
from fastspeech2_b200.hparams import load_hp
from fastspeech2_b200.synthetic import make_batch
from _synth import DROPOUT_SEED, TRAIN_CASES

pytestmark = pytest.mark.gpu
KEYS = ("xs", "ilens", "ys", "olens", "ds", "es", "ps")


def rel_err(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).abs().max() / (want.abs().max() + 1e-12))


# ---- unit level ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(3, 70, 256, 1024, 9, 1), (2, 133, 384, 384, 1, 0), (4, 41, 80, 256, 5, 0), (2, 50, 256, 256, 3, 1)])
def test_conv_fn_gradients(shape):
    B, L, K, N, taps, act = shape
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(B, L, K, generator=g); w = torch.randn(N, K, taps, generator=g) / math.sqrt(K * taps); b = torch.randn(N, generator=g)
    gy = torch.randn(B, L, N, generator=g)
    xr, wr, br = (t.double().requires_grad_() for t in (x, w, b))
    y = torch.nn.functional.conv1d(xr.transpose(1, 2), wr, br, padding=(taps - 1) // 2).transpose(1, 2)
    y = torch.relu(y) if act else y
    y.backward(gy.double())
    xc, wc, bc = (t.cuda().requires_grad_() for t in (x, w, b))
    out = T.ConvFn.apply(xc, wc, bc, act, None)
    out.backward(gy.cuda())
    assert rel_err(out, y) < 1e-5
    assert rel_err(xc.grad, xr.grad) < 1e-5 and rel_err(wc.grad, wr.grad) < 1e-5 and rel_err(bc.grad, br.grad) < 1e-5


@pytest.mark.parametrize("C", [256, 384])
def test_layernorm_fn_gradients(C):
    g = torch.Generator().manual_seed(C)
    x = torch.randn(5, 77, C, generator=g) * 2 + 0.3; w = 1 + 0.2 * torch.randn(C, generator=g); b = torch.randn(C, generator=g)
    gy = torch.randn(5, 77, C, generator=g)
    xr, wr, br = (t.double().requires_grad_() for t in (x, w, b))
    torch.nn.functional.layer_norm(xr, (C,), wr, br, 1e-5).backward(gy.double())
    xc, wc, bc = (t.cuda().requires_grad_() for t in (x, w, b))
    T.LayerNormFn.apply(xc, wc, bc, 1e-5).backward(gy.cuda())
    assert rel_err(xc.grad, xr.grad) < 1e-5 and rel_err(wc.grad, wr.grad) < 1e-5 and rel_err(bc.grad, br.grad) < 1e-5


@pytest.mark.parametrize("C,L,heads", [(256, 100, 2), (384, 333, 2)])
def test_attention_fn_gradients(C, L, heads):
    B, dk = 3, C // heads
    g = torch.Generator().manual_seed(C + L)
    q, k, v = (torch.randn(B, L, C, generator=g) for _ in range(3))
    lens = torch.tensor([L, L // 2, 7])
    drop = torch.rand(B, heads, L, L, generator=g) >= 0.2
    gy = torch.randn(B, L, C, generator=g)
    qr, kr, vr = (t.double().requires_grad_() for t in (q, k, v))
    split = lambda t: t.view(B, L, heads, dk).transpose(1, 2)
    s = split(qr) @ split(kr).transpose(-1, -2) / math.sqrt(dk)
    valid = torch.arange(L)[None] < lens[:, None]
    m = ~(valid[:, None, :] & valid[:, :, None])[:, None]
    p = torch.softmax(s.masked_fill(m, -float("inf")), -1).masked_fill(m, 0.0)
    pd = p * drop.double() / 0.8
    want = (pd @ split(vr)).transpose(1, 2).reshape(B, L, C)
    want.backward(gy.double())
    qc, kc, vc = (t.cuda().requires_grad_() for t in (q, k, v))
    got = T.AttentionFn.apply(qc, kc, vc, lens.cuda(), heads, 0.2, drop.to(torch.uint8).cuda())
    got.backward(gy.cuda())
    assert rel_err(got, want) < 1e-5
    for a, r in ((qc, qr), (kc, kr), (vc, vr)):
        assert torch.isfinite(a.grad).all() and rel_err(a.grad, torch.nan_to_num(r.grad)) < 2e-5


def test_batchnorm_fn_matches_torch_train_mode():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(4, 90, 256, generator=g) * 1.5 + 0.2
    bn = torch.nn.BatchNorm1d(256).double()
    with torch.no_grad():
        bn.weight.copy_(1 + 0.1 * torch.randn(256, generator=g)); bn.bias.copy_(torch.randn(256, generator=g))
    gy = torch.randn(4, 90, 256, generator=g)
    xr = x.double().requires_grad_()
    torch.tanh(bn(xr.transpose(1, 2))).transpose(1, 2).backward(gy.double())
    xc = x.cuda().requires_grad_()
    w, b = bn.weight.detach().float().cuda().requires_grad_(), bn.bias.detach().float().cuda().requires_grad_()
    rm, rv = torch.zeros(256).cuda(), torch.ones(256).cuda()
    T.BatchNormFn.apply(xc, w, b, rm, rv, 1e-5, 0.1, T.ACT_TANH).backward(gy.cuda())
    assert rel_err(xc.grad, xr.grad) < 2e-5 and rel_err(w.grad, bn.weight.grad) < 2e-5 and rel_err(b.grad, bn.bias.grad) < 2e-5
    assert rel_err(rm, bn.running_mean) < 1e-5 and rel_err(rv, bn.running_var) < 1e-5


def test_philox_mask_rate_and_determinism():
    src = T.MaskSource(seed=1234)
    m1 = src.next((7, 333, 256), 0.2, torch.device("cuda"))
    m2 = T.MaskSource(seed=1234).next((7, 333, 256), 0.2, torch.device("cuda"))
    assert torch.equal(m1, m2) and abs(float(m1.float().mean()) - 0.8) < 5e-3
    assert not torch.equal(m1, T.MaskSource(seed=99).next((7, 333, 256), 0.2, torch.device("cuda")))


# ---- model level: the unmodified reference in train mode with shared dropout masks ------------------------------------
class _Recorded(T.MaskSource):
    """Masks recorded from the reference run, in call order; sites where the reference drops a channel-first [B, C, time]
    tensor (conv predictors, Postnet) are permuted to this path's [B, time, C] layout."""

    def __init__(self, masks):
        super().__init__(seed=0, injected=None)
        self.recorded = list(masks)

    def next(self, shape, p, device):
        self.calls += 1
        m = self.recorded.pop(0)
        if tuple(m.shape) != tuple(shape):
            assert m.dim() == 3 and tuple(m.permute(0, 2, 1).shape) == tuple(shape), (self.calls, tuple(m.shape), tuple(shape))
            m = m.permute(0, 2, 1)
        return m.to(torch.uint8).contiguous().to(device)


@pytest.mark.parametrize("ragged", [False, True])
def test_train_step_matches_reference_autograd(weights, golden, ragged):
    """The reference's side is stored in tests/golden/train_{dense,ragged}.npz (make_golden.py --train-only): the dropout
    masks are redrawn here from the same seeded generator in the reference's call order, and the gradients are compared
    in their max-abs, their L2 norm and a seeded sample of entries of every parameter."""
    ref = golden("train_ragged" if ragged else "train_dense")
    kw = dict(TRAIN_CASES["ragged" if ragged else "dense"])
    bt = make_batch(kw.pop("B"), kw.pop("T"), kw.pop("L"), **kw)
    gen = torch.Generator().manual_seed(DROPOUT_SEED)
    recorded = [torch.rand(tuple(shape[:ndim]), generator=gen) >= p
                for shape, ndim, p in zip(ref["mask_shape"], ref["mask_ndim"], ref["mask_p"])]

    ours = FeedForwardTransformer(68, 80, load_hp(), precision="fp32")
    ours.load_state_dict(weights, strict=True)
    ours = ours.cuda().train()
    ours.dropout_masks = _Recorded(recorded)
    loss, rep = ours(*[bt[k].cuda() for k in KEYS])
    loss.backward()
    torch.cuda.synchronize()
    assert not ours.dropout_masks.recorded, "the reference made more dropout calls than this path"

    loss_ref = float(ref["loss"])
    assert abs(float(loss) - loss_ref) <= 1e-4 * abs(loss_ref)
    assert [list(r)[0] for r in rep] == list(ref["report_keys"])
    for a, vb in zip(rep, ref["report"]):
        va = list(a.values())[0]
        assert abs(va - vb) <= 1e-4 * max(1.0, abs(vb)), (a, vb)
    params = dict(ours.named_parameters())
    assert sorted(params) == sorted(ref["grad_names"])
    worst = ("", 0.0)
    for i, name in enumerate(ref["grad_names"]):
        p = params[name]
        assert p.numel() == ref["grad_numel"][i], name
        if not ref["grad_present"][i]:
            assert p.grad is None, f"{name}: the reference leaves no gradient here"
            continue
        assert p.grad is not None, f"{name}: missing gradient"
        assert torch.isfinite(p.grad).all(), name
        g = p.grad.detach().double().cpu().reshape(-1)
        scale = float(ref["grad_maxabs"][i])
        sel = slice(ref["grad_off"][i], ref["grad_off"][i + 1])
        err = float((g[torch.from_numpy(ref["grad_idx"][sel]).long()] - torch.from_numpy(ref["grad_val"][sel]).double()).abs().max())
        if err / (scale + 1e-12) > worst[1]:
            worst = (name, err / (scale + 1e-12))
        assert err <= 1e-2 * scale + 1e-6, f"{name}: grad max-abs err {err:.3e} vs scale {scale:.3e}"
        assert abs(float(g.abs().max()) - scale) <= 1e-2 * scale + 1e-6, (name, float(g.abs().max()), scale)
        norm = float(ref["grad_norm"][i])
        assert abs(float(g.norm()) - norm) <= 1e-2 * norm + 1e-6, (name, float(g.norm()), norm)
    print("worst relative gradient error:", worst)
    bufs = {n: b for n, b in ours.named_buffers() if "running" in n or "num_batches" in n}
    assert list(bufs) == list(ref["buf_names"])
    for j, (n1, b1) in enumerate(bufs.items()):
        assert torch.allclose(b1.cpu().double(), torch.from_numpy(ref[f"buf{j}"]).double(), rtol=1e-4, atol=1e-6), n1


def test_optimizer_step_through_the_reference_training_recipe(weights):
    """train_fastspeech.py:100-131 in miniature: forward, backward, clip_grad_norm_, Adam step, zero_grad, then an eval
    forward that sees the updated weights (the repack fingerprint follows the optimizer's in-place updates)."""
    m = FeedForwardTransformer(68, 80, load_hp(), precision="fp32")
    m.load_state_dict(weights, strict=True)
    m = m.cuda()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    bt = make_batch(2, 20, 150, seed=21)
    args = [bt[k].cuda() for k in KEYS]
    m.eval()
    with torch.no_grad():
        l0, _ = m(*args)
    m.train()
    losses = []
    for _ in range(3):
        loss, report = m(*args)
        loss.backward()
        gn = torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
        assert math.isfinite(float(gn))
        opt.step(); opt.zero_grad()
        losses.append(float(loss))
    m.eval()
    with torch.no_grad():
        l1, _ = m(*args)
    assert float(l1) < float(l0), (float(l0), float(l1), losses)
