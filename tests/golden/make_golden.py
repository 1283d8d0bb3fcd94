#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference.

It needs a checkout of the reference FastSpeech2 project, given as the first
argument; the tests themselves only read the stored fixtures:

    python tests/golden/make_golden.py /path/to/FastSpeech2 [--collate-only | --filelist-only | --train-only | --dropin-only]

The reference is imported through a `sys.modules` shim for five third-party
packages its import chain touches but the model path never uses (SURVEY.md
section 8c).  Weights come from `fastspeech2_b200.weights.synthetic_state_dict`
(seeded, module-independent) and are loaded with `load_state_dict(strict=True)`,
which also pins checkpoint-key compatibility.  Only inputs + outputs are stored
(a few hundred KB); tests regenerate the weights from the seed.
"""
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, REPO)

for name in ("librosa", "nltk", "g2p_en", "unidecode", "inflect"):
    sys.modules[name] = types.ModuleType(name)
sys.modules["g2p_en"].G2p = object
sys.modules["unidecode"].unidecode = lambda s: s
sys.modules["inflect"].engine = lambda: None
sys.path.insert(0, REF)
os.chdir(REF)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from fastspeech import FeedForwardTransformer  # noqa: E402  (the reference)
from core.duration_modeling.length_regulator import LengthRegulator  # noqa: E402
from utils.hparams import HParam  # noqa: E402
from fastspeech2_b200.weights import ModelDims, synthetic_state_dict  # noqa: E402
sys.path.insert(0, os.path.dirname(HERE))
from _synth import seeded_energy_pitch  # noqa: E402  (tests/_synth.py, shared with the tests)

WEIGHT_SEED = 7
torch.set_num_threads(1)  # deterministic reduction order for the fixtures


def build_reference():
    hp = HParam("configs/default.yaml")
    model = FeedForwardTransformer(68, 80, hp)
    model.load_state_dict(synthetic_state_dict(WEIGHT_SEED, ModelDims()), strict=True)
    model.eval()
    return model, hp


def ragged_case(seed, ilens, max_d=6, zero_prob=0.15):
    g = torch.Generator().manual_seed(seed)
    B, T = len(ilens), max(ilens)
    xs = torch.zeros(B, T, dtype=torch.int64)
    ds = torch.zeros(B, T, dtype=torch.int64)
    for b, n in enumerate(ilens):
        xs[b, :n] = torch.randint(1, 68, (n,), generator=g)
        d = torch.randint(1, max_d + 1, (n,), generator=g)
        d[torch.rand(n, generator=g) < zero_prob] = 0
        if d.sum() == 0:
            d[0] = 1
        ds[b, :n] = d
    olens = ds.sum(1)
    L = int(olens.max())
    es = torch.rand(B, L, generator=g) * 130.0
    ps = torch.rand(B, L, generator=g) * 600.0 + 71.0
    ps[torch.rand(B, L, generator=g) < 0.3] = 0.0
    for b in range(B):
        es[b, olens[b]:] = 0.0
        ps[b, olens[b]:] = 0.0
    ys = torch.randn(B, L, 80, generator=g)
    return xs, torch.tensor(ilens), olens, ds, es, ps, ys


def npz(name, **arrs):
    out = {}
    for k, v in arrs.items():
        out[k] = v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("wrote", name, {k: tuple(v.shape) for k, v in out.items()})


def main():
    model, hp = build_reference()
    with open(os.path.join(HERE, "state_dict_keys.json"), "w") as f:
        json.dump([[k, list(v.shape), str(v.dtype)] for k, v in model.state_dict().items()], f, indent=0)

    with torch.no_grad():
        # 1. teacher-forced _forward on a ragged batch (fastspeech.py:169-243, is_inference=False)
        xs, ilens, olens, ds, es, ps, ys = ragged_case(11, [17, 11, 5])
        b, a, d, e, p = model._forward(xs, ilens, olens, ds.clone(), es, ps, is_inference=False)
        npz("tf_ragged", xs=xs, ilens=ilens, olens=olens, ds=ds, es=es, ps=ps, ys=ys,
            before=b, after=a, d_outs=d, e_outs=e, p_outs=p)

        # 2. forward() loss + report_keys on the same batch (fastspeech.py:245-337)
        loss, report = model(xs, ilens, ys, olens, ds.clone(), es, ps)
        npz("tf_ragged_loss", loss=loss, report=np.array([list(r.values())[0] for r in report], dtype=np.float64))
        with open(os.path.join(HERE, "report_keys.json"), "w") as f:
            json.dump([list(r.keys())[0] for r in report], f)

        # 3. is_inference=True on a ragged batch (decoder unmasked, fastspeech.py:193-196,221-224)
        xs3, ilens3, *_ = ragged_case(12, [21, 13, 8])
        b, a, d, eh, ph = model._forward(xs3, ilens3, is_inference=True)
        npz("inf_ragged", xs=xs3, ilens=ilens3, before=b, after=a, d_outs=d,
            e_ids=eh.argmax(-1), p_ids=ph.argmax(-1))

        # 4. single-utterance inference() (fastspeech.py:339-357)
        x4 = torch.randint(1, 68, (23,), generator=torch.Generator().manual_seed(13))
        npz("inf_single", x=x4, mel=model.inference(x4))

        # 5. the reference's own unit-test shapes (tests/test_fastspeech2.py:7-20), eval mode
        x = torch.ones(2, 100).to(dtype=torch.int64)
        il = torch.tensor([100, 100])
        y = torch.ones(2, 100, 80)
        dur = torch.ones(2, 100)
        e1 = torch.ones(2, 100)
        loss, report = model(x, il, y, il.clone(), dur.clone(), e1, e1.clone())
        npz("unit_shapes", loss=loss, report=np.array([list(r.values())[0] for r in report], dtype=np.float64))

    # 6. LengthRegulator edge cases (length_regulator.py:38-95)
    lr = LengthRegulator()
    g = torch.Generator().manual_seed(14)
    hs = torch.randn(4, 9, 16, generator=g)
    il = torch.tensor([9, 6, 4, 1])
    d_int = torch.tensor([[2, 0, 3, 1, 0, 0, 4, 1, 2],
                          [1, 1, 0, 5, 0, 2, 7, 7, 7],      # entries past ilen are ignored
                          [0, 0, 0, 0, 3, 3, 3, 3, 3],      # all-zero slice -> filled with 1, in place
                          [0, 9, 9, 9, 9, 9, 9, 9, 9]], dtype=torch.int64)
    d_mut = d_int.clone()
    out_a = lr(hs, d_mut, il)
    d_alpha = d_int.clone()
    out_b = lr(hs, d_alpha, il, alpha=2.5)      # round-half-even of d*2.5; caller's ds NOT mutated
    d_f = torch.tensor([[1.0, 2.9, 0.5, 0.0, 1.0, 3.2, 0.0, 1.0, 2.0],
                        [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 5.0, 5.0, 5.0],
                        [0.5, 0.4, 0.0, 0.0, 1.0, 1.0, 1.0, 1.0, 1.0],   # sum != 0 but every int() is 0
                        [2.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]])
    d_f_mut = d_f.clone()
    # utterance 2 would expand to zero frames (torch.cat of empties is fine in the reference)
    out_c = lr(hs, d_f_mut, il)
    npz("length_regulator", hs=hs, ilens=il, d_int=d_int, d_int_after=d_mut, out_int=out_a,
        d_alpha_after=d_alpha, out_alpha=out_b, d_float=d_f, d_float_after=d_f_mut, out_float=out_c)

    # 7. bucketize edges (variance_predictor.py:154-159,227-232)
    eb, pb = model.energy_predictor.energy_bins, model.pitch_predictor.pitch_bins
    vals_e = torch.cat([eb[:4], eb[-3:], torch.tensor([-1.0, 0.0, 1e9, float("nan"), float("inf"), -float("inf")]),
                        eb[100:104] + 1e-4, eb[100:104] - 1e-4])
    vals_p = torch.cat([pb[:4], pb[-3:], torch.tensor([-1.0, 0.0, 1e9, float("nan"), float("inf"), -float("inf")]),
                        pb[100:104] * (1 + 1e-6), pb[100:104] * (1 - 1e-6)])
    npz("bucketize", vals_e=vals_e, ids_e=model.energy_predictor.to_one_hot(vals_e).argmax(-1),
        vals_p=vals_p, ids_p=model.pitch_predictor.to_one_hot(vals_p).argmax(-1), e_bins=eb, p_bins=pb)


def collate_fixture():
    """Reference collate_tts (dataset/dataloader.py:96-118) on seeded synthetic items."""
    from dataset.dataloader import collate_tts
    g = np.random.RandomState(15)
    items = []
    for i, (T, L) in enumerate([(7, 31), (12, 50), (3, 9), (12, 44)]):
        d = g.randint(1, 6, size=T); d[-1] += L - d.sum() if d.sum() <= L else 0
        items.append((g.randint(1, 68, size=T), g.randn(L, 80).astype(np.float32), f"utt{i}", L, d.astype(np.int64),
                      g.rand(L).astype(np.float32) * 100, g.rand(L).astype(np.float32) * 500))
    out = collate_tts(items)
    npz("collate", **{f"x{i}": it[0] for i, it in enumerate(items)}, **{f"mel{i}": it[1] for i, it in enumerate(items)},
        **{f"d{i}": it[4] for i, it in enumerate(items)}, **{f"e{i}": it[5] for i, it in enumerate(items)},
        **{f"p{i}": it[6] for i, it in enumerate(items)},
        inputs=out[0], ilens=out[1], mels=out[2], labels=out[3], olens=out[4], durations=out[6], energys=out[7], pitches=out[8])


def filelist_twin():
    """SURVEY 8d "ragged twin" of c2: the first 64 rows of the reference's filelists/train_filelist.txt (real phoneme
    ids through the reference's own phonemes_to_sequence, real durations, dataset/dataloader.py:47-64), teacher-forced
    through the live reference.  The full outputs are ~40 MB, so the fixture keeps every d_outs, the mels of the
    shortest and the longest utterance, e/p predictions of eight utterances, and per-utterance means of the rest."""
    from dataset.texts import phonemes_to_sequence
    with open(os.path.join(REF, "filelists", "train_filelist.txt")) as f:
        rows = [line.strip().split("|") for line in f][:64]
    ids = [phonemes_to_sequence(r[3].split()) for r in rows]
    durs = [[int(v) for v in r[2].split()][:len(i)] for r, i in zip(rows, ids)]
    B, T = len(ids), max(len(i) for i in ids)
    xs = torch.zeros(B, T, dtype=torch.int64)
    ds = torch.zeros(B, T, dtype=torch.int64)
    for b, (i, d) in enumerate(zip(ids, durs)):
        xs[b, :len(i)] = torch.tensor(i)
        ds[b, :len(d)] = torch.tensor(d)
    ilens = torch.tensor([len(i) for i in ids])
    olens = ds.sum(1)
    L = int(olens.max())
    es, ps = seeded_energy_pitch(16, olens, L)
    model, _ = build_reference()
    torch.set_num_threads(os.cpu_count())
    with torch.no_grad():
        b_, a_, d_, e_, p_ = model._forward(xs, ilens, olens, ds.clone(), es, ps, is_inference=False)
    torch.set_num_threads(1)
    lo, hi = int(olens.argmin()), int(olens.argmax())
    keep = sorted({lo, hi, 0, 9, 18, 27, 45, 63})
    valid = (torch.arange(L)[None, :] < olens[:, None]).float()
    npz("filelist64", xs=xs, ilens=ilens, olens=olens, ds=ds, es_seed=16,
        d_outs=d_, mel_rows=np.array([lo, hi]), after_lo=a_[lo, :olens[lo]], after_hi=a_[hi, :olens[hi]],
        before_lo=b_[lo, :olens[lo]],
        ep_rows=np.array(keep), e_sel=e_[keep], p_sel=p_[keep],
        after_mean=(a_.double() * valid[..., None]).sum((1, 2)) / (olens.double() * 80),
        after_absmean=(a_.double().abs() * valid[..., None]).sum((1, 2)) / (olens.double() * 80),
        before_mean=(b_.double() * valid[..., None]).sum((1, 2)) / (olens.double() * 80),
        e_mean=(e_.double() * valid).sum(1) / olens.double(), p_mean=(p_.double() * valid).sum(1) / olens.double())


GRAD_SAMPLES = 32      # gradient entries stored per parameter (the full gradients are ~100 MB per case)


def train_step_fixture():
    """`model.train(); loss, report = model(...); loss.backward()` of the reference on the CPU in fp32, with every dropout
    mask drawn in call order from one seeded generator (tests/_synth.py).  Stored: the shape and rate of each dropout
    call (the test redraws the same masks), the loss, the report, per parameter the max-abs and L2 norm of its gradient
    plus GRAD_SAMPLES entries at seeded positions, and BatchNorm's updated running statistics."""
    from fastspeech2_b200.synthetic import make_batch
    from _synth import DROPOUT_SEED, TRAIN_CASES
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    real = torch.nn.functional.dropout
    for case, kw in TRAIN_CASES.items():
        kw = dict(kw)
        bt = make_batch(kw.pop("B"), kw.pop("T"), kw.pop("L"), **kw)
        model, _ = build_reference()
        model.train()
        gen = torch.Generator().manual_seed(DROPOUT_SEED)
        shapes, rates = [], []

        def shared_dropout(input, p=0.5, training=True, inplace=False):
            if not training or p == 0.0:
                return input
            m = torch.rand(input.shape, generator=gen) >= p
            shapes.append(list(input.shape) + [1] * (4 - input.dim()))
            rates.append((input.dim(), p))
            return input * m.to(input.dtype) / (1.0 - p)

        torch.nn.functional.dropout = shared_dropout
        try:
            loss, report = model(*[bt[k] for k in ("xs", "ilens", "ys", "olens", "ds", "es", "ps")])
            loss.backward()
        finally:
            torch.nn.functional.dropout = real
        pick = torch.Generator().manual_seed(0)
        names, numel, has, maxabs, norm, off, idx, val = [], [], [], [], [], [0], [], []
        for name, p in model.named_parameters():
            names.append(name)
            numel.append(p.numel())
            has.append(p.grad is not None)
            g = p.grad.detach().reshape(-1) if p.grad is not None else torch.zeros(0)
            maxabs.append(float(g.abs().max()) if g.numel() else 0.0)
            norm.append(float(g.double().norm()) if g.numel() else 0.0)
            i = torch.randperm(g.numel(), generator=pick)[:GRAD_SAMPLES].sort().values if g.numel() else torch.zeros(0, dtype=torch.int64)
            idx.append(i.to(torch.int32))
            val.append(g[i])
            off.append(off[-1] + i.numel())
        bufs = {n: b for n, b in model.named_buffers() if "running" in n or "num_batches" in n}
        npz(f"train_{case}", mask_shape=np.array(shapes, dtype=np.int64), mask_ndim=np.array([r[0] for r in rates]),
            mask_p=np.array([r[1] for r in rates], dtype=np.float64), loss=loss.double(),
            report_keys=np.array([list(r.keys())[0] for r in report]),
            report=np.array([float(list(r.values())[0]) for r in report], dtype=np.float64),
            grad_names=np.array(names), grad_numel=np.array(numel), grad_present=np.array(has),
            grad_maxabs=np.array(maxabs), grad_norm=np.array(norm), grad_off=np.array(off),
            grad_idx=torch.cat(idx), grad_val=torch.cat(val),
            buf_names=np.array(list(bufs)), **{f"buf{i}": b for i, b in enumerate(bufs.values())})
    torch.set_num_threads(1)


def dropin_fixture():
    """What the reference's own scripts compute with the reference class, for the drop-in test: inference.synth's mel
    (the phoneme string through the reference's text front end, then model.inference; inference.py:111-130) and
    evaluation.evaluate's three mean L1 distances (evaluation.py:12-41), here on the CPU."""
    from dataset.texts import phonemes_to_sequence
    from fastspeech2_b200.synthetic import make_batch
    from _synth import EVAL_CASES, SYNTH_TEXT
    model, _ = build_reference()
    ids = torch.LongTensor(np.asarray(phonemes_to_sequence(SYNTH_TEXT)))
    l1 = torch.nn.L1Loss()
    diffs = []
    with torch.no_grad():
        mel = model.inference(ids)
        for i, (T, L) in enumerate(EVAL_CASES):
            bt = make_batch(1, T, L, seed=300 + i)
            _, _, d, e, p = model._forward(bt["xs"], bt["ilens"], bt["olens"], bt["ds"], es=bt["es"], ps=bt["ps"], is_inference=False)
            diffs.append([l1(p, bt["ps"]).item(), l1(e, bt["es"]).item(), l1(d, bt["ds"]).item()])
    npz("dropin_scripts", ids=ids, mel=mel, evaluate=np.array(diffs, dtype=np.float64).mean(0))


if __name__ == "__main__":
    if "--collate-only" in sys.argv:
        collate_fixture()
    elif "--filelist-only" in sys.argv:
        filelist_twin()
    elif "--train-only" in sys.argv:
        train_step_fixture()
    elif "--dropin-only" in sys.argv:
        dropin_fixture()
    else:
        main()
        collate_fixture()
        filelist_twin()
        train_step_fixture()
        dropin_fixture()
