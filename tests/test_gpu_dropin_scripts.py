"""The reference's own scripts' model calls, end to end on the B200 against this repo's class (SURVEY.md section 7 step 7 /
8b): what `inference.synth(text, model, hp)` (inference.py:111-130) and `evaluation.evaluate(hp, loader, model)`
(evaluation.py:12-41) do with the model, in a script started through the launcher `python -m fastspeech2_b200.dropin_run`
from a stand-in checkout whose own `fastspeech.py` the launcher must shadow.  The reference class's results of the same
two calls with identical weights -- the mel of the phoneme string, and the three mean L1 distances of the pitch, energy
and duration predictions -- are stored in tests/golden/dropin_scripts.npz (make_golden.py --dropin-only, CPU, fp32);
results must agree within the fp32 gate."""
import os
import subprocess
import sys
import textwrap

import pytest

from conftest import GOLDEN, REPO

pytestmark = pytest.mark.gpu

SCRIPT = textwrap.dedent('''
    import sys
    import numpy as np
    import torch
    from fastspeech import FeedForwardTransformer     # inference.py:9, evaluation.py:3
    from fastspeech2_b200 import synthetic_state_dict
    from fastspeech2_b200.hparams import load_hp
    from fastspeech2_b200.synthetic import make_batch

    golden, tests_dir = sys.argv[1], sys.argv[2]
    sys.path.insert(0, tests_dir)
    from _synth import EVAL_CASES
    ref = np.load(golden)
    assert FeedForwardTransformer.__module__.startswith("fastspeech2_b200"), FeedForwardTransformer.__module__
    hp = load_hp()
    mine = FeedForwardTransformer(68, hp.audio.num_mels, hp); mine.load_state_dict(synthetic_state_dict(7), strict=True)

    # ---- inference.synth: phoneme ids (the reference's text front end, stored) -> model.inference on the GPU
    assert hp.train.ngpu > 0
    mine.eval()
    mine = mine.to(torch.device("cuda"))
    with torch.no_grad():
        mel = mine.inference(torch.LongTensor(ref["ids"]).to(torch.device("cuda")))
    assert mel.is_cuda and mel.dim() == 2 and mel.shape[1] == hp.audio.num_mels
    assert tuple(mel.shape) == ref["mel"].shape, (tuple(mel.shape), ref["mel"].shape)
    err = float((mel.cpu() - torch.from_numpy(ref["mel"])).abs().max())
    print("synth: mel", tuple(mel.shape), "max-abs err vs the reference class on CPU %.3e" % err)
    assert err <= 1e-4, err

    # ---- evaluation.evaluate: batches of one (the reference's own ilens line assumes that), every tensor moved with
    # .cuda(), teacher-forced _forward, mean L1 of the pitch / energy / duration predictions over the batches
    l1 = torch.nn.L1Loss()
    diffs = []
    mine.eval()
    for i, (T, L) in enumerate(EVAL_CASES):
        bt = make_batch(1, T, L, seed=300 + i)
        with torch.no_grad():
            ilens = torch.tensor([bt["xs"][-1].shape[0]], dtype=torch.long)
            _, _, d, e, p = mine._forward(bt["xs"].cuda(), ilens.cuda(), bt["olens"].cuda(), bt["ds"].cuda(),
                                          es=bt["es"].cuda(), ps=bt["ps"].cuda(), is_inference=False)
            diffs.append([l1(p, bt["ps"].cuda()).item(), l1(e, bt["es"].cuda()).item(), l1(d, bt["ds"].cuda()).item()])
    mine.train()
    got, want = np.mean(diffs, 0), ref["evaluate"]
    print("evaluate: ours", got, "reference", want)
    assert np.allclose(got, want, rtol=1e-4, atol=1e-4), (got, want)
    assert mine.training
    print("DROPIN_GPU_OK")
''')


def test_unmodified_synth_and_evaluate_on_gpu(tmp_path):
    ref = tmp_path / "checkout"
    ref.mkdir()
    (ref / "fastspeech.py").write_text("class FeedForwardTransformer:\n    pass\n")   # the reference's module, shadowed
    (ref / "check_dropin_gpu.py").write_text(SCRIPT)
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([REPO, env.get("PYTHONPATH", "")])
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    r = subprocess.run([sys.executable, "-m", "fastspeech2_b200.dropin_run", "check_dropin_gpu.py",
                        os.path.join(GOLDEN, "dropin_scripts.npz"), os.path.join(REPO, "tests")],
                       cwd=ref, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "DROPIN_GPU_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-4000:]
