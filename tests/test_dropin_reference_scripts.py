"""Drop-in at the level of the reference's own scripts (SURVEY.md section 8b/8c), in a subprocess started through the
launcher `python -m fastspeech2_b200.dropin_run <script>` with cwd = a checkout of the reference, exactly how
INTEGRATION.md tells a reference user to switch over (a plain PYTHONPATH entry is not enough: a script's own directory
precedes it).  The checkout is a stand-in built in a temporary directory: its own `fastspeech.py` defines a different
`FeedForwardTransformer`, and the script uses the two import forms of the reference's scripts
(`from fastspeech import FeedForwardTransformer` in inference.py:9 / evaluation.py:3, `import fastspeech` in
train_fastspeech.py:1).  Checked:

  * both forms resolve to this repo's class, and the launcher hands the script its arguments;
  * the class is constructed from the config object, and its checkpoint layout is the reference's
    (tests/golden/state_dict_keys.json, written from the reference class by make_golden.py);
  * checkpoints move through a file and load strictly, and the `--old_model` partial load (inference.py:163) works.
CPU only: no forward is executed here (that is the GPU suite's job)."""
import os
import subprocess
import sys
import textwrap

from conftest import GOLDEN, REPO

STANDIN = textwrap.dedent('''
    """Stand-in for the reference's own model module: the drop-in must shadow it."""
    class FeedForwardTransformer:
        pass
''')

SCRIPT = textwrap.dedent('''
    import json, os, sys
    import torch
    import fastspeech                                 # train_fastspeech.py:1
    from fastspeech import FeedForwardTransformer     # inference.py:9, evaluation.py:3
    from fastspeech2_b200.hparams import load_hp

    assert fastspeech.FeedForwardTransformer is FeedForwardTransformer
    assert FeedForwardTransformer.__module__.startswith("fastspeech2_b200"), FeedForwardTransformer.__module__
    keys_json, ckpt = sys.argv[1], sys.argv[2]
    hp = load_hp()
    mine = FeedForwardTransformer(68, hp.audio.num_mels, hp)
    sd = mine.state_dict()
    ref = json.load(open(keys_json))
    assert [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()] == ref

    torch.manual_seed(3)
    other = FeedForwardTransformer(68, hp.audio.num_mels, hp)
    with torch.no_grad():
        for p in other.parameters():
            p.normal_()
    torch.save({"model": other.state_dict()}, ckpt)
    loaded = torch.load(ckpt)["model"]
    mine.load_state_dict(loaded, strict=True)
    assert all(torch.equal(v, mine.state_dict()[k]) for k, v in loaded.items())
    assert float(mine.encoder.embed[-1].alpha) == float(other.encoder.embed[-1].alpha)
    old = {k: v for k, v in FeedForwardTransformer(68, hp.audio.num_mels, hp).state_dict().items() if "postnet" not in k}
    mine.load_state_dict(old, strict=False)                                  # inference.py:163 (--old_model)
    now = mine.state_dict()
    assert all(torch.equal(now[k], old[k] if "postnet" not in k else loaded[k]) for k in now)
    print("DROPIN_OK", sum(p.numel() for p in mine.parameters()))
''')


def _checkout(tmp_path):
    ref = tmp_path / "checkout"
    ref.mkdir()
    (ref / "fastspeech.py").write_text(STANDIN)
    return ref


def test_reference_scripts_import_our_class(tmp_path):
    ref = _checkout(tmp_path)
    (ref / "check_dropin.py").write_text(SCRIPT)
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([REPO, env.get("PYTHONPATH", "")])
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    r = subprocess.run([sys.executable, "-m", "fastspeech2_b200.dropin_run", "check_dropin.py",
                        os.path.join(GOLDEN, "state_dict_keys.json"), str(tmp_path / "ckpt.pyt")],
                       cwd=ref, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "DROPIN_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_plain_pythonpath_is_shadowed_by_the_script_directory(tmp_path):
    """Documents why the launcher exists: with cwd (or the script directory) first on sys.path the reference's own
    fastspeech.py wins over a PYTHONPATH entry."""
    ref = _checkout(tmp_path)
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(REPO, "dropin"), REPO, env.get("PYTHONPATH", "")])
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    code = "import importlib.util; print(importlib.util.find_spec('fastspeech').origin)"
    r = subprocess.run([sys.executable, "-c", code], cwd=ref, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == str(ref / "fastspeech.py"), r.stdout + r.stderr[-2000:]
