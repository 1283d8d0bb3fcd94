"""Seeded synthetic side inputs shared by tests/golden/make_golden.py and the tests (so fixtures need not store them)."""
import torch


def seeded_energy_pitch(seed, olens, L):
    """Per-frame energy U(0,130) and pitch (0 w.p. 0.3 else U(71,671)), zero past each utterance's length."""
    g = torch.Generator().manual_seed(seed)
    B = olens.numel()
    es = torch.rand(B, L, generator=g) * 130.0
    ps = torch.rand(B, L, generator=g) * 600.0 + 71.0
    ps[torch.rand(B, L, generator=g) < 0.3] = 0.0
    for b in range(B):
        es[b, olens[b]:] = 0.0
        ps[b, olens[b]:] = 0.0
    return es, ps


# Train-mode step against the reference (tests/test_gpu_train.py): make_batch arguments per case, and the seed of the
# generator both runs draw their dropout masks from, in call order.
TRAIN_CASES = {
    "dense": dict(B=2, T=20, L=150, seed=16),
    "ragged": dict(B=3, T=23, L=181, seed=17, ilens=[23, 17, 9], olens=[181, 140, 66]),
}
DROPOUT_SEED = 5

# The reference scripts' two model calls (tests/test_gpu_dropin_scripts.py): the phoneme string handed to
# inference.synth, and the (T, L) of the batches of one that evaluation.evaluate iterates over (make_batch seed 300 + i).
SYNTH_TEXT = "HH AH0 L OW1 W ER1 L D DH IH1 S IH1 Z AH0 T EH1 S T AH1 V DH AH0 B IY1 T UW1 HH AH1 N D R AH0 D P AE1 TH"
EVAL_CASES = [(23, 180), (41, 333), (9, 70)]
