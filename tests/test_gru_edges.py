"""Counts model (GRU) at edges the golden and ragged-shape tests do not reach, against the CPU oracle (oracle/gru_oracle.py).

  * feature widths around the fused layer-0 input projection of the tensor-core recurrence: it zero-pads K = F to 16 and
    stages each tile's x with 16 * F threads.  F = 16 uses every staging thread, F = 17 is the first width on the
    unfused path (separate input-projection kernel), odd F gives feature rows aligned to 4 bytes only;
  * both recurrent kernels forced at window lengths of 1-4 steps: the two-tile ping-pong kernel stages gi and x up to three
    steps ahead, and the automatic selection never runs it at small batches.

Bar as in tests/test_gpu_parity.py: logits within LOGIT_TOL scaled by the position's largest logit, labels identical
wherever the oracle's top-2 margin exceeds NEAR_TIE.
"""
import numpy as np
import pytest

from oracle import gru_oracle, synth
from tests.test_gpu_parity import LOGIT_TOL, _scaled_err, label_parity

pytestmark = pytest.mark.gpu


def _run(F, B, T, seed, precision="tc", rec="auto"):
    from medaka_b200 import models
    sd = synth.synth_state_dict(seed, num_features=F)
    feats = synth.synth_features(B, T, F, seed=seed + 100)
    ref_probs, ref_logits = gru_oracle.predict_on_batch(gru_oracle.build(sd, num_features=F), feats)
    m = models.GRUModel(num_features=F)
    m.load_state_dict(sd)
    m.set_precision(precision)
    m.set_rec_mode(rec)
    try:
        out = m.forward_arrays(feats, want_logits=True, want_labels=True)
    finally:
        m.close()
    err = _scaled_err(out.logits, ref_logits)
    flips, tie_flips, ties = label_parity(out.labels, ref_probs)
    print("F=%d B=%d T=%d %s/%s: scaled logit err %.3e, label mismatches %d/%d (+%d among %d near-ties)" % (
        F, B, T, precision, rec, err, flips, out.labels.size, tie_flips, ties))
    assert err <= LOGIT_TOL
    assert flips == 0
    assert np.array_equal(out.labels, np.argmax(out.probs, -1))


@pytest.mark.parametrize("precision", ["tc", "fp32"])
@pytest.mark.parametrize("F", [1, 7, 15, 16, 17, 33])
def test_feature_widths(F, precision):
    _run(F, 37, 150, seed=40 + F, precision=precision)


@pytest.mark.parametrize("rec", ["pp", "one"])
@pytest.mark.parametrize("B", [1, 17, 40])
@pytest.mark.parametrize("T", [1, 2, 3, 4])
def test_recurrent_kernels_short_windows(T, B, rec):
    _run(10, B, T, seed=60 + T, rec=rec)
