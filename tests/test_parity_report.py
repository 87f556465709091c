"""Parity report (GPU): prints a JSON report (`pytest -s` shows it; profiles/parity_r02.json is one such report)
- for every case the scaled and element-wise logit error of the CUDA path against the fp32 CPU reference,
the number of positions whose reference top-2 probability margin is below 1e-5 ("near ties"), the label flips among
the decided and the near-tie positions, and the same two flip counts for the CPU reference against ITSELF run with a
different thread count (8 vs 1): the reference's own argmax is not stable inside that margin, which is why label
identity is asserted outside it and only counted inside it.

Cases: the six reference-generated goldens (tests/golden/gru_forward.npz, incl. the adversarial near-tie head); one
full reference batch 200 x 10000 (medaka/medaka.py:266-272 default) against the oracle; the benched 1111 x 10000 grid
(ping-pong kernels, fused head, coalesced from 200-window submits) on 16 sampled windows; F = 20 features normalised
`fwd_rev` on the device; the one-tile kernels forced beyond a wave (two tiles per CTA, old path).
"""
import json
import os

import numpy as np
import pytest

from oracle import features_oracle, gru_oracle, synth

pytestmark = pytest.mark.gpu
NEAR_TIE = 1e-5
LOGIT_TOL = 1e-3


def _entry(logits, labels, ref_logits, ref_probs):
    scale = np.abs(ref_logits).max(-1, keepdims=True)
    d = np.abs(logits - ref_logits)
    top2 = np.sort(ref_probs, -1)[..., -2:]
    near = (top2[..., 1] - top2[..., 0]) <= NEAR_TIE
    mism = labels != np.argmax(ref_probs, -1)
    return {"positions": int(labels.size), "scaled_logit_err": float((d / scale).max()),
            "elementwise_rel_err": float((d / np.maximum(np.abs(ref_logits), 1e-30)).max()),
            "near_ties": int(near.sum()), "flips_decided": int((mism & ~near).sum()),
            "flips_near_tie": int((mism & near).sum())}


def _cpu_self_check(sd, feats, F, ref_probs_8):
    """torch CPU, 1 thread against the 8-thread result: flips among decided / near-tie positions."""
    import torch
    m = gru_oracle.build(sd, num_features=F)
    p1, _ = gru_oracle.predict_on_batch(m, feats, threads=1)
    torch.set_num_threads(8)
    top2 = np.sort(ref_probs_8, -1)[..., -2:]
    near = (top2[..., 1] - top2[..., 0]) <= NEAR_TIE
    mism = np.argmax(p1, -1) != np.argmax(ref_probs_8, -1)
    return {"cpu_1_vs_8_threads_flips_decided": int((mism & ~near).sum()),
            "cpu_1_vs_8_threads_flips_near_tie": int((mism & near).sum()),
            "cpu_1_vs_8_threads_max_prob_diff": float(np.abs(p1 - ref_probs_8).max())}


def test_parity_report(golden_dir):
    import torch
    from medaka_b200 import common, features, models
    report = {"near_tie_margin": NEAR_TIE, "logit_tolerance_scaled": LOGIT_TOL, "torch": torch.__version__, "cases": {}}
    cases = report["cases"]
    g = np.load(os.path.join(golden_dir, "gru_forward.npz"))

    def run(sd, feats, F, mode="auto", precision="tc"):
        m = models.GRUModel(num_features=F)
        m.load_state_dict(sd)
        m.set_precision(precision)
        m.set_rec_mode(mode)
        out = m.forward_arrays(feats, want_logits=True, want_labels=True)
        m.close()
        return out

    # ---- reference-generated goldens (the real GRUModel + TorchModel.predict_on_batch, 8 threads)
    for case in ("small", "long", "hot", "f20", "b1", "neartie"):
        seed, B, T, F, head_gain, rec_gain = g[case + "_args"]
        maker = synth.synth_state_dict_neartie if case == "neartie" else synth.synth_state_dict
        sd = maker(int(seed), num_features=int(F), head_gain=head_gain, rec_gain=rec_gain)
        feats = synth.synth_features(int(B), int(T), int(F), seed=100 + int(seed))
        for mode in ("one", "pp"):
            out = run(sd, feats, int(F), mode)
            e = _entry(out.logits, out.labels, g[case + "_logits"], g[case + "_probs"])
            e.update(_cpu_self_check(sd, feats, int(F), g[case + "_probs"]))
            e["source"] = "reference golden (tests/golden/gru_forward.npz)"
            cases["%s/%s" % (case, mode)] = e
            assert e["scaled_logit_err"] <= LOGIT_TOL and e["flips_decided"] == 0, (case, mode, e)

    # ---- one full reference batch: 200 windows x 10000 columns (about a minute of CPU)
    sd = synth.synth_state_dict(0)
    torch.set_num_threads(8)
    feats = synth.synth_features_fast(200, 10000, 10, seed=11)
    ref_probs, ref_logits = gru_oracle.predict_on_batch(gru_oracle.build(sd), feats)
    for mode in ("one", "pp"):
        out = run(sd, feats, 10, mode)
        e = _entry(out.logits, out.labels, ref_logits, ref_probs)
        e["source"] = "oracle (torch fp32 nn.GRU, 8 threads)"
        cases["batch_200x10000/%s" % mode] = e
        assert e["scaled_logit_err"] <= LOGIT_TOL and e["flips_decided"] == 0, (mode, e)

    # ---- the benched grid: 1111 x 10000 through 200-window submits (coalesced, ping-pong, fused head), 16 windows checked
    feats = synth.synth_features_fast(1111, 10000, 10, seed=12)
    pick = np.linspace(0, 1110, 16).astype(int)
    ref_probs, ref_logits = gru_oracle.predict_on_batch(gru_oracle.build(sd), feats[pick])
    m = models.GRUModel(num_features=10)
    m.load_state_dict(sd)
    m.reserve(m.preferred_batch_size(), 10000)
    tickets, outs = [], []
    for i, a in enumerate(range(0, 1111, 200)):
        x = m.pinned("pin%d" % i, feats[a:a + 200].shape, np.float32)
        np.copyto(x, feats[a:a + 200])
        p = m.pinned("pp%d" % i, x.shape[:2] + (5,), np.float32)
        lg = m.pinned("pl%d" % i, x.shape[:2] + (5,), np.float32)
        lb = m.pinned("pb%d" % i, x.shape[:2], np.uint8)
        tickets.append(m.submit_arrays(x, p, lb, lg))
        outs.append((p, lg, lb))
    for t in tickets:
        m.wait(t)
    logits = np.concatenate([o[1] for o in outs])[pick]
    labels = np.concatenate([o[2] for o in outs])[pick]
    m.close()
    e = _entry(logits, labels, ref_logits, ref_probs)
    e["source"] = "oracle on 16 of 1111 windows; engine fed with 200-window submits"
    cases["grid_1111x10000_coalesced/auto"] = e
    assert e["scaled_logit_err"] <= LOGIT_TOL and e["flips_decided"] == 0, e

    # ---- F = 20, counts normalised 'fwd_rev' on the device, then the forward
    counts, pos = synth.synth_counts(60 * 500, seed=5, num_dtypes=2)
    enc = features.CountsFeatureEncoder(normalise="fwd_rev", dtypes=("r9", "r10"))
    s = enc._post_process_pileup(counts, pos, common.Region("ref", int(pos["major"][0]), int(pos["major"][-1]) + 1))
    exp_f, _ = features_oracle.post_process_pileup(counts.copy(), pos, "fwd_rev", ("r9", "r10"))
    assert np.array_equal(s.features, exp_f)
    feats = s.features.reshape(60, 500, 20)
    sd20 = synth.synth_state_dict(3, num_features=20)
    ref_probs, ref_logits = gru_oracle.predict_on_batch(gru_oracle.build(sd20, num_features=20), feats)
    for mode in ("one", "pp"):
        out = run(sd20, feats, 20, mode)
        e = _entry(out.logits, out.labels, ref_logits, ref_probs)
        e["source"] = "oracle; features from the GPU normalise kernel (bit-exact against its oracle)"
        cases["f20_fwd_rev_60x500/%s" % mode] = e
        assert e["scaled_logit_err"] <= LOGIT_TOL and e["flips_decided"] == 0, (mode, e)

    # ---- one-tile kernels beyond a wave (two tiles per CTA on the round-1 path)
    feats = synth.synth_features(1217, 33, 10, seed=13)
    ref_probs, ref_logits = gru_oracle.predict_on_batch(gru_oracle.build(sd), feats)
    out = run(sd, feats, 10, "one")
    e = _entry(out.logits, out.labels, ref_logits, ref_probs)
    e["source"] = "oracle"
    cases["1217x33_two_tiles_round1_kernel/one"] = e
    assert e["scaled_logit_err"] <= LOGIT_TOL and e["flips_decided"] == 0, e

    report["summary"] = {
        "max_scaled_logit_err": max(c["scaled_logit_err"] for c in cases.values()),
        "flips_decided_total": sum(c["flips_decided"] for c in cases.values()),
        "near_ties_total": sum(c["near_ties"] for c in cases.values()),
        "flips_near_tie_total": sum(c["flips_near_tie"] for c in cases.values()),
        "cpu_self_flips_near_tie_total": sum(c.get("cpu_1_vs_8_threads_flips_near_tie", 0) for c in cases.values()),
        "cpu_self_flips_decided_total": sum(c.get("cpu_1_vs_8_threads_flips_decided", 0) for c in cases.values()),
    }
    print(json.dumps(report, indent=1, sort_keys=True))
