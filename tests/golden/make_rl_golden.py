"""Golden outputs of the REFERENCE's read-level network (build container only).

Run:  python tests/golden/make_rl_golden.py     (needs /root/reference; writes tests/golden/rl_forward.npz)

Imports medaka.architectures.latent_space_lstm.LatentSpaceLSTM UNMODIFIED (behind the inert stand-ins of make_golden.py
for the absent third-party modules), loads seeded parameters (oracle/rl_oracle.py::synth_rl_state_dict: the state-dict
keys are the reference class's own), puts it in eval mode and records `predict_on_batch`-style outputs for seeded
read-level feature tensors.  The restatement in oracle/rl_oracle.py is asserted against them here.

CASES draw their inputs from rl_oracle.synth_rl_features (trailing empty reads only, like collate padding).  EDGE_CASES
are hand-built from such tensors: empty reads in the middle of a window (reads that do not reach it), reads non-zero in
a single cell, a window with no reads at all (NaN rows for that window only, in the reference as in the oracle), the
encoder's default depth of 100 reads, and feature columns beyond the four the network reads.  Their inputs are stored
next to the outputs (<name>_x).  Regenerating must leave the outputs of the existing cases unchanged; that is asserted.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import make_golden  # noqa: E402
from oracle import rl_oracle  # noqa: E402

CASES = {            # name: (seed, B, P, D, use_dwells, gain)
    "small": (0, 2, 96, 7, False, 1.0),
    "deep": (1, 1, 300, 40, False, 1.0),
    "dwells": (2, 3, 130, 9, True, 1.0),
    "hot": (3, 2, 500, 12, False, 2.5),
}


def _interior_empty(x):
    x[0, :, 0] = 0                      # leading empty read
    x[0, :, 5] = 0                      # reads 4 and 6 share a pair around it
    x[1, :, 4:8] = 0                    # a whole group of 4
    x[1, :, 9] = 0
    x[2, :, 1:3] = 0                    # two in a row: reads 0 and 3 pair up
    x[2, :, 11] = 0                     # last read
    return x


def _one_cell(x):
    P = x.shape[1]
    x[0, :, 2] = 0
    x[0, 0, 2, 0] = 3                   # base only, first position
    x[0, :, 5] = 0
    x[0, P - 1, 5, 1] = 20              # quality only, last position
    x[1, :, 0] = 0
    x[1, 70, 0, 3] = 1                  # mapQ only (not an input of the network, but it makes the read count)
    x[1, :, 7] = 0
    x[1, 127, 7, 2] = 1                 # strand only, last position of a 128-position tile
    return x


def _empty_window(x):
    x[2] = 0
    return x


def _deep100(x):
    x[1, :, 40:60] = 0                  # five empty groups in the middle of the window
    return x


def _extra_channels(x):
    rs = np.random.RandomState(7)
    B, P, D, _ = x.shape
    extra = rs.randint(1, 100, size=(B, P, D, 2)).astype(np.int8)
    extra *= (x != 0).any(-1, keepdims=True)            # extra columns present where the read is
    x = np.concatenate([x, extra], axis=-1)
    x[1, :, 8] = 0
    x[1, 30:60, 8, 5] = 4                # non-zero only in an extra column
    x[2, :, 3] = 0
    x[2, 99, 3, 4] = -1                  # a single cell of an extra column
    return x


EDGE_CASES = {       # name: (seed, B, P, D, use_dwells, gain, empty_rows of the synthetic start, edit)
    "interior_empty": (10, 3, 150, 12, False, 1.0, 0, _interior_empty),
    "one_cell": (11, 2, 140, 8, False, 1.0, 0, _one_cell),
    "empty_window": (12, 4, 160, 6, False, 1.0, 1, _empty_window),
    "deep100": (13, 2, 120, 100, False, 1.0, 3, _deep100),
    "extra_channels": (14, 3, 110, 9, False, 1.0, 1, _extra_channels),
}


def _run(LatentSpaceLSTM, name, seed, x, dw, gain):
    sd = rl_oracle.synth_rl_state_dict(seed, use_dwells=dw, gain=gain)
    ref = LatentSpaceLSTM(use_dwells=dw)
    ref.load_state_dict(sd)
    ref.eval()
    torch.set_num_threads(8)
    with torch.inference_mode():
        probs = ref(torch.from_numpy(x)).numpy()
    mine = rl_oracle.predict(rl_oracle.build(sd, use_dwells=dw), x)
    nan = np.isnan(probs)
    assert np.array_equal(nan, np.isnan(mine)), name
    err = float(np.abs(mine[~nan] - probs[~nan]).max())
    assert err < 2e-6, (name, err)
    print(name, probs.shape, "restatement vs reference %.2e" % err, "mean max prob %.3f" % probs[~nan.any(-1)].max(-1).mean(),
          "nan rows %d" % nan.any(-1).sum())
    return probs


def main():
    make_golden.install_stubs()
    sys.path.insert(0, "/root/reference")
    from medaka.architectures.latent_space_lstm import LatentSpaceLSTM
    path = os.path.join(HERE, "rl_forward.npz")
    old = dict(np.load(path)) if os.path.exists(path) else {}
    out = {}
    for name, (seed, B, P, D, dw, gain) in CASES.items():
        x = rl_oracle.synth_rl_features(B, P, D, use_dwells=dw, seed=100 + seed)
        out[name + "_args"] = np.array([seed, B, P, D, int(dw), gain], dtype=np.float64)
        out[name + "_probs"] = _run(LatentSpaceLSTM, name, seed, x, dw, gain)
    for name, (seed, B, P, D, dw, gain, empty_rows, edit) in EDGE_CASES.items():
        x = edit(rl_oracle.synth_rl_features(B, P, D, use_dwells=dw, seed=100 + seed, empty_rows=empty_rows))
        out[name + "_args"] = np.array([seed, B, P, D, int(dw), gain], dtype=np.float64)
        out[name + "_x"] = x
        out[name + "_probs"] = probs = _run(LatentSpaceLSTM, name, seed, x, dw, gain)
        if name == "empty_window":          # NaN for the window without reads, and only there
            assert np.isnan(probs[2]).all() and np.isfinite(np.delete(probs, 2, 0)).all()
        else:
            assert np.isfinite(probs).all(), name
    for k, v in old.items():                # regenerating keeps every committed entry
        assert k in out and np.array_equal(out[k], v, equal_nan=True), k
    np.savez_compressed(path, **out)


if __name__ == "__main__":
    main()
