"""Read-level consensus network (SURVEY.md 8 row f4, network half): LatentSpaceLSTM.forward
(medaka/architectures/latent_space_lstm.py:154-207).  Goldens = outputs of the reference's own class on seeded parameters
(tests/golden/make_rl_golden.py).  Bar: probabilities within 2e-5 absolute of the reference (fp32 against fp32 in a different
summation order), labels identical wherever the reference's top-2 margin exceeds 1e-4."""
import os

import numpy as np
import pytest

from oracle import rl_oracle

GOLD = os.path.join(os.path.dirname(__file__), "golden", "rl_forward.npz")
TOL = 2e-5


# synthetic inputs (trailing empty reads) and hand-built ones stored with the golden: interior empty reads, single-cell
# reads, a window without reads (NaN rows), 100 reads, extra feature columns (tests/golden/make_rl_golden.py)
SYNTH_CASES = ["small", "deep", "dwells", "hot"]
EDGE_CASES = ["interior_empty", "one_cell", "empty_window", "deep100", "extra_channels"]
# (k = 17 convolution, LSTM recurrences) on the tensor cores (True) or the fp32 CUDA cores (False)
PAIRS = {"tc": (True, True), "fp32": (False, False), "tc_lstm32": (True, False), "fp32_lstmtc": (False, True)}


def _case(g, name):
    seed, B, P, D, dw, gain = g[name + "_args"]
    sd = rl_oracle.synth_rl_state_dict(int(seed), use_dwells=bool(dw), gain=float(gain))
    if name + "_x" in g:
        x = g[name + "_x"]
    else:
        x = rl_oracle.synth_rl_features(int(B), int(P), int(D), use_dwells=bool(dw), seed=100 + int(seed))
    return sd, x, bool(dw), g[name + "_probs"]


@pytest.mark.parametrize("name", SYNTH_CASES + EDGE_CASES)
def test_oracle_matches_reference_class(name):
    g = np.load(GOLD)
    sd, x, dw, want = _case(g, name)
    got = rl_oracle.predict(rl_oracle.build(sd, use_dwells=dw), x)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert nan.any() == (name == "empty_window")
    assert np.abs(got[~nan] - want[~nan]).max() < 2e-6


def _check(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    assert np.abs(got - want).max() < TOL, np.abs(got - want).max()
    top2 = np.sort(want, -1)[..., -2:]
    decided = (top2[..., 1] - top2[..., 0]) > 1e-4
    assert np.array_equal(np.argmax(got, -1)[decided], np.argmax(want, -1)[decided])


def _model(sd, pair, use_dwells=False):
    from medaka_b200 import read_level
    m = read_level.LatentSpaceLSTM(use_dwells=use_dwells)
    m.load_state_dict(sd)
    m.set_conv(*PAIRS[pair])
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("conv", list(PAIRS))
@pytest.mark.parametrize("name", SYNTH_CASES + EDGE_CASES)
def test_device_matches_reference_class(name, conv):
    """Both implementations of the k = 17 convolution (tcgen05 implicit GEMM, fp32 CUDA cores) with both implementations
    of the LSTM recurrence.  A window without reads is NaN exactly where the reference is; the rest holds the usual bar."""
    g = np.load(GOLD)
    sd, x, dw, want = _case(g, name)
    m = _model(sd, conv, dw)
    got = m.forward_arrays(x)
    m.close()
    nan = np.isnan(want).any(-1)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    print("%s/%s: max abs err %.2e" % (name, conv, np.abs(got[~nan] - want[~nan]).max()))
    _check(got[~nan], want[~nan])


@pytest.mark.gpu
@pytest.mark.parametrize("conv", list(PAIRS))
@pytest.mark.parametrize("B,P,D", [(1, 17, 1), (9, 65, 5), (3, 1000, 30), (17, 200, 3), (2, 129, 9),
                                   (3, 1, 4), (4, 8, 2), (2, 16, 8), (3, 127, 4), (2, 128, 8), (2, 256, 2),
                                   (3, 257, 4), (2, 300, 100)])
def test_device_matches_oracle_ragged_shapes(B, P, D, conv):
    """Position counts off the 64- and 128-position convolution tiles and the 16-position pooling tile, windows shorter
    than the convolution's 8-position halo (P = 1), windows off the LSTM tiles, single reads, 100 reads (25 groups of 4),
    windows split over several device calls."""
    sd = rl_oracle.synth_rl_state_dict(5)
    x = rl_oracle.synth_rl_features(B, P, D, seed=B * 1000 + P, empty_rows=min(2, D - 1))
    want = rl_oracle.predict(rl_oracle.build(sd), x)
    m = _model(sd, conv)
    m.max_cells = 40000                      # forces several device calls for the larger shapes
    got = m.forward_arrays(x)
    m.close()
    print("%dx%dx%d/%s: max abs err %.2e" % (B, P, D, conv, np.abs(got - want).max()))
    _check(got, want)


@pytest.mark.gpu
def test_predict_on_batch_interface_and_encoder_check():
    from medaka_b200 import features, read_level, torch_ext
    sd = rl_oracle.synth_rl_state_dict(6)
    m = read_level.LatentSpaceLSTM()
    m.load_state_dict(sd)
    m.check_feature_encoder_compatibility(features.ReadAlignmentFeatureEncoder(include_dwells=False))
    with pytest.raises(ValueError):
        m.check_feature_encoder_compatibility(features.CountsFeatureEncoder())

    class B(object):
        read_level_features = rl_oracle.synth_rl_features(2, 80, 6, seed=3)
    out = m.predict_on_batch(B)
    assert tuple(out.shape) == (2, 80, 5) and abs(float(out.sum(-1).mean()) - 1.0) < 1e-5
    m.close()


def test_collate_pads_read_level_samples():
    """Batch.collate on 3-D features (medaka/torch_ext.py:127-141): zero-padded to the deepest sample, uint8."""
    from medaka_b200 import common, torch_ext
    rs = np.random.RandomState(0)
    feats = [rs.randint(0, 6, size=(50, d, 4)).astype(np.int8) for d in (3, 7, 5)]
    samples = [common.Sample(ref_name="c", features=f, labels=None, ref_seq=None, positions=None, label_probs=None,
                             depth=None) for f in feats]
    b = torch_ext.Batch.collate(samples)
    x = b.read_level_features.numpy()
    assert b.counts_matrix is None and x.shape == (3, 50, 7, 4) and x.dtype == np.uint8
    for i, f in enumerate(feats):
        assert np.array_equal(x[i, :, :f.shape[1]], f.astype(np.uint8)) and not x[i, :, f.shape[1]:].any()
    assert b.features is b.read_level_features


@pytest.mark.gpu
def test_read_level_prediction_end_to_end(tmp_path):
    """BAM file -> native reader -> mdk_read_matrix -> windows -> Batch.collate -> LatentSpaceLSTM engine -> store, against
    the oracles driven over the same reads."""
    from medaka_b200 import common, datastore, features, prediction, read_level
    from oracle import read_matrix_oracle, synth
    from tests import bamutil
    rs = np.random.RandomState(3)
    recs = synth.synth_reads(90, 2600, seed=21, mean_len=700)
    recs.sort(key=lambda r: r["pos"])
    for i, r in enumerate(recs):
        r["query_name"], r["ref"], r["tags"] = "q%d" % i, 0, {}
        r["qual"] = rs.randint(1, 50, len(r["seq"])).tolist()
    path = str(tmp_path / "reads.bam")
    bamutil.write_bam(path, [("ctg", 2600)], recs)
    sd = rl_oracle.synth_rl_state_dict(9)
    model = read_level.LatentSpaceLSTM()
    model.load_state_dict(sd)
    enc = features.ReadAlignmentFeatureEncoder(include_dwells=False)
    region = common.Region("ctg", 0, 2600)
    out = str(tmp_path / "probs.npzstore")
    prediction.predict_regions(out, path, [region], model, enc, chunk_len=500, chunk_ovlp=100, batch_size=3, bam_chunk=100000)
    mat, pos, _, _ = read_matrix_oracle.read_alignment(recs, 0, 2600)
    oracle_model = rl_oracle.build(sd)
    n = 0
    with datastore.DataStore(out, "r") as ds:
        for name in sorted(ds.sample_registry):
            s = ds.load_sample(name)
            a = int(np.flatnonzero((pos["major"] == s.positions["major"][0]) & (pos["minor"] == s.positions["minor"][0]))[0])
            b = a + len(s.positions)
            assert np.array_equal(pos[a:b], s.positions)
            want = rl_oracle.predict(oracle_model, mat[a:b][None].astype(np.int8))[0]
            assert np.abs(s.label_probs - want).max() < TOL
            n += 1
    assert n >= 5
    model.close()
