"""Variant decoding (SURVEY.md section 8 row f2): oracle vs the reference's own results (CPU), CUDA path vs both (GPU).

Goldens: tests/golden/variants.npz, written by tests/golden/make_variant_golden.py from the UNMODIFIED
medaka.labels.HaploidLabelScheme.decode_variants / medaka.variant.join_samples (with variant_columns compiled from the
reference's src/medaka_rnn_variants.c), plus the reference's literal cases (medaka/test/test_labels.py:279-399).
"""
import json
import os

import numpy as np
import pytest

from oracle import labels_oracle, synth, variants_oracle as vo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (ref with gaps, call with gaps, slice, pos, ref, alt): medaka/test/test_labels.py:279-366
LITERAL_CASES = [
    ('CATG', 'TATG', slice(None, None), 0, 'C', 'T'),
    ('CAT*G', 'CA*CG', slice(None, None), 2, 'T', 'C'),
    ('CAT*G', 'CA*TG', slice(None, None), None, None, None),
    ('CATG', 'CTGG', slice(None, None), 1, 'AT', 'TG'),
    ('C*ATG', 'CGATG', slice(None, None), 0, 'C', 'CG'),
    ('CATG**', 'CATGGT', slice(None, None), 3, 'G', 'GGT'),
    ('CATG', '*ATG', slice(None, None), 0, 'CA', 'A'),
    ('CATG', 'CAT*', slice(None, None), 2, 'TG', 'T'),
    ('CATG', '**TG', slice(None, None), 0, 'CAT', 'T'),
    ('CATG', 'CA**', slice(None, None), 1, 'ATG', 'A'),
    ('CA*TG', 'CGCTG', slice(None, None), 1, 'A', 'GC'),
    ('CATG', 'CG*G', slice(None, None), 1, 'AT', 'G'),
    ('CA*TG', 'CGC*G', slice(None, None), 1, 'AT', 'GC'),
    ('TCATG', 'T*ATG', slice(1, None), 0, 'TC', 'T'),
    ('TCATG', 'T*ATG', slice(None, None), 0, 'TC', 'T'),
    ('TCATG', 'T*ATG', slice(2, None), None, None, None),
]


def literal_sample(ref, call, pri_prob=0.9):
    """haploid_sample_from_labels (medaka/test/test_labels.py:34-75) with sec=None, sec_prob=0."""
    major, minor, m = [], [], -1
    for c in ref:
        if c == '*':
            minor.append(minor[-1] + 1)
        else:
            m += 1
            minor.append(0)
        major.append(m)
    pos = np.empty(len(ref), dtype=[('major', int), ('minor', int)])
    pos['major'], pos['minor'] = major, minor
    probs = np.zeros((len(ref), 5))
    for i, l in enumerate(call):
        probs[i, vo.ENC[l]] = pri_prob
        others = np.where(probs[i] == 0)[0]
        other = vo.ENC[ref[i]] if vo.ENC[ref[i]] in others else others[0]
        probs[i, other] = 1 - np.sum(probs[i])
    return pos, probs, ref.replace('*', '')


def golden():
    g = np.load(os.path.join(ROOT, "tests", "golden", "variants.npz"))
    return {k: json.loads(str(g[k])) for k in g.files if k != "meta"}


def same_records(got, exp, qual_tol=2e-3):
    assert len(got) == len(exp), (len(got), len(exp))
    for a, b in zip(got, exp):
        assert (a['pos'], a['ref'], a['alt']) == (b['pos'], b['ref'], b['alt'][0]), (a, b)
        assert abs(a['qual'] - b['qual']) <= qual_tol, (a, b)


# ------------------------------------------------------------------------------------------------ oracle (CPU)
def test_oracle_matches_reference_golden():
    for name, rec in golden().items():
        if name.startswith("join"):
            continue
        d = synth.synth_variant_pileup(**rec['kwargs'])
        for ambig in (0, 1):
            got = vo.decode_variants(d['positions'], d['label_probs'], d['ref_seq'], ambig_ref=bool(ambig))
            same_records(got, rec['ambig%d' % ambig])
            assert [g_['gq'] for g_ in got] == [e['gq'] for e in rec['ambig%d' % ambig]]


def test_oracle_reference_literals():
    pri = vo.phred(1 - 0.9) - vo.phred(0.9)
    for ref, call, sl, pos, vref, valt in LITERAL_CASES:
        p, probs, ref_seq = literal_sample(ref, call)
        got = vo.decode_variants(p[sl], probs[sl], ref_seq)
        if pos is None:
            assert got == []
            continue
        v = got[0]
        assert (v['pos'], v['ref'], v['alt']) == (pos, vref, valt), (ref, call, v)
        a, b = v['run']
        n_diff = sum(x != y for x, y in zip(ref[sl][a:b], call[sl][a:b]))
        assert abs(v['qual'] - n_diff * pri) < 2e-3


def test_oracle_join_matches_reference_golden():
    for name, rec in golden().items():
        if not name.startswith("join"):
            continue
        d = synth.synth_variant_pileup(**rec['kwargs'])
        n = len(d['positions'])
        step = rec['chunk_len'] - rec['overlap']
        ranges = [(lo, lo + rec['chunk_len']) for lo in range(0, n - rec['chunk_len'] + 1, step)]
        if not ranges or ranges[-1][1] < n:
            ranges.append((max(0, n - rec['chunk_len']), n))
        # trimmed views: identical columns across overlaps -> cut at the overlap mid-point (common.py:376-382)
        cuts = [0]
        for (a0, b0), (a1, b1) in zip(ranges[:-1], ranges[1:]):
            ov = b0 - a1
            cuts.append(a1 + ov // 2)
        cuts.append(n)
        pieces = [(d['positions'][a:b], d['label_probs'][a:b], i == len(cuts) - 2)
                  for i, (a, b) in enumerate(zip(cuts[:-1], cuts[1:]))]
        joined = vo.join_cuts(pieces, d['ref_seq'])
        sizes = [sum(hi - lo for _, lo, hi in j) for j in joined]
        assert sizes == [sz for _, sz in rec['joined']]
        offs = np.cumsum([0] + sizes)
        got = []
        for a, b in zip(offs[:-1], offs[1:]):
            got.extend(vo.decode_variants(d['positions'][a:b], d['label_probs'][a:b], d['ref_seq']))
        same_records(got, rec['variants'])
        assert rec['same_as_whole']


def test_reference_c_variant_columns_matches_oracle():
    """The verdicts of the reference's own src/medaka_rnn_variants.c on 20 seeded pileups, recorded in
    tests/golden/variant_columns.npz by tests/golden/make_variant_columns_golden.py."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "variant_columns.npz"))
    offs = np.concatenate(([0], np.cumsum(g["lengths"])))
    assert len(g["lengths"]) == 20
    for a, b in zip(offs[:-1], offs[1:]):
        minor = g["minor"][a:b].astype(np.int64)
        ref, pred = g["reference"][a:b].astype(np.int64), g["prediction"][a:b].astype(np.int64)
        assert np.array_equal(labels_oracle.variant_columns(minor, ref, pred), g["is_var"][a:b])


# ------------------------------------------------------------------------------------------------ CUDA path (GPU)
def _records(variants):
    return [dict(pos=v.pos, ref=v.ref, alt=v.alt[0], qual=v.qual, gq=v.genotype_data['GQ']) for v in variants]


@pytest.mark.gpu
def test_gpu_decode_variants_matches_reference_golden():
    from medaka_b200 import common, labels
    ls = labels.HaploidLabelScheme()
    for name, rec in golden().items():
        if name.startswith("join"):
            continue
        d = synth.synth_variant_pileup(**rec['kwargs'])
        s = common.Sample(d['ref_name'], None, None, None, d['positions'], d['label_probs'], None)
        for ambig in (0, 1):
            got = _records(ls.decode_variants(s, d['ref_seq'], ambig_ref=bool(ambig)))
            same_records(got, rec['ambig%d' % ambig])
        allv = ls.decode_variants(s, d['ref_seq'], return_all=True)
        assert len(allv) == rec['return_all_n']
        for v, e in zip(allv[:400], rec['return_all_head']):
            assert (v.pos, v.ref, v.alt, v.genotype_data['GT']) == (e['pos'], e['ref'], e['alt'], e['gt'])
            assert abs(v.qual - e['qual']) <= 2e-3
        # integer outputs against the oracle: labels, variant columns, run boundaries
        is_major = d['positions']['minor'] == 0
        codes = np.zeros(len(is_major), dtype=np.uint8)
        codes[is_major] = ls.encode_reference(d['ref_seq'], d['positions']['major'][is_major])
        arr = labels.decode_variant_arrays(d['label_probs'], d['positions']['minor'], codes)
        assert np.array_equal(arr['pred'], np.argmax(d['label_probs'], -1))
        exp_var = labels_oracle.variant_columns(d['positions']['minor'], codes, arr['pred'])
        assert np.array_equal(arr['is_var'], exp_var)
        edges = np.flatnonzero(np.diff(np.concatenate(([0], exp_var.astype(np.int8), [0]))))
        assert np.array_equal(arr['run_start'], edges[0::2]) and np.array_equal(arr['run_len'], edges[1::2] - edges[0::2])
        # per-run sums are the left-to-right float32 sums of the per-column qualities
        for a, n_, sp, sr in zip(arr['run_start'], arr['run_len'], arr['run_pred_q'], arr['run_ref_q']):
            acc_p = acc_r = np.float32(0)
            for k in range(int(a), int(a + n_)):
                acc_p, acc_r = acc_p + arr['pred_q'][k], acc_r + arr['ref_q'][k]
            assert acc_p == sp and acc_r == sr


@pytest.mark.gpu
def test_gpu_decode_variants_reference_literals():
    from medaka_b200 import common, labels
    ls = labels.HaploidLabelScheme()
    pri = float(vo.phred(1 - 0.9) - vo.phred(0.9))
    for ref, call, sl, pos, vref, valt in LITERAL_CASES:
        p, probs, ref_seq = literal_sample(ref, call)
        s = common.Sample('contig1', None, None, None, p, probs, None).slice(sl)
        ls.verbose = True
        v = ls.decode_variants(s, ref_seq)
        if pos is None:
            assert len(v) == 0
            continue
        v = v[0]
        n_diff = sum(a != b for a, b in zip(v.info['pred_seq'], v.info['ref_seq']))
        assert (v.chrom, v.pos, v.ref, v.alt, v.genotype_data['GT']) == ('contig1', pos, vref, [valt], '1')
        assert abs(float(v.qual) - n_diff * pri) < 2e-3
        assert int(v.genotype_data['GQ']) == round(n_diff * pri)
    with pytest.raises(ValueError):
        p, probs, ref_seq = literal_sample('C*ATG', 'CGATG')
        ls.decode_variants(common.Sample('c', None, None, None, p[1:], probs[1:], None), ref_seq)


@pytest.mark.gpu
def test_gpu_join_samples_matches_reference_golden():
    from medaka_b200 import common, labels, variant
    ls = labels.HaploidLabelScheme()
    for name, rec in golden().items():
        if not name.startswith("join"):
            continue
        d = synth.synth_variant_pileup(**rec['kwargs'])
        n = len(d['positions'])
        step = rec['chunk_len'] - rec['overlap']
        ranges = [(lo, lo + rec['chunk_len']) for lo in range(0, n - rec['chunk_len'] + 1, step)]
        if not ranges or ranges[-1][1] < n:
            ranges.append((max(0, n - rec['chunk_len']), n))
        samples = [common.Sample(d['ref_name'], None, None, None, d['positions'][a:b], d['label_probs'][a:b], None)
                   for a, b in ranges]
        joined = list(variant.join_samples(variant.trimmed_samples(samples), d['ref_seq'], ls))
        assert [[s.name, s.size] for s in joined] == rec['joined']
        got = _records(variant.variants_from_samples(samples, d['ref_seq'], ls))
        same_records(got, rec['variants'])


@pytest.mark.gpu
def test_gpu_decode_variants_large_matches_oracle():
    """Config-4 scale (one 0.7 M-column joined sample): the records equal the oracle's; every reported variant changes
    the draft; the runs partition exactly the variant columns."""
    from medaka_b200 import common, labels
    d = synth.synth_variant_pileup(seed=77, n_major=600000, p_mut=0.01, n_frac=0.001)
    ls = labels.HaploidLabelScheme()
    s = common.Sample(d['ref_name'], None, None, None, d['positions'], d['label_probs'], None)
    vs = ls.decode_variants(s, d['ref_seq'])
    assert len(vs) > 1000 and all(v.ref != v.alt[0] for v in vs)
    exp = vo.decode_variants(d['positions'], d['label_probs'], d['ref_seq'])
    same_records(_records(vs), [dict(e, alt=[e['alt']]) for e in exp])
    is_major = d['positions']['minor'] == 0
    codes = np.zeros(len(is_major), dtype=np.uint8)
    codes[is_major] = ls.encode_reference(d['ref_seq'], d['positions']['major'][is_major])
    arr = labels.decode_variant_arrays(d['label_probs'], d['positions']['minor'], codes)
    assert int(arr['run_len'].sum()) == int(arr['is_var'].sum())
    assert np.all(arr['run_start'][1:] > arr['run_start'][:-1] + arr['run_len'][:-1])   # runs are separated
