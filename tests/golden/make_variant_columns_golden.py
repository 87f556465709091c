"""Record the reference's own variant_columns() on seeded random pileups (needs `make -C oracle`).

oracle/_ref/libmedaka_rnn_variants.so is the reference's src/medaka_rnn_variants.c compiled by oracle/Makefile; it is
called through ctypes on 20 seeded column sequences (insertion columns, reference and predicted labels) and its
per-column verdicts are stored next to the inputs in tests/golden/variant_columns.npz, so that
tests/test_variants.py can hold the oracle to the reference's C without building it.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def trials(seed=9, n_trials=20):
    """(minor, reference, prediction) per trial: ~30 % insertion columns, ~15 % of the predictions differ."""
    rs = np.random.RandomState(seed)
    for _ in range(n_trials):
        n = int(rs.randint(1, 3000))
        is_minor = rs.uniform(size=n) < 0.3
        is_minor[0] = False
        idx = np.arange(n)
        last_major = np.maximum.accumulate(np.where(~is_minor, idx, -1))
        minor = idx - last_major
        ref = rs.randint(0, 5, n)
        pred = np.where(rs.uniform(size=n) < 0.85, ref, rs.randint(0, 5, n))
        yield minor, ref, pred


def main():
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libmedaka_rnn_variants.so"))
    lib.variant_columns.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_size_t]
    lib.variant_columns.restype = None
    cols = {"minor": [], "reference": [], "prediction": [], "is_var": []}
    lengths = []
    for minor, ref, pred in trials():
        n = len(minor)
        m = np.ascontiguousarray(minor, dtype=np.uintp)
        r32, p32 = np.ascontiguousarray(ref, dtype=np.int32), np.ascontiguousarray(pred, dtype=np.int32)   # wchar_t
        out = np.zeros(n, dtype=np.bool_)
        lib.variant_columns(m.ctypes.data, r32.ctypes.data, p32.ctypes.data, out.ctypes.data, n)
        lengths.append(n)
        cols["minor"].append(minor.astype(np.int32))
        cols["reference"].append(ref.astype(np.uint8))
        cols["prediction"].append(pred.astype(np.uint8))
        cols["is_var"].append(out)
    arrays = {k: np.concatenate(v) for k, v in cols.items()}
    np.savez_compressed(os.path.join(HERE, "variant_columns.npz"), lengths=np.array(lengths, dtype=np.int32), **arrays)
    print("trials", len(lengths), "columns", sum(lengths), "variant columns", int(arrays["is_var"].sum()))


if __name__ == "__main__":
    main()
