"""The legacy 802.11b transmit filter (BB11BPMDSpreadFIR4SSE, kernel/bb/dot11b/bbb_fir.c) — the oracle's restatement against what the reference's
own compiled code (oracle/build_ref.sh) made: vectors under golden/fir37 and digests of its output on seeded inputs (golden/ref_digests.json)."""
import os, sys, numpy as np, pytest
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_py
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
H37 = np.array([1, 0, -1, 0, 1, 0, -1, 0, 2, 0, -3, 0, 5, 0, -11, 0, 54, 128, 163, 128, 54, 0, -11, 0, 5, 0, -3, 0, 2, 0, -1, 0, 1, 0, -1, 0, 1])

@pytest.mark.parametrize("name", ["random", "saturating", "dbpsk_chips", "qpsk_chips"])
def test_restatement_reproduces_vectors_made_by_the_reference_code(name):
    x = np.fromfile(os.path.join(GOLD, "fir37", f"fir37_{name}.in.i8"), np.int8).reshape(-1, 2)
    y = np.fromfile(os.path.join(GOLD, "fir37", f"fir37_{name}.out.i8"), np.int8).reshape(-1, 2)
    assert (oracle_py.fir37_legacy(x, 0) == y).all()
    if name == "saturating": assert y.max() == 127 and y.min() == -128        # the vector does reach both rails

def test_restatement_equals_the_compiled_reference_body():
    import golden_vectors as gv
    for key, x in gv.fir37_ref_inputs("cpu"):
        assert gv.fir37_ref_output_equals(key, x, oracle_py.fir37_legacy(x, 0)), key

def test_assembly_variant_is_the_plain_filter():
    """variant 1 (FIR37SSE_INLINE): y[n] = sat8((sum_k h[k] x[n + 8 - k]) >> 8) wherever the 16-bit lane tree does not saturate."""
    rng = np.random.default_rng(6)
    x = rng.integers(-40, 41, (4096, 2)).astype(np.int8)
    y = oracle_py.fir37_legacy(x, 1).astype(int)
    xp = np.concatenate([x.astype(int), np.zeros((64, 2), int)])
    xp[:8] = 0                                                                  # the first eight inputs never enter
    for c in range(2):
        full = np.convolve(xp[:, c], H37)
        want = np.clip(full[8:8 + len(x)] >> 8, -128, 127)
        assert (y[:, c] == want).all()
    # ... and the intrinsic variant differs from it only by what the +-1 outer taps can do
    d = np.abs(oracle_py.fir37_legacy(x, 0).astype(int) - y)
    assert d.max() <= 1 and d.any()

def _chips_of_capture(name):
    y = np.fromfile(os.path.join(GOLD, name), np.int8).reshape(-1, 2).astype(int)
    n = (len(y) - 30) // 4
    # the only odd-index taps are the two 128s next to the centre: sample 25 + 4k is chip k alone (63 / -64)
    re, im = y[25:25 + 4 * n:4, 0], y[25:25 + 4 * n:4, 1]
    chips = np.zeros((16 + 4 * n + 64, 2), np.int8)
    chips[16:16 + 4 * n:4, 0] = np.where(re > 32, 127, np.where(re < -32, -128, 0)); chips[16:16 + 4 * n:4, 1] = np.where(im > 32, 127, np.where(im < -32, -128, 0))
    return y, chips[: len(chips) // 8 * 8]

@pytest.mark.parametrize("name", ["1long44.mf.bin", "2long44.mf.bin"])
def test_reference_sample_files_were_shaped_by_a_close_relative_of_this_filter(name):
    """kernel/HWTest/exe/tx samples/*.mf.bin: chips read off the file, through the restated filter -> within 3 LSB (1 Mbps; 4 LSB at 2 Mbps, whose chip
    levels the file does not let one read exactly) of the file everywhere, 60 % / 40 % of the samples exact.  (A least-squares fit of the taps from the file gives non-integer outer taps and a ripple longer than 37 taps, so the
    files were not made by bbb_fir.c as it stands; this is evidence of kinship, not a pin.  The pin is the reference's compiled filter body.)"""
    y, chips = _chips_of_capture(name)
    out = oracle_py.fir37_legacy(chips, 0).astype(int)
    m = min(len(out), len(y)) - 64
    d = np.abs(out[32:m] - y[32:m])
    assert d.max() <= (3 if name.startswith("1") else 4), d.max()
    assert (d == 0).all(axis=1).mean() > (0.6 if name.startswith("1") else 0.4)
