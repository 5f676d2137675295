"""GPU parity tests for the legacy 802.11b transmit filter (pytest -m gpu): sb200_tx11b_fir37 and the BB11BPMDSpreadFIR4SSE / ...ASM entry
points against oracle/tx11b_legacy.cpp and against what the reference's own compiled code made: the vectors under tests/golden/fir37 and
digests of its output on seeded inputs (tests/golden/ref_digests.json)."""
import os, ctypes as C, numpy as np, pytest
import oracle_py
from sora_b200 import api

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

@pytest.fixture(scope="module")
def eng():
    return api.Engine(0)

@pytest.mark.parametrize("name", ["random", "saturating", "dbpsk_chips", "qpsk_chips"])
def test_device_reproduces_vectors_made_by_the_reference_code(eng, name):
    x = np.fromfile(os.path.join(GOLD, "fir37", f"fir37_{name}.in.i8"), np.int8).reshape(-1, 2)
    y = np.fromfile(os.path.join(GOLD, "fir37", f"fir37_{name}.out.i8"), np.int8).reshape(-1, 2)
    assert (eng.tx11b_fir37(x, 0) == y).all()

@pytest.mark.parametrize("variant", [0, 1])
def test_device_matches_oracle_on_ragged_batches(eng, variant):
    rng = np.random.default_rng(70 + variant)
    F, L = 37, 4096
    x = rng.integers(-128, 128, (F, L, 2)).astype(np.int8)
    x[3] = 127; x[4] = -128; x[5] = np.where(rng.integers(0, 2, (L, 2)) > 0, 127, -128)       # the rails of the 16-bit lane tree
    lens = (rng.integers(0, L // 8 + 1, F) * 8).astype(np.uint32); lens[0] = 0; lens[1] = 8; lens[2] = L; lens[3:6] = L
    off = np.arange(F, dtype=np.uint64) * L
    out = np.full_like(x, 99)
    eng.tx11b_fir37_raw(x.ctypes.data, F * L, off.ctypes.data, lens.ctypes.data, F, variant, out.ctypes.data)
    for f in range(F):
        n = int(lens[f])
        assert (out[f, :n] == oracle_py.fir37_legacy(x[f, :n], variant)).all(), (f, n)
        assert (out[f, n:] == 99).all()                                                          # nothing outside a frame's own range is touched

def test_device_equals_the_compiled_reference_body(eng):
    import golden_vectors as gv
    for key, x in gv.fir37_ref_inputs("gpu"):
        assert gv.fir37_ref_output_equals(key, x, eng.tx11b_fir37(x, 0)), key

def test_legacy_entry_points_and_errors(eng):
    lib = api.load_library()
    rng = np.random.default_rng(10)
    x = rng.integers(-128, 128, (1024, 2)).astype(np.int8); y = np.zeros_like(x); n = C.c_uint32(0)
    for fn, variant in ((lib.BB11BPMDSpreadFIR4SSE, 0), (lib.BB11BPMDSpreadFIR4ASM, 1)):
        fn.restype = C.c_int32
        assert fn(C.c_void_p(x.ctypes.data), C.c_uint32(len(x)), C.c_void_p(y.ctypes.data), C.byref(n)) == 0 and n.value == len(x)
        assert (y == oracle_py.fir37_legacy(x, variant)).all()
        assert fn(C.c_void_p(x.ctypes.data), C.c_uint32(1020), C.c_void_p(y.ctypes.data), C.byref(n)) == C.c_int32(0x80004005).value     # uiInputSize & 7 -> E_FAIL (bbb_fir.c:100-103)
    off = np.zeros(1, np.uint64); ln = np.array([12], np.uint32)
    with pytest.raises(api.Sb200Error): eng.tx11b_fir37_raw(x.ctypes.data, 1024, off.ctypes.data, ln.ctypes.data, 1, 0, y.ctypes.data)
    ln[0] = 2048
    with pytest.raises(api.Sb200Error): eng.tx11b_fir37_raw(x.ctypes.data, 1024, off.ctypes.data, ln.ctypes.data, 1, 0, y.ctypes.data)
    ln[0] = 64
    with pytest.raises(api.Sb200Error): eng.tx11b_fir37_raw(x.ctypes.data, 1024, off.ctypes.data, ln.ctypes.data, 1, 2, y.ctypes.data)

def test_filtered_chips_of_the_reference_capture_decode_on_the_device(eng):
    """Chips read off kernel/HWTest/exe/tx samples/1long44.mf.bin -> the device filter -> the device 802.11b receiver returns frame.txt's bytes."""
    import test_cpu_oracle_tx11b_legacy as t
    frame = np.array([int(x, 16) for x in open(os.path.join(GOLD, "frame.txt")).read().split()], np.uint8)
    _, chips = t._chips_of_capture("1long44.mf.bin")
    w = eng.tx11b_fir37(chips, 0)
    iq = w.astype(np.int16) << 8
    iq = np.ascontiguousarray(np.concatenate([np.zeros((280, 2), np.int16), iq, np.zeros(((-len(iq)) % 28 + 56, 2), np.int16)]))
    res, out = eng.rx11b_batch(iq, np.zeros(1, np.uint64), np.array([len(iq)], np.uint32))
    ores, oout = oracle_py.rx11b_batch(iq, np.zeros(1, np.uint64), np.array([len(iq)], np.uint32))
    assert res[0]["status"] == 1 and res[0]["rate_kbps"] == 1000 and res[0]["length"] == 114 and (out[0, :113] == frame[:113]).all()
    assert ores[0]["status"] == 1 and (oout[0, :113] == frame[:113]).all()
