"""CPU tests of the 802.11a transmit restatement (oracle/tx11a.cpp): fixed-point TX -> fixed-point RX round trip at all 8 rates
(SURVEY.md §8c item 4), IFFT<128> sanity, tables against the reference, and how close it comes to usr/HwVeri/data/ofdm.bin."""
import os, sys, zlib, numpy as np, pytest
import oracle_py
from sora_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

def _rx(samples8, lead=400, trail=400):
    iq = np.concatenate([np.zeros((lead, 2), np.int16), samples8.astype(np.int16) << 8, np.zeros((trail, 2), np.int16)])   # ConvertModFile2DumpFile_8b
    return oracle_py.rx11a_run(iq)

@pytest.mark.parametrize("rate", sorted(synth.RATES))
def test_tx_oracle_to_rx_oracle_roundtrip(rate):
    rng = np.random.default_rng(rate)
    for L in (1, 37, 200, 1496, 2496):
        payload = rng.integers(0, 256, L).astype(np.uint8)
        for seed in (0xFF, 0x5B):
            td = oracle_py.tx11a_modulate(payload, rate, seed)
            res, out = _rx(td)
            assert len(res) == 1 and res[0]["status"] == 1 and res[0]["rate_kbps"] == rate and res[0]["length"] == L + 4, (rate, L, res)
            assert (out[0, :L] == payload).all() and int.from_bytes(bytes(out[0, L:L + 4]), "little") == zlib.crc32(payload.tobytes())

def test_ifft128_close_to_float():
    rng = np.random.default_rng(0)
    x = np.zeros((128, 2), np.int16); idx = np.r_[1:27, 102:128]; x[idx] = rng.integers(-10720, 10720, (52, 2))
    got = oracle_py.ifft128(x).astype(np.float64)
    want = np.fft.ifft(x[:, 0] + 1j * x[:, 1]) * 128 / 2 ** 7        # 3 radix stages with >> 2 each and the 8-point stage with >> 3 ... net 1/128 ... checked by scale fit below
    g = got[:, 0] + 1j * got[:, 1]
    k = np.vdot(want, g) / np.vdot(want, want)
    assert abs(abs(k) - 1) < 0.02 and abs(np.angle(k)) < 0.01 and np.abs(g - k * want).max() < 12

def test_near_match_with_reference_modulator_output():
    """ofdm.bin was made by the reference's *legacy* transmitter (different window, IFFT rounding differs by one LSB here and
    there): not a pin for the brick restatement, but the two must agree on every sample away from the symbol edges to +-1."""
    gold = np.fromfile(os.path.join(ROOT, "tests", "golden", "ofdm.bin"), dtype=np.int8).reshape(-1, 2).astype(np.int32)
    mine = oracle_py.tx11a_modulate(np.full(200, 0x31, np.uint8), 24000, 0xFF, 32).astype(np.int32)
    assert mine.shape == gold.shape
    pos = np.arange(len(gold)); edge = np.zeros(len(gold), bool)
    for b in [0, 320] + list(range(640, len(gold), 160)):
        edge |= (pos >= b - 3) & (pos < b + 8)
    inner = ~edge
    assert np.abs(mine[inner] - gold[inner]).max() <= 1
    assert (mine == gold).all(1).mean() > 0.93

def test_tx_tables_vs_reference():
    """The transmit FFT tables against the reference headers' (golden/ref_digests.json)."""
    import refcheck as rc, golden_vectors as gv
    for N in (128, 32):
        for M in (1, 2, 3):
            assert gv.ref_table_equals(f"twiddle_{N}_{M}", rc.gen_twiddle(N, M)), (N, M)
    assert gv.ref_table_equals("bitrev_128", [int(format(i, "07b")[::-1], 2) for i in range(128)])
    assert gv.ref_table_equals("twiddle_8", [[32767, 0], [23169, -23169], [32767, 0], [-23169, -23169]])


# ---- the reference's LEGACY transmitter (BB11ATxFrameMod): pinned by its own output file and by vectors made from its own tables ------------
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LEGACY_RATES = (6000, 9000, 12000, 18000, 24000, 36000, 48000, 54000)

def test_legacy_tx_reproduces_ofdm_bin():
    """usr/HwVeri/data/ofdm.bin is the output of the reference's legacy modulator for 200 x 0x31 at 24 Mbps: the restatement
    (oracle/tx11a_legacy.cpp) gives the same 3680 signal samples, sample for sample (the file then holds zeros where
    UpsampleTailAndCopyNT would put the 8-sample window tail, and zero padding up to a 64-byte multiple)."""
    ref = np.fromfile(os.path.join(GOLD, "ofdm.bin"), np.int8).reshape(-1, 2)
    got = oracle_py.tx11a_legacy_modulate(np.full(200, 0x31, np.uint8), 24000)
    assert len(got) == 3688 and len(ref) == 3712
    assert (got[:3680] == ref[:3680]).all()
    assert not ref[3680:].any()

@pytest.mark.parametrize("kbps", LEGACY_RATES)
def test_legacy_tx_vectors_from_reference_tables(kbps):
    """tests/golden/legacy_tx/: one frame per rate made by driving the reference's own LUTs (scrambler, encoder, interleaver, mapper, pilots,
    preamble) the way its C code drives them (tests/golden/make_legacy_tx_vectors.py).  The function-driven restatement must reproduce every
    sample, and the receive oracle must decode the waveform to the frame body: a table-derived known answer at every rate, 54 Mbps included."""
    body = np.fromfile(os.path.join(GOLD, "legacy_tx", f"legacy_tx_{kbps}.bin"), np.uint8)
    ref = np.fromfile(os.path.join(GOLD, "legacy_tx", f"legacy_tx_{kbps}.i8"), np.int8).reshape(-1, 2)
    got = oracle_py.tx11a_legacy_modulate(body, kbps)
    assert got.shape == ref.shape and (got == ref).all()
    iq = np.concatenate([np.zeros((400, 2), np.int16), ref.astype(np.int16) << 8, np.zeros((428, 2), np.int16)])      # ConvertModFile2DumpFile_8b
    res, out = oracle_py.rx11a_run(iq)
    assert len(res) == 1 and res[0]["status"] == 1 and res[0]["rate_kbps"] == kbps and res[0]["length"] == len(body) + 4
    assert bytes(out[0, :len(body)]) == bytes(body)

def test_legacy_tx_vectors_regenerate_from_the_reference():
    """The vectors are what the reference's own transmit lookup tables (kept as data in legacy_tx/lutst_tables.npz) make."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mk", os.path.join(GOLD, "make_legacy_tx_vectors.py")); mk = importlib.util.module_from_spec(spec); spec.loader.exec_module(mk)
    T = mk.stored_tables()
    frame = mk.build(T)
    for kbps in (9000, 54000):
        body = np.fromfile(os.path.join(GOLD, "legacy_tx", f"legacy_tx_{kbps}.bin"), np.uint8)
        assert (frame(body, kbps) == np.fromfile(os.path.join(GOLD, "legacy_tx", f"legacy_tx_{kbps}.i8"), np.int8).reshape(-1, 2)).all()
    pre = np.fromfile(os.path.join(GOLD, "preamble40_11a.i16"), np.int16)
    assert (pre == T["preamble40_11a"]).all()

def test_legacy_tx_ack_frame_round_trip():
    """BB11AModulateACK's path (BB11ATxBufferMod6M: the buffer already ends in its FCS): the 14-byte ACK of the Dot11ADummy fixtures."""
    import golden_vectors as gv
    w = oracle_py.tx11a_legacy_modulate(np.frombuffer(gv.ACK_PSDU, np.uint8), 6000, append_crc=False)
    assert len(w) == 640 + 160 * 7 + 8
    iq = np.concatenate([np.zeros((400, 2), np.int16), w.astype(np.int16) << 8, np.zeros((428, 2), np.int16)])
    res, out = oracle_py.rx11a_run(iq)
    assert len(res) == 1 and res[0]["status"] == 1 and bytes(out[0, :14]) == gv.ACK_PSDU
