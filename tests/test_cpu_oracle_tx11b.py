"""CPU tests of the 802.11b transmit restatement (oracle/tx11b.cpp): stage tables rebuilt from the reference's formulas, the
shaper's impulse response, and the fixed-point TX -> fixed-point RX round trip at all four rates through the receive oracle (which
is pinned by the reference's own *.mf.bin captures)."""
import numpy as np, pytest
import oracle_py

def _rx(samples8, lead=300, trail=600):
    iq = np.concatenate([np.zeros((lead, 2), np.int16), samples8.astype(np.int16) << 8, np.zeros((trail, 2), np.int16)])
    res, out = oracle_py.rx11b_batch(iq, np.array([0], np.uint64), np.array([len(iq)], np.uint32), out_stride=4096)
    return res[0], out[0]

@pytest.mark.parametrize("rate", [1000, 2000, 5500, 11000])
def test_tx_oracle_to_rx_oracle_roundtrip(rate):
    rng = np.random.default_rng(rate)
    for L in (1, 37, 200, 1496):
        if rate == 1000 and L > 400: continue                              # 1 Mbps at 1500 B is 4.3 M samples of scalar receive oracle
        payload = rng.integers(0, 256, L).astype(np.uint8)
        td = oracle_py.tx11b_modulate(payload, rate)
        cpb = {1000: 88, 2000: 44, 5500: 16, 11000: 8}[rate]
        assert len(td) == ((24 * 88 + (L + 4) * cpb + 5) * 4 + 7) // 8 * 8
        res, out = _rx(td)
        assert res["status"] == 1 and res["rate_kbps"] == rate and res["length"] == L + 4, (rate, L, res)
        assert (out[:L] == payload).all()

def test_shaper_taps_and_impulse_response():
    h = oracle_py.tx11b_taps()
    # pulse.hpp:292-300 evaluated independently: 80 * 4 cos(pi i / 2) / (pi (1 - i^2)), 80 at i = +-1, rounded like (short)(x + .5)
    want = []
    for i in range(8, -12, -1):
        x = 1.0 if abs(i) == 1 else 4 * np.cos(3.141593 * i / 2) / 3.141593 / (1 - i * i)
        want.append(int(np.trunc(x * 80 + .5)))
    assert list(h) == want and h[8] == 102 and h[7] == 80 and h[9] == 80 and h[6] == 34
    # the first chip of every frame is +1 (scrambled sync, phase 0): the head of the waveform is the impulse response until chip 2 arrives
    td = oracle_py.tx11b_modulate(np.zeros(1, np.uint8), 1000)
    assert (td[:4, 0] == h[:4]).all() and (td[:, 1] == 0).all()

def test_differential_reference_carries_over_and_global_phase():
    """init_phase = 3 (pi) negates a DBPSK/CCK frame as a whole; the receiver is differential and must not care."""
    p = np.arange(60, dtype=np.uint8)
    for rate in (1000, 11000):
        a = oracle_py.tx11b_modulate(p, rate, 0).astype(np.int32); b = oracle_py.tx11b_modulate(p, rate, 3).astype(np.int32)
        assert (a == -b).all()
        res, out = _rx(b.astype(np.int8))
        assert res["status"] == 1 and (out[:60] == p).all()

def test_final_phase_chains_frames():
    """last_phase after a frame is the reference phase the next one starts from: two frames modulated back to back on one context are
    the second frame's waveform rotated by that phase (0 / pi for DBPSK, quarter turns otherwise)."""
    p = np.arange(33, dtype=np.uint8)
    for rate in (1000, 2000, 5500, 11000):
        _, fin = oracle_py.tx11b_modulate(p, rate, 0, return_phase=True)
        assert fin in (0, 1, 2, 3) and (rate != 1000 or fin in (0, 3))
        a = oracle_py.tx11b_modulate(p, rate, 0).astype(np.int32); b = oracle_py.tx11b_modulate(p, rate, fin).astype(np.int32)
        z = {0: 1, 1: -1j, 2: 1j, 3: -1}[fin & 1 and 3 or 0]            # the preamble is DBPSK: only bit 0 of the reference enters (barkerspread.hpp:96)
        assert ((a[:, 0] + 1j * a[:, 1]) * z == b[:, 0] + 1j * b[:, 1]).all()

def test_plcp_length_extension_bit():
    """11 Mbps: LENGTH in microseconds is ambiguous by one byte; the service bit 7 resolves it (PHY_11b.hpp:82-104).  The receive
    oracle applies the same rule, so every length in a run of 11 consecutive ones must come back exactly."""
    for L in range(100, 111):
        p = (np.arange(L) * 7 + 3).astype(np.uint8)
        res, out = _rx(oracle_py.tx11b_modulate(p, 11000))
        assert res["status"] == 1 and res["length"] == L + 4 and (out[:L] == p).all(), (L, res)

def test_tx11b_constants_vs_reference():
    """The constants oracle/tx11b.cpp restates, against the reference's barkerspread.hpp, cck.hpp and dot11_plcp.h (golden/ref_digests.json)."""
    import golden_vectors as gv
    assert gv.ref_table_equals("Barker11", [1, -1, 1, 1, -1, 1, 1, 1, -1, -1, -1])
    assert gv.ref_table_equals("DQPSKEncode", [[1, 0], [0, -1], [0, 1], [-1, 0]]) and gv.ref_table_equals("CCK11D3D2", [[1, 0], [-1, 0], [0, 1], [0, -1]])
    assert gv.ref_table_equals("DOT11B_PLCP_LONG_TX_SCRAMBLER_REGISTER", [0x6C]) and gv.ref_table_equals("DOT11B_PLCP_LONG_PREAMBLE_SFD", [0xF3A0])
