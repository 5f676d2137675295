"""CPU tests of the 802.11n two-stream transmit restatement (oracle/tx11n.cpp).  The reference ships no 802.11n vector, so the
receive oracle cannot be pinned by one; instead the two halves of the reference's 802.11n code — modulator graphs and demodulator
graph — are restated independently and played against each other here: every frame the transmit restatement makes must come out of
the receive restatement bit for bit (L-SIG / HT-SIG fields, CRC-8, HT interleavers, stream parser, pilots, cyclic shifts)."""
import zlib, numpy as np, pytest
import oracle_py

def _rx(o0, o1, chan=((1, 0), (0, 1)), noise=0.0, seed=0, lead=400, trail=300, cfo_hz=0.0):
    a = o0.astype(np.float64); b = o1.astype(np.float64)
    rot = np.exp(2j * np.pi * cfo_hz * np.arange(len(a)) / 40e6)
    ca = (a[:, 0] + 1j * a[:, 1]) * rot; cb = (b[:, 0] + 1j * b[:, 1]) * rot
    r0 = chan[0][0] * ca + chan[0][1] * cb; r1 = chan[1][0] * ca + chan[1][1] * cb
    rng = np.random.default_rng(seed)
    def pack(r):
        x = np.stack([r.real, r.imag], 1)
        x = np.concatenate([np.zeros((lead, 2)), x, np.zeros((trail, 2))])
        if noise: x = x + rng.normal(0, noise, x.shape)
        return np.clip(np.round(x), -32768, 32767).astype(np.int16)
    return oracle_py.rx11n_run(pack(r0), pack(r1), 4, 1536)

@pytest.mark.parametrize("mcs", [8, 9, 10])
def test_tx_oracle_to_rx_oracle_roundtrip(mcs):
    rng = np.random.default_rng(mcs)
    for L in (1, 2, 37, 200, 777, 1496):
        p = rng.integers(0, 256, L).astype(np.uint8)
        o0, o1 = oracle_py.tx11n_modulate(p, mcs)
        for chan, noise in ((((1, 0), (0, 1)), 0.0), (((1.0, 0.3j), (-0.2, 0.9)), 40.0), (((0.6, -0.5), (0.4j, 0.7)), 0.0)):
            res, out = _rx(o0, o1, chan, noise, seed=L)
            assert len(res) == 1 and res[0]["status"] == 1 and res[0]["mcs"] == mcs and res[0]["length"] == L + 4, (mcs, L, chan, res)
            assert (out[0, :L] == p).all() and int.from_bytes(bytes(out[0, L:L + 4]), "little") == zlib.crc32(p.tobytes())

def test_roundtrip_with_carrier_offset():
    """+-40 kHz between the two restated halves: joint CFO estimate, NCO and pilot tracking of the receive side against the transmit side's
    preambles and pilots (the pilot polarity index of the modulator is one ahead of the standard's; the receiver's tracking is polarity-blind)."""
    p = np.arange(400, dtype=np.uint8)
    for mcs in (8, 9, 10):
        for cfo in (-40e3, 13e3, 40e3):
            res, out = _rx(*oracle_py.tx11n_modulate(p, mcs), chan=((1.0, 0.3j), (-0.2, 0.9)), noise=25.0, seed=7, cfo_hz=cfo)
            assert len(res) == 1 and res[0]["status"] == 1 and (out[0, :400] == p).all(), (mcs, cfo, res)
            est_hz = res[0]["cfo_est"] / 65536.0 * 20e6                                      # 2^16 / 2 pi radians per 20 Msps sample
            assert abs(est_hz + cfo) < 3e3, (mcs, cfo, est_hz)                               # CFO_est is the correction, i.e. minus the offset

def test_symbol_counts_and_flush_padding():
    """HT-SIG announces ceil((8 (L + 4) + 22) / N_DBPS) symbols; the graph emits one more when the padded byte stream does not end on a
    stream-parser burst (odd symbol counts at MCS 8 and MCS 10): the receiver must stop at the announced count either way."""
    for mcs, ndbps in ((8, 52), (9, 104), (10, 156)):
        for L in range(1, 60):
            o0, _ = oracle_py.tx11n_modulate(np.zeros(L, np.uint8), mcs)
            want = -(-((L + 4) * 8 + 22) // ndbps)
            n_tx = (len(o0) - 1600) // 160
            assert n_tx in (want, want + 1) and (mcs != 9 or n_tx == want), (mcs, L, n_tx, want)
    res, _ = _rx(*oracle_py.tx11n_modulate(np.arange(30, dtype=np.uint8), 8))
    assert res[0]["nsym"] == -(-(34 * 8 + 22) // 52) + 4                                  # total_symbols counts data + 4 (PHY_11n.hpp:508)

def test_second_stream_is_a_cyclically_delayed_copy_in_the_legacy_part():
    """L-STF, L-LTF, L-SIG and HT-SIG go out on both antennas, the second one delayed by 200 ns (8 samples) per symbol body."""
    o0, o1 = oracle_py.tx11n_modulate(np.arange(100, dtype=np.uint8), 9)
    assert (np.roll(o0[:320], 8, axis=0) == o1[:320]).all()
    for s in range(3):                                                                    # SIG symbols: 32-sample GI + 128 body
        b0 = o0[640 + 160 * s + 32: 640 + 160 * s + 160]; b1 = o1[640 + 160 * s + 32: 640 + 160 * s + 160]
        assert (np.roll(b0, 8, axis=0) == b1).all() and (o1[640 + 160 * s: 640 + 160 * s + 32] == b1[96:]).all()
    # HT-LTF: stream 1 sends (+, -), stream 2 (+, +) delayed by 400 ns
    h = 640 + 480 + 160
    assert (o0[h:h + 160] == -o0[h + 160:h + 320]).all() and (o1[h:h + 160] == o1[h + 160:h + 320]).all()
    assert (np.roll(o0[h + 32:h + 160], 16, axis=0) == o1[h + 32:h + 160]).all()

def test_preamble_and_pilot_tables_vs_reference():
    """The preamble tables of oracle/tx11n.cpp and the HT pilot polarity against the reference's _b_*.h tables (golden/ref_digests.json)."""
    import golden_vectors as gv
    a, b, c, d = oracle_py.tx11n_preamble_tables()
    assert gv.ref_table_equals("L_STF", a) and gv.ref_table_equals("L_LTF", b)
    assert gv.ref_table_equals("HT_STF", c) and gv.ref_table_equals("HT_LTF", d)
    # the 127-entry pilot polarity table of the HT pilot generator is the 802.11a one (entry i = p(i+1)): x^7 + x^4 + 1 from all ones
    st = 0x7F; seq = []
    for _ in range(127): o = ((st >> 6) ^ (st >> 3)) & 1; st = ((st << 1) | o) & 0x7F; seq.append(1 - 2 * o)
    assert gv.ref_table_equals("_pilot_sign", [seq[(k + 1) % 127] for k in range(127)])
