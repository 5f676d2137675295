"""CPU tests of the 802.11n 2x2 oracle (no GPU): tables against the reference headers, SIG parsing, loop-back at MCS 8..10."""
import numpy as np, pytest
import oracle_py
from sora_b200 import synth


def test_tables_vs_reference_headers_11n():
    """The oracle's 802.11n tables against the reference headers' (golden/ref_digests.json)."""
    import golden_vectors as gv
    T = oracle_py.tables11n()
    assert gv.ref_table_equals("demap11n_bpsk", T["demap"]) and gv.ref_table_equals("demap11n_qpsk", T["demap"])
    assert gv.ref_table_equals("LUT_CRC8", T["crc8"])
    for q, name in enumerate(("BPSK", "QPSK")):
        for s in range(2):
            assert gv.ref_table_equals(f"deint11n_{name}_S{s}", T["deint"][q, s, :52 * (q + 1)]), (name, s)
            assert gv.ref_table_equals(f"deint11n_{name}_S{s}", synth.ht_interleave_map(q + 1, s))      # modulator and receiver agree on the permutation
    assert gv.ref_table_equals("lltf_plus", T["lltf_sign"].astype(bool)) and gv.ref_table_equals("htltf_plus", T["htltf_sign"].astype(bool))
    assert gv.ref_table_equals("DOT11N_NDBPS_MCS8_14", [synth.HT_MCS[m][2] for m in range(8, 15)])

def test_dsp_math_tables_closed_form():
    T = oracle_py.tables11n()
    i = np.arange(65536); r = i * 2.0 * np.pi / 65535.0
    assert (T["sincos"][:, 0] == np.trunc(np.cos(r) * 32767.5)).all() and (T["sincos"][:, 1] == np.trunc(np.sin(r) * 32767.5)).all()
    assert (T["atan"] == np.trunc(np.arctan(np.arange(4097) / 4096.0) / (np.pi / 4) * 8192)).all()
    L = oracle_py.lib()
    for x, y in ((1000, 0), (1000, 1000), (0, 1000), (-1000, 1000), (1000, -1000), (-7, -3), (0, 0), (30000, 12345), (5, 20000)):
        got = L.sbo_dsp_atan(x, y)
        want = 0.0 if x == 0 and y == 0 else (np.arctan(y / x) if x else np.sign(y) * np.pi / 2) * 32768 / np.pi
        assert abs(((got - want + 32768) % 65536) - 32768) <= 24 or abs(abs(got - want) - 32768) <= 24, (x, y, got, want)   # atan is pi-periodic here

@pytest.mark.parametrize("mcs", [8, 9, 10])
def test_roundtrip_11n(mcs):
    for L, snr, cfo in ((60, None, 0.0), (431, 28, 25e3), (1500, 30, -40e3)):
        iq0, iq1, ps = synth.make_frames_11n(2, psdu_len=L, mcs=mcs, snr_db=snr, lead=400, trail=200, cfo_hz=cfo)
        F, slot, _ = iq0.shape
        res, out = oracle_py.rx11n_batch(iq0.reshape(-1, 2), iq1.reshape(-1, 2), np.arange(F) * slot, np.full(F, slot), out_stride=1536)
        assert (res["status"] == 1).all() and (res["mcs"] == mcs).all() and (res["length"] == L).all(), res
        assert (out[:, :L] == ps).all()
        ndbps = synth.HT_MCS[mcs][2]
        assert (res["nsym"] == -(-(8 * L + 22) // ndbps) + 4).all()
        if cfo: assert np.all(np.abs(res["cfo_est"] + cfo / 20e6 * 65535) < 12)

def test_11n_edges_and_failures():
    res, _ = oracle_py.rx11n_run(np.zeros((4000, 2), np.int16), np.zeros((4000, 2), np.int16)); assert len(res) == 0
    rng = np.random.default_rng(3)
    res, _ = oracle_py.rx11n_run(rng.normal(0, 3000, (30000, 2)).astype(np.int16), rng.normal(0, 3000, (30000, 2)).astype(np.int16))
    assert all(r["status"] != 1 for r in res)
    iq0, iq1, ps = synth.make_frames_11n(1, psdu_len=300, mcs=9, snr_db=30, lead=400, trail=200)
    a, b = iq0[0].copy(), iq1[0].copy()
    a[3000:3300] = rng.integers(-4000, 4000, (300, 2)); b[3000:3300] = rng.integers(-4000, 4000, (300, 2))      # payload hit
    res, _ = oracle_py.rx11n_run(a, b); assert len(res) >= 1 and res[0]["status"] == oracle_py.E_CRC32_FAIL
    a, b = iq0[0].copy(), iq1[0].copy()
    s = 400 + 640 + 160                                                                                              # HT-SIG1 symbol
    a[s:s + 160] = rng.integers(-4000, 4000, (160, 2)); b[s:s + 160] = rng.integers(-4000, 4000, (160, 2))
    res, _ = oracle_py.rx11n_run(a, b); assert len(res) >= 1 and res[0]["status"] == oracle_py.E_PLCP_FAIL
    # a legacy 802.11a frame on both antennas: L-SIG parses, HT-SIG CRC does not
    iq, _ = synth.make_frames(1, psdu_len=200, rate_kbps=6000, snr_db=30, lead=400, trail=200, gain=0.6)
    res, _ = oracle_py.rx11n_run(iq[0], iq[0]); assert len(res) >= 1 and res[0]["status"] == oracle_py.E_PLCP_FAIL
    # two frames in one capture
    iq0, iq1, ps = synth.make_frames_11n(2, psdu_len=120, mcs=10, snr_db=30, lead=400, trail=300)
    res, out = oracle_py.rx11n_run(iq0.reshape(-1, 2), iq1.reshape(-1, 2))
    assert len(res) == 2 and (res["status"] == 1).all() and (out[:, :120] == ps).all()
