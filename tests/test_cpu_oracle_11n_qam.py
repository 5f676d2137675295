"""802.11n MCS 11..14 (16-QAM / 64-QAM over two streams) in the oracle (no GPU).  The reference's graphs carry these branches
(fb11ndemod_config.hpp:196-236, fb11nmod_config.hpp:133-155) but its HT-SIG parser refuses every MCS >= 11 (PHY_11n.hpp:497); the oracle keeps that
behaviour by default and opens the gate with set_ht_mcs_limit(15) (SURVEY.md §8(f) rank 4).  Pins: the tables against the reference headers, the
restated modulator graph against the restated receive graph, and an independent float clause-20 modulator."""
import os, sys, zlib, numpy as np, pytest
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_py
from sora_b200 import synth

@pytest.fixture()
def qam_enabled():
    oracle_py.set_ht_mcs_limit(15)
    yield
    oracle_py.set_ht_mcs_limit(11)

def test_qam_tables_vs_reference_headers():
    """The oracle's 16-/64-QAM demap and HT deinterleave tables against the reference headers' (golden/ref_digests.json)."""
    import golden_vectors as gv
    T = oracle_py.tables11n()
    for i, n in enumerate(("16qam1", "16qam2")): assert gv.ref_table_equals("demap11n_" + n, T["demap16"][i]), n
    for i, n in enumerate(("64qam1", "64qam2", "64qam3")): assert gv.ref_table_equals("demap11n_" + n, T["demap64"][i]), n
    for q, (name, nb) in enumerate((("BPSK", 1), ("QPSK", 2), ("QAM16", 4), ("QAM64", 6))):
        for s in range(2):
            assert gv.ref_table_equals(f"deint11n_{name}_S{s}", T["deint"][q, s, :52 * nb]), (name, s)
            assert gv.ref_table_equals(f"deint11n_{name}_S{s}", synth.ht_interleave_map(nb, s))       # the independent modulator uses the same permutation
    assert gv.ref_table_equals("DOT11N_NDBPS_MCS8_14", [synth.HT_MCS[m][2] for m in range(8, 15)])

def _rx(o0, o1, chan, noise, seed=1, lead=400, trail=300):
    a = o0[:, 0] + 1j * o0[:, 1]; b = o1[:, 0] + 1j * o1[:, 1]
    r0 = chan[0][0] * a + chan[0][1] * b; r1 = chan[1][0] * a + chan[1][1] * b
    rng = np.random.default_rng(seed)
    def pack(r):
        x = np.concatenate([np.zeros((lead, 2)), np.stack([r.real, r.imag], 1), np.zeros((trail, 2))])
        if noise: x = x + rng.normal(0, noise, x.shape)
        return np.clip(np.round(x), -32768, 32767).astype(np.int16)
    return oracle_py.rx11n_run(pack(r0), pack(r1), 4, 1536)

@pytest.mark.parametrize("mcs", [11, 12, 13, 14])
def test_restated_modulator_to_restated_receiver(qam_enabled, mcs):
    rng = np.random.default_rng(mcs)
    for L in (1, 2, 37, 200, 777, 1496):
        p = rng.integers(0, 256, L).astype(np.uint8)
        o0, o1 = oracle_py.tx11n_modulate(p, mcs)
        for chan, noise in ((((1, 0), (0, 1)), 0.0), (((1.0, 0.3j), (-0.2, 0.9)), 12.0), (((0.6, -0.5), (0.4j, 0.7)), 0.0)):
            res, out = _rx(o0, o1, chan, noise, seed=L)
            assert len(res) == 1 and res[0]["status"] == 1 and res[0]["mcs"] == mcs and res[0]["length"] == L + 4, (mcs, L, chan, res)
            assert (out[0, :L] == p).all() and int.from_bytes(bytes(out[0, L:L + 4]), "little") == zlib.crc32(p.tobytes())

@pytest.mark.parametrize("mcs", [11, 12, 13, 14])
def test_independent_float_modulator_to_receiver(qam_enabled, mcs):
    for L, snr, cfo in ((60, None, 0.0), (431, 36, 25e3), (1500, 38, -40e3)):
        iq0, iq1, ps = synth.make_frames_11n(2, psdu_len=L, mcs=mcs, snr_db=snr, lead=400, trail=200, cfo_hz=cfo)
        F, slot, _ = iq0.shape
        res, out = oracle_py.rx11n_batch(iq0.reshape(-1, 2), iq1.reshape(-1, 2), np.arange(F) * slot, np.full(F, slot), out_stride=1536)
        assert (res["status"] == 1).all() and (res["mcs"] == mcs).all() and (res["length"] == L).all(), res
        assert (out[:, :L] == ps).all()
        assert (res["nsym"] == -(-(8 * L + 22) // synth.HT_MCS[mcs][2]) + 4).all()

def test_reference_behaviour_is_the_default():
    """With the gate where the reference has it, an MCS 12 frame ends at HT-SIG with E_ERROR_PLCP_HEADER_FAIL (PHY_11n.hpp:496-501)."""
    assert oracle_py.lib().sbo_ht_mcs_limit() == 11
    p = np.arange(100, dtype=np.uint8)
    o0, o1 = oracle_py.tx11n_modulate(p, 12)
    res, _ = _rx(o0, o1, ((1, 0), (0, 1)), 0.0)
    assert len(res) >= 1 and res[0]["status"] == oracle_py.E_PLCP_FAIL and res[0]["mcs"] == 12

def test_symbol_counts_qam(qam_enabled):
    """TBB11nSrc + the FlushPort paddings (encoder burst 1 / 2 / 3 bytes, parser burst 52 / 78 bytes): emitted symbols >= signalled symbols, never more than one extra."""
    L = oracle_py.lib()
    for mcs in (11, 12, 13, 14):
        for n in range(1, 1497, 7):
            sig = C_uint32(); ns = L.sbo_tx11n_nsym(n, mcs, byref(sig))
            assert sig.value == -(-((n + 4) * 8 + 22) // synth.HT_MCS[mcs][2]) and 0 <= ns - sig.value <= 1, (mcs, n, ns, sig.value)
from ctypes import c_uint32 as C_uint32, byref
