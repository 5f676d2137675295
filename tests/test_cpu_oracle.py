"""CPU suite (pytest -m "not gpu"): the oracle against the reference's golden fixtures and closed-form tables, the host
logic, the ABI surface.  No CUDA compute is called here."""
import hashlib, zlib, os, re, sys, subprocess, ctypes
import numpy as np, pytest
import oracle_py
from sora_b200 import synth
from sora_b200.dumpfile import load_dump, write_dump

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

def _fs6():
    iq = load_dump(os.path.join(GOLD, "fsample-6.dmp"))
    return (iq.astype(np.int32) << 2).astype(np.int16)   # xmmAdjustSignBit: 14-bit samples to the top of 16 (dot11a/dot11/arx_fd.c:530)

def test_fsample6_golden_frame():
    """SURVEY.md §8c pin (1): kernel/test-data/fsample-6.dmp must decode to one CRC-good 6 Mbps, LENGTH 1392 frame."""
    res, out = oracle_py.rx11a_run(_fs6())
    assert len(res) == 1
    r = res[0]
    assert r["status"] == oracle_py.E_FRAME_OK and r["rate_kbps"] == 6000 and r["length"] == 1392 and r["nsym"] == 466
    psdu = out[0, :1392]
    assert oracle_py.crc32(psdu[:-4]) == int(r["crc32"]) == int.from_bytes(psdu[-4:].tobytes(), "little")
    gold = np.fromfile(os.path.join(GOLD, "fsample-6.psdu.bin"), np.uint8)
    assert (psdu == gold).all()
    import golden_vectors as gv                                                      # the golden file is the reference's capture, byte for byte
    assert hashlib.sha256(open(os.path.join(GOLD, "fsample-6.dmp"), "rb").read()).hexdigest() == gv.ref_digests()["files"]["kernel/test-data/fsample-6.dmp"]

def _ofdm_bin():
    raw = np.fromfile(os.path.join(GOLD, "ofdm.bin"), dtype=np.int8).reshape(-1, 2)
    iq = raw.astype(np.int16) << 8                       # ConvertModFile2DumpFile_8b (demod11/modulate11a.cpp:178-179)
    return np.concatenate([np.zeros((400, 2), np.int16), iq, np.zeros((400, 2), np.int16)])

def test_ofdm_bin_golden_frame():
    """The reference's own modulator output (usr/HwVeri/data/ofdm.bin): 24 Mbps, LENGTH 204, 200 x 0x31 + FCS."""
    res, out = oracle_py.rx11a_run(_ofdm_bin())
    assert len(res) == 1 and res[0]["status"] == 1 and res[0]["rate_kbps"] == 24000 and res[0]["length"] == 204
    assert (out[0, :200] == 0x31).all() and bytes(out[0, 200:204]) == bytes.fromhex("388d4983")
    assert zlib.crc32(bytes(out[0, :200])) == int.from_bytes(bytes(out[0, 200:204]), "little")

@pytest.mark.parametrize("name", ["dummy_20m", "dummy_16_40m", "dummy_8_20m", "dummy_8_ack_40m"])
def test_reference_dummy_frames(name):
    """kernel/sample/mac/Dot11ADummy*.txt: four waveforms of the reference's own (legacy) modulator.  The two long ones carry the very
    frame of fsample-6.dmp (three independent renderings of one PSDU must decode to the same 1392 bytes); the two short ones are the
    14-byte ACK that BB11AModulateACK builds, whose bytes are known in full."""
    import golden_vectors as gv
    iq, rate, want = gv.dummy_vectors()[name]
    res, out = oracle_py.rx11a_run(iq)
    assert len(res) == 1 and res[0]["status"] == oracle_py.E_FRAME_OK and res[0]["rate_kbps"] == rate
    L = int(res[0]["length"]); psdu = bytes(out[0, :L])
    assert zlib.crc32(psdu[:-4]) == int.from_bytes(psdu[-4:], "little") == int(res[0]["crc32"])
    if want is None:
        assert L == 1392 and psdu == bytes(gv.fsample6_psdu()) and int(res[0]["crc32"]) == 0x80EF9B11
    else:
        assert psdu == want
        # the ACK is a legal control frame: FC 0x00D4, duration 0, RA, FCS (dot11 ACK layout, atx_fe.c:168-180)
        assert psdu[:2] == b"\xd4\x00" and psdu[2:4] == b"\x00\x00" and L == 14

def test_reference_dummy_frames_gain_invariant():
    """The decode does not hinge on the gain chosen in golden_vectors: any power of two that clears the energy threshold gives the same bytes."""
    import golden_vectors as gv
    v = np.fromfile(os.path.join(GOLD, "dot11a_dummy_16_40m.i16"), np.int16).reshape(-1, 2).astype(np.int32)
    for sh in (2, 3):
        iq = np.concatenate([np.zeros((400, 2), np.int16), (v << sh).astype(np.int16), np.zeros((428, 2), np.int16)])
        res, out = oracle_py.rx11a_run(iq)
        assert len(res) == 1 and res[0]["status"] == 1 and bytes(out[0, :1392]) == bytes(gv.fsample6_psdu())

def test_dump_roundtrip(tmp_path):
    iq = _fs6()[:28 * 40]
    p = tmp_path / "x.dmp"; write_dump(str(p), iq)
    assert (load_dump(str(p)) == iq).all()

@pytest.mark.parametrize("rate", sorted(synth.RATES))
def test_roundtrip_all_rates(rate):
    iq, ps = synth.make_frames(3, psdu_len=211, rate_kbps=rate, snr_db=28, seed0=rate)
    F, slot, _ = iq.shape
    res, out = oracle_py.rx11a_batch(iq.reshape(-1, 2), np.arange(F) * slot, np.full(F, slot))
    assert (res["status"] == 1).all() and (res["rate_kbps"] == rate).all() and (res["length"] == 211).all()
    assert (out[:, :211] == ps).all()

def test_two_thread_topology_gives_the_same_results():
    """The CPU baseline's variant (ii) — front end and Viterbi on two threads joined by a ring like TThreadSeparator — is the same decoder."""
    parts = []
    for rate in (6000, 36000, 54000):
        iq, _ = synth.make_frames(3, psdu_len=300, rate_kbps=rate, snr_db=12 if rate == 36000 else 28, seed0=rate + 9)
        parts.append(iq)
    slot = max(p.shape[1] for p in parts); F = 9
    iq = np.zeros((F, slot, 2), np.int16)
    for i, p in enumerate(parts): iq[3 * i: 3 * i + 3, :p.shape[1]] = p
    flat = iq.reshape(-1, 2).copy(); flat[5 * slot + 700: 5 * slot + 760] = 0          # damage one SIGNAL/early symbol region
    off = np.arange(F) * slot; ln = np.full(F, slot); ln[7] = 2000                      # and truncate one slot
    r1, o1 = oracle_py.rx11a_batch(flat, off, ln)
    for npipes in (1, 3):
        r2, o2 = oracle_py.rx11a_batch_2t(flat, off, ln, npipes=npipes)
        assert (r1 == r2).all() and (o1 == o2).all()

def test_stream_mode_multiple_frames():
    """RxThread semantics: several frames in one capture are found one after another (fb11a_demod.cpp:29-81)."""
    iq, ps = synth.make_frames(4, psdu_len=150, rate_kbps=24000, snr_db=30, lead=400, trail=300)
    res, out = oracle_py.rx11a_run(iq.reshape(-1, 2), max_frames=8)
    assert len(res) == 4 and (res["status"] == 1).all()
    assert (out[:4, :150] == ps).all()

def test_edge_inputs():
    z = np.zeros((3000, 2), np.int16)
    res, _ = oracle_py.rx11a_run(z); assert len(res) == 0
    res, _ = oracle_py.rx11a_run(np.zeros((5, 2), np.int16)); assert len(res) == 0
    rng = np.random.default_rng(1)
    res, _ = oracle_py.rx11a_run(rng.normal(0, 4000, (20000, 2)).astype(np.int16))
    assert all(r["status"] != 1 for r in res)
    iq, _ = synth.make_frames(1, psdu_len=2500, rate_kbps=54000)          # MTU (PHY_11a.hpp:571)
    res, _ = oracle_py.rx11a_run(iq[0]); assert res[0]["status"] == 1 and res[0]["length"] == 2500
    iq, _ = synth.make_frames(1, psdu_len=2501, rate_kbps=54000)
    res, _ = oracle_py.rx11a_run(iq[0]); assert res[0]["status"] == oracle_py.E_PLCP_FAIL

def test_fft64_close_to_float():
    rng = np.random.default_rng(0)
    x = rng.integers(-6000, 6000, (64, 2)).astype(np.int16)
    y = oracle_py.fft64(x).astype(np.float64)
    ref = np.fft.fft(x[:, 0] + 1j * x[:, 1]) / 64.0
    err = np.abs((y[:, 0] + 1j * y[:, 1]) - ref)
    assert err.max() < 8.0            # fixed point, 3 truncating stages and one's-complement negations: a few LSB
    z = oracle_py.ifft64(oracle_py.fft64(x)).astype(np.float64)
    assert np.abs(z / 1.0 - x / 64.0).max() < 12.0    # two fixed-point transforms back to back (each 2^-6): sanity bound only

def test_viterbi_known_answer():
    rng = np.random.default_rng(5)
    for cr, rate in ((0, (1, 2)), (1, (2, 3)), (2, (3, 4))):
        L = 100; n = 8 * L + 16 + 6; n += (-n) % 48
        bits = rng.integers(0, 2, (1, n)).astype(np.uint8); bits[:, 8 * L + 16:] = 0
        A, B = synth.conv_encode(bits); coded = synth.puncture(A, B, rate)[0]
        soft = np.where(coded > 0, 7, 0).astype(np.uint8)
        out = oracle_py.viterbi_block(soft, cr, L)
        assert (np.unpackbits(out, bitorder="little")[:8 * L + 16] == bits[0, :8 * L + 16]).all()

def test_signal_field_known_answer():
    sig = np.zeros(24, np.uint8); sig[0:4] = [1, 1, 0, 1]; L = 1392
    sig[5:17] = [(L >> i) & 1 for i in range(12)]; sig[17] = sig[:17].sum() & 1
    A, B = synth.conv_encode(sig); coded = synth.puncture(A, B, (1, 2))
    soft = np.where(coded > 0, 7, 0).astype(np.uint8)
    w = oracle_py.lib().sbo_viterbi_signal(soft.ctypes.data_as(ctypes.c_void_p))
    assert (w & 0xF) == 0xB and ((w >> 5) & 0xFFF) == 1392

def test_tables_vs_reference_headers():
    """The closed-form tables of oracle/ and csrc/ against the reference headers' lookup tables (golden/ref_digests.json)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import refcheck as rc, golden_vectors as gv
    for N in (16, 64):
        for M in (1, 2, 3):
            assert gv.ref_table_equals(f"twiddle_{N}_{M}", rc.gen_twiddle(N, M)), (N, M)
    assert gv.ref_table_equals("bitrev_64", [int(f"{i:06b}"[::-1], 2) for i in range(64)])
    assert gv.ref_table_equals("usin_lut", rc.gen_sin()) and gv.ref_table_equals("ucos_lut", rc.gen_cos()) and gv.ref_table_equals("uatan2_lut", rc.gen_atan2())
    ga, gb = rc.gen_vit()
    assert gv.ref_table_equals("VIT_MA", ga) and gv.ref_table_equals("VIT_MB", gb)
    for cls, n, b in (("BPSK", 48, 1), ("QPSK", 96, 2), ("QAM16", 192, 4), ("QAM64", 288, 6)):
        assert gv.ref_table_equals(f"deint11a_{cls}", rc.gen_deinterleave(n, b)), cls
    # LTS signs and pilot polarity used by oracle/rx11a.cpp and csrc/tables.cuh
    exp = np.array([1 if (-26 <= (i if i < 32 else i - 64) <= 26 and synth._LTS[(i if i < 32 else i - 64) + 26] > 0) else 0 for i in range(64)])
    assert gv.ref_table_equals("LTS_Sequence_11a", exp)
    pol = synth._PILOT_POL
    exp = np.array([0 if pol[(i + 1) % 127] > 0 else -1 for i in range(127)] + [0])
    assert gv.ref_table_equals("PilotSgn", exp)
    # demap tables shipped as data
    tb = ctypes.POINTER(ctypes.c_uint8)
    a_, b_, d_ = tb(), tb(), tb()
    oracle_py.lib().sbo_tables(ctypes.byref(a_), ctypes.byref(b_), ctypes.byref(d_))
    got = np.ctypeslib.as_array(d_, shape=(1024,))
    for i, name in enumerate(("m_bpsk_lut", "m_qam16_lut2", "m_qam64_lut2", "m_qam64_lut3")):
        assert gv.ref_table_equals(name, got[256 * i: 256 * (i + 1)]), name

def test_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "sora_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 8
    from sora_b200 import api
    lib = api.load_library()            # loads without a GPU; no compute entry point is called
    for name in declared:
        assert hasattr(lib, name), name
    assert sorted(api.EXPORTS) == declared
    leg = open(os.path.join(ROOT, "include", "sora_b200_legacy.h")).read()
    legacy = sorted(set(re.findall(r"\b(BB11[AB][A-Z][a-z][A-Za-z0-9]*|SoraGenRadioRxStreamOffline)\s*\(", leg)))
    assert len(legacy) >= 13 and "BB11BSpd" in legacy and "BB11BRx" in legacy
    for name in legacy:
        assert hasattr(lib, name), name

def test_brick_adaptors_compile(tmp_path):
    """The header-only adaptors (11a/b/n receive, 11a transmit) instantiate against the BRICK contract with plain g++."""
    obj = str(tmp_path / "tu.o")
    subprocess.check_call(["g++", "-std=c++17", "-O0", "-Wall", "-I", os.path.join(ROOT, "sora_b200", "brick"), "-c",
                           os.path.join(ROOT, "tests", "cpp", "brick_adaptors_tu.cpp"), "-o", obj])
    assert os.path.getsize(obj) > 0

def test_product_never_touches_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "sora_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                txt = open(os.path.join(dirpath, f), errors="replace").read()
                assert "oracle_py" not in txt and "libsora_oracle" not in txt and 'oracle/' not in txt.replace("oracle/ is test", ""), f

def test_engine_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from sora_b200 import api
    with pytest.raises(api.Sb200Error):
        api.Engine(0)

def _capture_44(rate, psdu_len, seed, snr_db=None):
    """An 802.11a PPDU captured at 44 Msps: the 40 Msps float waveform band-limited-interpolated by 11/10."""
    r = np.random.RandomState(seed); ps = synth.psdu_with_fcs(r.randint(0, 256, psdu_len - 4).astype(np.uint8))
    td = synth.modulate(ps[None, :], rate)[0]
    X = np.fft.fft(np.concatenate([np.zeros(100), td, np.zeros(100)])); N = len(X); M = N * 11 // 10
    Y = np.zeros(M, complex); h = N // 2; Y[:h] = X[:h]; Y[-h:] = X[-h:]
    td44 = np.fft.ifft(Y) * M / N
    iq = synth.to_iq16(td44[None, :], lead=44, trail=300 + (-(344 + len(td44))) % 28, snr_db=snr_db, rng=np.random.default_rng(seed))[0]
    return iq, ps

def test_44msps_resampler_and_decode():
    """fb11ademod_config.hpp:244-317 (CreateDemodGraph11a_44M): 11:10 linear resampler in front of the 40 Msps graph."""
    x = np.zeros((28 * 11, 2), np.int16); x[:, 0] = np.arange(len(x)) * 37 % 2001 - 1000; x[:, 1] = 7
    y = oracle_py.resample_44_40(x)
    assert len(y) == 280 and (y[0] == x[0]).all() and (y[10] == x[11]).all()
    xi = x.astype(np.int64)
    assert y[1, 0] == (xi[1, 0] * 115 + xi[2, 0] * 13) >> 7 and y[9, 0] == (xi[9, 0] * 13 + xi[10, 0] * 115) >> 7
    for rate in (6000, 24000, 54000):
        iq, ps = _capture_44(rate, 150, rate)
        res, out = oracle_py.rx11a_run(oracle_py.resample_44_40(iq))
        assert len(res) == 1 and res[0]["status"] == 1 and res[0]["rate_kbps"] == rate and (out[0, :150] == ps).all()
