"""Loaders for the reference-held 802.11a waveforms under tests/golden (shared by the CPU and the GPU suites).

Every vector is a TRANSMIT waveform of the reference (what its modulator handed to the DAC); the receive chain sees it through a
noiseless unit channel: 20 Msps vectors are sample-repeated to the 40 Msps capture rate (TDownSample2 keeps samples 0 and 2 of
every 4, samples.hpp:27-49, so the decimated stream is the vector itself), 8-bit vectors are shifted like
ConvertModFile2DumpFile_8b does (demod11/modulate11a.cpp:178-179), and a power-of-two gain lifts the 16-bit ones over
cca_pwr_threshold."""
import hashlib, json, os, numpy as np
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

ACK_PSDU = bytes.fromhex("d40000000250f2000004b033a9eb")      # ACK to 02:50:F2:00:00:04 incl. FCS (what BB11AModulateACK encodes, atx_fe.c:168-195)

def _pad(iq, lead=400, trail=428):
    return np.concatenate([np.zeros((lead, 2), np.int16), iq, np.zeros((trail, 2), np.int16)])

def dummy_vectors():
    """name -> (iq int16 [n,2] at 40 Msps, expected rate_kbps, expected PSDU bytes or None for 'equals fsample-6.psdu.bin')"""
    out = {}
    v = np.fromfile(os.path.join(GOLD, "dot11a_dummy_20m.i16"), np.int16).reshape(-1, 2)
    out["dummy_20m"] = (_pad(np.repeat((v.astype(np.int32) << 1).astype(np.int16), 2, axis=0)), 6000, None)
    v = np.fromfile(os.path.join(GOLD, "dot11a_dummy_16_40m.i16"), np.int16).reshape(-1, 2)
    out["dummy_16_40m"] = (_pad((v.astype(np.int32) << 2).astype(np.int16)), 6000, None)
    v = np.fromfile(os.path.join(GOLD, "dot11a_dummy_8_20m.i8"), np.int8).reshape(-1, 2)
    out["dummy_8_20m"] = (_pad(np.repeat(v.astype(np.int16) << 8, 2, axis=0)), 6000, ACK_PSDU)
    v = np.fromfile(os.path.join(GOLD, "dot11a_dummy_8_ack_40m.i8"), np.int8).reshape(-1, 2)
    out["dummy_8_ack_40m"] = (_pad(v.astype(np.int16) << 8), 6000, ACK_PSDU)
    return out

def fsample6_psdu():
    return np.fromfile(os.path.join(GOLD, "fsample-6.psdu.bin"), np.uint8)

# ---- what the reference holds or computes, as digests (golden/ref_digests.json, made by golden/make_ref_digests.py) ------------------------
def digest(a):
    """SHA-256 of an integer array's values (as little-endian int64, row-major): equal digests = equal shape-flattened values."""
    return hashlib.sha256(np.ascontiguousarray(np.asarray(a).astype("<i8")).tobytes()).hexdigest()

_DIGESTS = None
def ref_digests():
    global _DIGESTS
    if _DIGESTS is None:
        with open(os.path.join(GOLD, "ref_digests.json")) as f: _DIGESTS = json.load(f)
    return _DIGESTS

def ref_table_equals(name, a):
    return digest(a) == ref_digests()["tables"][name]

def fir37_ref_inputs(which=None):
    """(key, int8 [n, 2]) seeded inputs on which the reference's legacy 802.11b transmit filter was run: "cpu" for the oracle's test
    (random, rail-to-rail and zero-stuffed chips), "gpu" for the device's (random, up to 100 000 samples)."""
    if which in (None, "cpu"):
        rng = np.random.default_rng(5)
        for n in (0, 8, 16, 24, 64, 1000 // 8 * 8, 40000):
            for kind in range(3):
                if kind == 0: x = rng.integers(-128, 128, (n, 2)).astype(np.int8)
                elif kind == 1: x = np.where(rng.integers(0, 2, (n, 2)) > 0, 127, -128).astype(np.int8)
                else: x = np.zeros((n, 2), np.int8); x[::4, 0] = np.where(rng.integers(0, 2, (n + 3) // 4) > 0, 127, -128)
                yield f"cpu_n{n}_kind{kind}", x
    if which in (None, "gpu"):
        rng = np.random.default_rng(9)
        for n in (8, 64, 4096, 100000 // 8 * 8):
            yield f"gpu_n{n}", rng.integers(-128, 128, (n, 2)).astype(np.int8)

def fir37_ref_output_equals(key, x, y):
    """y (what the project computed from x) == the reference filter's output for the stored input `key`; x must be that input."""
    want = ref_digests()["fir37"][key]
    assert digest(x) == want["in"], f"{key}: the seeded input differs from the one the reference was run on (numpy's generator stream changed?)"
    return digest(y) == want["out"]
