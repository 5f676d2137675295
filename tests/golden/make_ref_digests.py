#!/usr/bin/env python3
"""SHA-256 digests of what the reference holds or computes, for the tests that compare the project with it: lookup tables parsed out of its
headers (tools/refcheck.py), a few constants of its 802.11b transmitter, its fsample-6.dmp capture, and the output of its legacy 802.11b
transmit filter (oracle/_ref, built from the same tree by oracle/build_ref.sh) for the seeded inputs of the filter tests.  The tests hash
what the project computes and compare (golden_vectors.digest); the reference itself is needed only to rerun this script.

  oracle/build_ref.sh REFERENCE_ROOT && python tests/golden/make_ref_digests.py REFERENCE_ROOT      -> tests/golden/ref_digests.json"""
import json, os, re, sys, hashlib
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__)); ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tools")); sys.path.insert(0, os.path.dirname(HERE))
import golden_vectors as gv, oracle_py

def header_tables(rc):
    t = {}
    for N in (16, 32, 64, 128):
        for M in (1, 2, 3):
            t[f"twiddle_{N}_{M}"] = rc.ref_twiddle(N, M)[: N // 4]
    t["twiddle_8"] = np.array(rc.parse_array(rc._read("kernel/core/inc/fft_lut_twiddle.h"), "wFFTLUT8")).reshape(-1, 2)
    for N in (64, 128):
        t[f"bitrev_{N}"] = rc.ref_bitrev(N)
    t["usin_lut"], t["ucos_lut"], t["uatan2_lut"] = rc.ref_trig()
    t["VIT_MA"], t["VIT_MB"] = rc.ref_vit()
    for cls in ("BPSK", "QPSK", "QAM16", "QAM64"):
        t[f"deint11a_{cls}"] = rc.ref_deinterleave(cls)
    t["LTS_Sequence_11a"] = rc.parse_array(rc._read("kernel/bb/Brick11/src/channel_11a.hpp"), "LTS_Sequence_11a")
    t["PilotSgn"] = rc.parse_array(rc._read("kernel/bb/Brick11/src/pilot.hpp"), "PilotSgn")
    t.update(rc.ref_demap_luts())
    d = rc._read("kernel/bb/Brick11/src/dsp_demap.h"); d = d[d.index("This LUT is constructed"):]
    for n in ("bpsk", "qpsk", "16qam1", "16qam2", "64qam1", "64qam2", "64qam3"):
        t[f"demap11n_{n}"] = rc.parse_array(d, "dsp_demapper::lookup_table_" + n)
    t["LUT_CRC8"] = rc.ref_crc8()
    for cls in ("BPSK", "QPSK", "QAM16", "QAM64"):
        for s in range(2):
            t[f"deint11n_{cls}_S{s}"] = rc.ref_deinterleave_11n(f"{cls}_S{s}")
    t["lltf_plus"], t["htltf_plus"] = rc.ref_ltf_masks()
    t["DOT11N_NDBPS_MCS8_14"] = [rc.ref_ht_ndbps()[m][1] for m in range(8, 15)]
    return t

def tx11n_tables(ref):
    """The 802.11n preamble tables (pairs {re, im}) and the 127-entry HT pilot polarity table."""
    src = os.path.join(ref, "kernel/bb/Brick11/src")
    def pairs(path, name):
        s = open(os.path.join(src, path)).read(); i = s.index(name + "[] ="); j = s.index("};", i)
        return np.array(re.findall(r"\{\s*(-?\d+)\s*,\s*(-?\d+)\s*\}", s[i:j]), dtype=np.int64)
    s = open(os.path.join(src, "_b_dot11_pilot.h")).read(); i = s.index("dot11_ofdm_pilot::_pilot_sign[pilot_size] ="); j = s.index("};", i)
    return {"L_STF": pairs("_b_lstf.h", "L_STF::_stf"), "L_LTF": pairs("_b_lltf.h", "L_LTF::_ltf"), "HT_STF": pairs("_b_htstf.h", "HT_STF::_stf"),
            "HT_LTF": pairs("_b_htltf.h", "HT_LTF::_ltf"), "_pilot_sign": [int(v) for v in re.findall(r"-?\d+", s[s.index("{", i):j])]}

def tx11b_constants(ref):
    """Barker code, DQPSK / CCK phase tables ({re, im} pairs) and the long-preamble PLCP constants of the reference's 802.11b transmitter."""
    def c_array(path, name):
        s = open(os.path.join(ref, path)).read(); i = s.index(name + "[] ="); j = s.index("};", i)
        return [int(v) for v in re.findall(r"-?\d+", s[s.index("{", i):j])]
    plcp = open(os.path.join(ref, "kernel/inc/dot11_plcp.h")).read()
    define = lambda n: [int(re.search(r"#define\s+" + n + r"\s+(0x[0-9A-Fa-f]+|\d+)", plcp).group(1), 0)]
    return {"Barker11": c_array("kernel/bb/Brick11/src/barkerspread.hpp", "Barker11"),
            "DQPSKEncode": c_array("kernel/bb/Brick11/src/cck.hpp", "DQPSKEncode"), "CCK11D3D2": c_array("kernel/bb/Brick11/src/cck.hpp", "CCK11D3D2"),
            "DOT11B_PLCP_LONG_TX_SCRAMBLER_REGISTER": define("DOT11B_PLCP_LONG_TX_SCRAMBLER_REGISTER"),
            "DOT11B_PLCP_LONG_PREAMBLE_SFD": define("DOT11B_PLCP_LONG_PREAMBLE_SFD")}

def fir37_outputs():
    """The reference filter body on the seeded inputs of test_cpu_oracle_tx11b_legacy / test_gpu_tx11b_legacy (gv.fir37_ref_inputs)."""
    assert oracle_py.ref_fir37_available(), "build oracle/_ref first (oracle/build_ref.sh REFERENCE_ROOT)"
    return {key: {"in": gv.digest(x), "out": gv.digest(oracle_py.ref_fir37(x))} for key, x in gv.fir37_ref_inputs()}

if __name__ == "__main__":
    ref = os.path.abspath(sys.argv[1])
    import refcheck as rc
    rc.REF = ref
    tables = header_tables(rc); tables.update(tx11n_tables(ref)); tables.update(tx11b_constants(ref))
    out = {"tables": {k: gv.digest(v) for k, v in sorted(tables.items())},
           "files": {"kernel/test-data/fsample-6.dmp": hashlib.sha256(open(os.path.join(ref, "kernel/test-data/fsample-6.dmp"), "rb").read()).hexdigest()},
           "fir37": fir37_outputs()}
    with open(os.path.join(HERE, "ref_digests.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True); f.write("\n")
    print(len(out["tables"]), "tables,", len(out["fir37"]), "filter cases")
