#!/usr/bin/env python3
"""Parse LUT *data* out of the reference headers (read-only, only in the build container) and
compare it with the closed-form generators used by oracle/ and sora_b200/csrc.

Used two ways:
  * tests/golden/make_ref_digests.py digests the parsed tables into tests/golden/ref_digests.json, which the suite compares the
    closed-form generators below with
  * `python tools/refcheck.py --emit-demap` regenerates sora_b200/csrc/demap_lut.inc (the only
    tables with no closed form: Brick11/src/demapper.h:56-130)
"""
import re, sys, os, math
import numpy as np

REF = os.environ.get("SORA_REFERENCE", "/root/reference")

def _read(rel):
    with open(os.path.join(REF, rel), "r", errors="replace") as f:
        return f.read()

def parse_array(text, name, kind="int"):
    """Return flat list of ints found in the brace initialiser following `name`."""
    m = re.search(re.escape(name) + r"\s*(\[[^\]]*\]\s*)*=\s*\{", text)
    if not m:
        raise KeyError(name)
    i = m.end() - 1
    depth = 0
    j = i
    while True:
        c = text[j]
        if c == '{': depth += 1
        elif c == '}':
            depth -= 1
            if depth == 0: break
        j += 1
    body = text[i:j+1]
    body = re.sub(r"//[^\n]*", "", body)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    body = re.sub(r"__int8\s*\(\s*(0x[0-9A-Fa-f]+)\s*\)", r"\1", body)
    toks = re.findall(r"-?0x[0-9A-Fa-f]+|-?\d+", body)
    return [int(t, 0) for t in toks]

def ref_twiddle(N, M):
    t = _read("kernel/core/inc/fft_lut_twiddle.h")
    name = f"wFFTLUT{N}_{M}" if N != 8 else "wFFTLUT8"
    return np.array(parse_array(t, name), dtype=np.int64).reshape(-1, 2)

def gen_twiddle(N, M):
    j = np.arange(N // 4)
    re_ = np.trunc(32767.0 * np.cos(2 * np.pi * j * M / N))
    im_ = np.trunc(-32767.0 * np.sin(2 * np.pi * j * M / N))
    return np.stack([re_, im_], 1).astype(np.int64)

def ref_bitrev(N):
    t = _read("kernel/core/inc/fft_lut_bitreversal.h")
    return np.array(parse_array(t, f"FFT{N}LUTMap"), dtype=np.int64)

def ref_trig():
    t = _read("kernel/core/inc/intalglut.h")
    s = np.array(parse_array(t, "usin_lut"), dtype=np.int64)
    c = np.array(parse_array(t, "ucos_lut"), dtype=np.int64)
    a = np.array(parse_array(t, "uatan2_lut"), dtype=np.int64)
    return s, c, a

P_REF = 3.141593
def gen_sin():
    i = np.arange(65536)
    return np.round(32767.0 * np.sin(2 * P_REF * i / 65536)).astype(np.int64)
def gen_cos():
    i = np.arange(65536)
    return np.round(32767.0 * np.cos(2 * P_REF * i / 65536)).astype(np.int64)
def gen_atan2():
    y = np.arange(256).astype(np.int8).astype(np.float64)[:, None]
    x = np.arange(256).astype(np.int8).astype(np.float64)[None, :]
    return np.trunc(np.arctan2(y, x) / P_REF * 32768.0).astype(np.int64).reshape(-1)

def ref_vit():
    t = _read("kernel/bb/Brick11/src/viterbilut.h")
    a = np.array(parse_array(t, "VIT_MA"), dtype=np.int64) & 0xFF
    b = np.array(parse_array(t, "VIT_MB"), dtype=np.int64) & 0xFF
    return a.reshape(-1, 16), b.reshape(-1, 16)

def gen_vit():
    A = np.zeros((64, 16), dtype=np.int64); B = np.zeros((64, 16), dtype=np.int64)
    for s in range(8):
        for g in range(8):
            for lane in range(16):
                n = 16 * (g >> 1) + lane
                p = (n >> 1) + 32 * (g & 1)
                b = n & 1
                pb = [(p >> k) & 1 for k in range(6)]
                ea = b ^ pb[1] ^ pb[2] ^ pb[4] ^ pb[5]
                eb = b ^ pb[0] ^ pb[1] ^ pb[2] ^ pb[5]
                A[s * 8 + g, lane] = (14 - 2 * s) if ea else 2 * s
                B[s * 8 + g, lane] = (14 - 2 * s) if eb else 2 * s
    return A, B

def ref_deinterleave(cls):
    t = _read("kernel/bb/Brick11/src/deinterleaver.hpp")
    i0 = t.index("class T11aDeinterleave" + cls)
    nxt = t.find("DEFINE_LOCAL_CONTEXT", i0)
    seg = t[i0: nxt if nxt > 0 else len(t)]
    pairs = re.findall(r"pbOutput\[(\d+)\]\s*=\s*pbInput\[(\d+)\]", seg)
    out = {}
    for o, i in pairs: out[int(o)] = int(i)
    n = max(out) + 1
    return np.array([out[k] for k in range(n)])

def gen_deinterleave(ncbps, nbpsc):
    """out[k] = in[j]: k = index before interleaving (coded order), j = position on air."""
    s = max(nbpsc // 2, 1)
    k = np.arange(ncbps)
    i = (ncbps // 16) * (k % 16) + k // 16
    j = s * (i // s) + (i + ncbps - (16 * i) // ncbps) % s
    return j

# ---- 802.11n tables -----------------------------------------------------------------------------------------------------
def ref_deinterleave_11n(cls):
    """cls e.g. 'BPSK_S0', 'QPSK_S1' (Brick11/src/deinterleaver_11n.hpp)."""
    t = _read("kernel/bb/Brick11/src/deinterleaver_11n.hpp")
    i0 = t.index("class T11nDeinterleave" + cls)
    nxt = t.find("DEFINE_LOCAL_CONTEXT", i0)
    seg = t[i0: nxt if nxt > 0 else len(t)]
    out = {int(o): int(i) for o, i in re.findall(r"pbOutput\[(\d+)\]\s*=\s*pbInput\[(\d+)\]", seg)}
    return np.array([out[k] for k in range(max(out) + 1)])

def ref_demap_11n():
    t = _read("kernel/bb/Brick11/src/dsp_demap.h")
    t = t[t.index("This LUT is constructed"):]
    return {n: np.array(parse_array(t, "dsp_demapper::lookup_table_" + n), dtype=np.int64) for n in ("bpsk", "qpsk")}

def ref_crc8():
    return np.array(parse_array(_read("kernel/core/inc/CRC8.h"), "LUT_CRC8"), dtype=np.int64)

def ref_ltf_masks():
    """-> (lltf_plus[64], htltf_plus[64]) booleans: carriers whose training symbol is +1 (channel_11n.hpp:7-32, 300-325)."""
    t = _read("kernel/bb/Brick11/src/channel_11n.hpp")
    l = np.array(parse_array(t, "_80211_LLTFMask"), dtype=np.int64) & 0xFFFFFFFF
    h = np.array(parse_array(t, "_80211n_HTLTFMask"), dtype=np.int64) & 0xFFFFFFFF
    assert set(l.tolist()) <= {0x0000FFFF, 0xFFFF0000} and set(h.tolist()) <= {0, 0xFFFFFFFF}
    return l == 0xFFFF0000, h == 0

def ref_ht_ndbps():
    """{mcs: (N_CBPS, N_DBPS)} from DOT11N_RATE_PARAMS (ieee80211const.h:35-55)."""
    v = parse_array(_read("kernel/bb/Brick11/src/ieee80211const.h"), "DOT11N_RATE_PARAMS")
    return {m: (v[2 * m], v[2 * m + 1]) for m in range(16)}

def ref_demap_luts():
    t = _read("kernel/bb/Brick11/src/demapper.h")
    return {n: np.array(parse_array(t, "DemapperCore::" + n), dtype=np.uint8)
            for n in ("m_bpsk_lut", "m_qam16_lut2", "m_qam64_lut2", "m_qam64_lut3")}

def rle(a):
    out = []; prev = None; cnt = 0
    for v in a:
        if v == prev: cnt += 1
        else:
            if prev is not None: out.append((int(prev), cnt))
            prev = v; cnt = 1
    out.append((int(prev), cnt))
    return out

def emit_demap(path):
    luts = ref_demap_luts()
    with open(path, "w") as f:
        f.write("// GENERATED by tools/refcheck.py --emit-demap : run-length coded soft-demap tables.\n"
                "// Data (no closed form) from the reference's hand-tuned 3-bit soft demapper,\n"
                "// kernel/bb/Brick11/src/demapper.h:56-130.  Index = (uint8)(clamped value), entry = soft 0..7.\n"
                "// Format: {value, run_length} pairs, runs sum to 256.\n")
        for n, a in luts.items():
            r = rle(a)
            assert sum(c for _, c in r) == 256
            f.write(f"static const unsigned char SB_RLE_{n.upper()}[][2] = {{")
            f.write(",".join("{%d,%d}" % (v, c) for v, c in r))
            f.write("};\n")

def main():
    if "--emit-demap" in sys.argv:
        emit_demap(sys.argv[sys.argv.index("--emit-demap") + 1]); return
    ok = True
    for N in (16, 64, 128):
        for M in (1, 2, 3):
            r = ref_twiddle(N, M); g = gen_twiddle(N, M)
            d = int((r[:len(g)] != g).sum()); print(f"twiddle {N}_{M}: n={len(r)} mismatches={d}"); ok &= d == 0
    r = ref_twiddle(8, 1); print("twiddle8", r.tolist())
    for N in (4, 8, 16, 64, 128):
        r = ref_bitrev(N); print(f"bitrev{N}", r[:16].tolist())
    s, c, a = ref_trig()
    print("sin mism", int((s != gen_sin()).sum()), "cos mism", int((c != gen_cos()).sum()), "atan2 mism", int((a != gen_atan2()).sum()), len(a))
    ra, rb = ref_vit(); ga, gb = gen_vit()
    print("vit", ra.shape, int((ra != ga).sum()), int((rb != gb).sum()))
    for cls, n, b in (("BPSK", 48, 1), ("QPSK", 96, 2), ("QAM16", 192, 4), ("QAM64", 288, 6)):
        r = ref_deinterleave(cls); g = gen_deinterleave(n, b)
        print("deint", cls, len(r), int((r != g).sum()))
    print("ALL OK" if ok else "MISMATCH")

if __name__ == "__main__":
    main()
