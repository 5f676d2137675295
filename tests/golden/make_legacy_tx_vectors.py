#!/usr/bin/env python3
"""Known-answer vectors of the reference's LEGACY 802.11a transmitter at all eight rates, made from the reference's own lookup tables.

The data-path stages of BB11ATxFrameMod are table driven: scrambler
(lutst/scramble_11a.c), convolutional encoder with puncturing (conv_encoder_{1_2,2_3,3_4}.c), interleaver (interleave_{6,12,24,48}m.c),
mapper (mapa_{bpsk,qpsk,16qam,64qam}.c), pilot polarity (pilotsgn.c), preamble (preamble40_11a.c).  This script reads those tables as DATA
and drives them exactly like the reference's C code does (atx_tpl.h Scramble11a, convenc.h ConvEncode_*, ainterleave.h Interleave*, amap.h
Map*_11a, addpilot.h, ofdmsymbol.h Generate*Symbol incl. the two alternating 9 Mbps symbol kinds, atx_tpl_imp.h); the only stage taken from
the oracle is the fixed-point IFFT<128> (oracle `ifft128`, itself pinned by usr/HwVeri/data/ofdm.bin).  Outputs, under tests/golden/legacy_tx/:
  legacy_tx_<kbps>.i8   complex int8 samples (640 + 160 (1 + nsym) + 8) of one frame per rate
  legacy_tx_<kbps>.bin  the frame body (without FCS) that was modulated
  lutst_tables.npz      the tables it read, as data: the CPU suite regenerates every vector from them without the reference tree
The CPU suite then requires oracle/tx11a_legacy.cpp (function-driven restatement) to reproduce every file sample for sample, and the receive
oracle and the GPU to decode every file to its body: table-derived vectors for the rates the reference ships no waveform of (incl. 54 Mbps)."""
import os, re, sys, zlib, numpy as np
HERE = os.path.dirname(os.path.abspath(__file__)); ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
TABLES = ("scramble_11a", "conv_encoder_1_2", "conv_encoder_2_3", "conv_encoder_3_4", "interleave_6m", "interleave_12m",
          "interleave_24m", "interleave_48m", "mapa_bpsk", "mapa_qpsk", "mapa_16qam", "mapa_64qam", "pilotsgn", "preamble40_11a")
STORED = os.path.join(HERE, "legacy_tx", "lutst_tables.npz")

def table(ref, name):
    """One lookup table of kernel/bb/dot11a/lutst/<name>.c under the reference root `ref` (the values of its initialiser)."""
    t = open(os.path.join(ref, "kernel/bb/dot11a/lutst", name + ".c")).read(); body = t[t.index("{", t.index("=")):]
    return np.array([int(x, 0) for x in re.findall(r"-?(?:0x[0-9a-fA-F]+|\d+)", body)], dtype=np.int64)

def stored_tables():
    with np.load(STORED) as z: return {k: z[k].astype(np.int64) for k in TABLES}

def save_tables(T):
    """Each table in the narrowest integer type that holds it (stored_tables() widens them back to int64)."""
    narrow = lambda v: v.astype(next(t for t in (np.int8, np.uint8, np.int16, np.uint16, np.int32, np.uint32) if np.iinfo(t).min <= v.min() and v.max() <= np.iinfo(t).max))
    np.savez_compressed(STORED, **{k: narrow(T[k]) for k in TABLES})

def build(T):
    """T: table name -> int64 values (table() per name, or stored_tables()).  Returns frame(body, kbps) -> int8 [n, 2]."""
    import oracle_py
    SCR = T["scramble_11a"]; PRE = T["preamble40_11a"].reshape(-1, 2)
    MAP = {1: T["mapa_bpsk"].reshape(-1, 8, 2), 2: T["mapa_qpsk"].reshape(-1, 4, 2), 4: T["mapa_16qam"].reshape(-1, 2, 2), 6: T["mapa_64qam"].reshape(-1, 2, 2)}
    IL = {1: (T["interleave_6m"].reshape(-1, 6), 6, 3, 2), 2: (T["interleave_12m"].reshape(-1, 3), 12, 3, 4),
          4: (T["interleave_24m"].reshape(-1, 6), 24, 6, 4), 6: (T["interleave_48m"].reshape(-1, 9), 36, 9, 4)}     # table, input bytes, words used, bytes per word
    def enc12(inp, st):                                    # ConvEncode_1_2
        out = []
        for c in inp:
            w = int(T["conv_encoder_1_2"][(st << 8) | c]); out += [w & 0xFF, w >> 8]; st = c >> 2
        return out, st
    def enc23(inp, st):                                    # ConvEncode_2_3
        out = []
        for i in range(0, len(inp), 2):
            c1, c2 = inp[i], inp[i + 1]
            l1 = int(T["conv_encoder_2_3"][((c1 << 6) | st) & 0xFFFF]); l2 = int(T["conv_encoder_2_3"][((c2 << 6) | (c1 >> 2)) & 0xFFFF])
            out += [l1 & 0xFF, ((l1 >> 8) | (l2 << 4)) & 0xFF, (l2 >> 4) & 0xFF]; st = c2 >> 2
        return out, st
    def enc34(inp, st):                                    # ConvEncode_3_4
        out = []; L = T["conv_encoder_3_4"]
        for i in range(0, len(inp), 3):
            c1, c2, c3 = inp[i], inp[i + 1], inp[i + 2]
            b = [((c1 & 0x3F) << 6) | st, ((c2 & 0xF) << 8) | c1, ((c3 & 0x3) << 10) | (c2 << 2) | (c1 >> 6), (c3 << 4) | (c2 >> 4)]
            out += [int(L[x & 0xFFFF]) & 0xFF for x in b]; st = c3 >> 2
        return out, st
    def enc34_9m(inp, st, kind):                           # ConvEncode_3_4_9MSpecial1 / 2: 36 bits per symbol out of 5 bytes
        c1, c2, c3, c4, c5 = inp; L = T["conv_encoder_3_4"]
        if kind == 1:
            b = [((c1 & 0x3F) << 6) | st, ((c2 & 0xF) << 8) | c1, ((c3 & 0x3) << 10) | (c2 << 2) | (c1 >> 6), (c3 << 4) | (c2 >> 4), ((c4 & 0x3F) << 6) | (c3 >> 2), ((c5 & 0xF) << 8) | c4]
            st = ((c5 & 0xF) << 2) | ((c4 >> 6) & 0x3)
        else:
            b = [((c2 & 0x3) << 10) | ((c1 & 0xF0) << 2) | st, (c2 << 4) | (c1 >> 4), ((c3 & 0x3F) << 6) | (c2 >> 2), ((c4 & 0xF) << 8) | c3, ((c5 & 0x3) << 10) | (c4 << 2) | (c3 >> 6), (c5 << 4) | (c4 >> 4)]
            st = c5 >> 2
        return [int(L[x & 0xFFFF]) & 0xFF for x in b], st
    def interleave(enc, nb):
        tab, nin, nw, bpw = IL[nb]; acc = [0] * nw
        for j in range(nin):
            row = tab[(j << 8) + enc[j]]
            for k in range(nw): acc[k] |= int(row[k])
        out = []
        for k in range(nw): out += [(acc[k] >> (8 * b)) & 0xFF for b in range(bpw)]
        return out
    def mapper(il, nb):
        if nb == 1: return np.concatenate([MAP[1][il[i]] for i in range(6)])
        if nb == 2: return np.concatenate([MAP[2][il[i]] for i in range(12)])
        if nb == 4: return np.concatenate([MAP[4][il[i]] for i in range(24)])
        out = []
        for i in range(12):
            u = il[3 * i] | (il[3 * i + 1] << 8) | (il[3 * i + 2] << 16)
            out += [MAP[6][u & 0xFFF], MAP[6][(u >> 12) & 0xFFF]]
        return np.concatenate(out)
    def sat(a): return np.clip(a, -32768, 32767)
    def wrap(a): return ((np.asarray(a, np.int64) + 32768) % 65536) - 32768
    def symbol(mapped48, neg, last):
        f = np.zeros((64, 2), np.int64); it = iter(mapped48)
        for i in list(range(38, 64)) + list(range(1, 27)):
            if i in (43, 57, 7, 21): continue
            f[i] = next(it)
        one = 32 * 335; s = -1 if neg else 1
        f[7] = [s * one, 0]; f[21] = [-s * one, 0]; f[57] = [s * one, 0]; f[43] = [s * one, 0]
        t = np.zeros((128, 2), np.int16); t[:32] = f[:32]; t[96:] = f[32:]
        o = oracle_py.ifft128(t).astype(np.int64)
        sym = np.zeros((160, 2), np.int64); sym[32:] = wrap(o * 4); sym[:32] = sym[128:]
        sym[0] >>= 2; sym[1] >>= 1; sym[2] = wrap(sym[2] - (sym[2] >> 2))
        sym[:4] = sat(sym[:4] + last); sym[0] = wrap(sym[0] + last[0])
        nl = np.zeros((4, 2), np.int64); nl[0] = wrap(sym[32] - (sym[32] >> 2)); nl[1] = sym[33] >> 1; nl[2] = sym[34] >> 2
        return np.clip(sym >> 6, -128, 127).astype(np.int8), nl
    RATE = {6000: (0xB, 1, 24, "12"), 9000: (0xF, 1, 36, "9m"), 12000: (0xA, 2, 48, "12"), 18000: (0xE, 2, 72, "34"),
            24000: (0x9, 4, 96, "12"), 36000: (0xD, 4, 144, "34"), 48000: (0x8, 6, 192, "23"), 54000: (0xC, 6, 216, "34")}
    def frame(body, kbps):
        code, nb, dbps, enc = RATE[kbps]
        psdu = bytes(body) + zlib.crc32(bytes(body)).to_bytes(4, "little"); L = len(psdu)
        nsym = (16 + 6 + 8 * L + dbps - 1) // dbps
        out = [np.clip(PRE >> 6, -128, 127).astype(np.int8)]
        pt = PRE[512:515]; last = np.zeros((4, 2), np.int64); last[0] = pt[0] - (pt[0] >> 2); last[1] = pt[1] >> 1; last[2] = pt[2] >> 2
        sig = code | (L << 5); p = sig ^ (sig >> 16); p ^= p >> 8; p ^= p >> 4; p ^= p >> 2; p ^= p >> 1; sig |= (p & 1) << 17
        e, _ = enc12([sig & 0xFF, (sig >> 8) & 0xFF, (sig >> 16) & 0xFF], 0)
        s, last = symbol(mapper(interleave(e, 1), 1), 0, last); out.append(s)
        total = nsym * dbps // 8 + (1 if kbps == 9000 and nsym % 2 else 0)          # bytes the scrambler fills (9 Mbps symbols take 4.5 bytes)
        reg = 0xFF; sc = []
        for i in range(total + 8):
            reg = int(SCR[reg >> 1])
            src = 0 if i < 2 else (psdu[i - 2] if i - 2 < L else 0)
            v = src ^ reg
            if i == 2 + L: v = reg & 0xC0
            sc.append(v)
        st = 0; pi = 0; pos = 0
        for n in range(nsym):
            neg = T["pilotsgn"][pi] != 0; pi = (pi + 1) % 127
            if enc == "12": e, st = enc12(sc[pos:pos + dbps // 8], st); pos += dbps // 8
            elif enc == "23": e, st = enc23(sc[pos:pos + 24], st); pos += 24
            elif enc == "34": e, st = enc34(sc[pos:pos + dbps // 8], st); pos += dbps // 8
            else:                                                                      # 9 Mbps: Generate9MSymbol1 / 2 alternate, 4 then 5 bytes further (atx_9.c)
                e, st = enc34_9m(sc[pos:pos + 5], st, 1 if n % 2 == 0 else 2); pos += 4 if n % 2 == 0 else 5
            s, last = symbol(mapper(interleave(e, nb), nb), neg, last); out.append(s)
        tail = np.zeros((8, 2), np.int8); tail[:4] = np.clip(last >> 6, -128, 127)
        out.append(tail)
        return np.concatenate(out)
    return frame

if __name__ == "__main__":
    # usage: python tests/golden/make_legacy_tx_vectors.py REFERENCE_ROOT
    T = {k: table(sys.argv[1], k) for k in TABLES}
    d = os.path.join(HERE, "legacy_tx"); os.makedirs(d, exist_ok=True)
    save_tables(T)
    frame = build(T)
    rng = np.random.default_rng(0x11A)
    for kbps, n in ((6000, 40), (9000, 57), (12000, 64), (18000, 77), (24000, 100), (36000, 131), (48000, 190), (54000, 211)):
        body = rng.integers(0, 256, n).astype(np.uint8)
        w = frame(body, kbps)
        w.tofile(os.path.join(d, f"legacy_tx_{kbps}.i8")); body.tofile(os.path.join(d, f"legacy_tx_{kbps}.bin"))
        print(kbps, n, "bytes ->", len(w), "samples")
