"""The glue's service database (welle.io_b200/host/fig-db.h) against the reference's FIBProcessor (backend/fib-processor.cpp, compiled
unmodified into oracle/_ref): the same FIB sequences go into both, the text dumps of ensemble / services / components / sub-channels /
labels / date-time and the order of the FIG-derived callbacks must be identical.  CPU only."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT


def crc16(data):
    crc = 0xFFFF
    for b in data:
        crc ^= b << 8
        for _ in range(8):
            crc = ((crc << 1) ^ 0x1021) & 0xFFFF if crc & 0x8000 else (crc << 1) & 0xFFFF
    return crc ^ 0xFFFF


# ---- FIG encoders (ETSI EN 300 401 clause 6 and 8): each returns the complete FIG (header byte included)
def fig0(ext, body, pd=0, cn=0, oe=0):
    body = bytes(body)
    return bytes([(0 << 5) | (1 + len(body)), (cn << 7) | (oe << 6) | (pd << 5) | ext]) + body


def fig0_0(eid, change=0, cif_hi=3, cif_lo=17, occ=0):
    b = [eid >> 8, eid & 0xFF, (change << 6) | cif_hi, cif_lo]
    if change:
        b.append(occ)
    return fig0(0, b)


def subch_short(subch, start, table_index):
    return [(subch << 2) | (start >> 8), start & 0xFF, table_index & 0x3F]


def subch_long(subch, start, option, level, size):
    return [(subch << 2) | (start >> 8), start & 0xFF, 0x80 | (option << 4) | ((level - 1) << 2) | (size >> 8), size & 0xFF]


def service_entry(sid, comps, pd):
    b = list(sid.to_bytes(4 if pd else 2, "big")) + [len(comps)]
    for c in comps:
        if c["tmid"] == 3:
            b += [(3 << 6) | (c["scid"] >> 6), ((c["scid"] & 0x3F) << 2) | (c["ps"] << 1) | c["ca"]]
        else:
            b += [(c["tmid"] << 6) | c["ty"], (c["subch"] << 2) | (c["ps"] << 1) | c.get("ca", 0)]
    return b


def fig0_3_entry(scid, dg, dscty, subch, addr):      # 7 bytes: the reference strides 56 bits per entry (CAOrg present)
    return [scid >> 4, ((scid & 0xF) << 4) | 1, (dg << 7) | dscty, (subch << 2) | (addr >> 8), addr & 0xFF, 0x12, 0x34]


def fig0_9(lto_sign, lto_hours, lto_half, ecc):
    return fig0(9, [(lto_sign << 5) | (lto_hours << 1) | lto_half, ecc, 0x01])


def fig0_10(mjd, hours, minutes, seconds=None):
    v = (mjd << 14) | ((1 if seconds is not None else 0) << 11) | (hours << 6) | minutes
    b = list(v.to_bytes(4, "big"))
    if seconds is not None:
        b += [(seconds << 2), 0]
    return fig0(10, b)


def fig0_17_entry(sid, lang, pty, cc=None):
    b = [sid >> 8, sid & 0xFF, (0x20 if lang is not None else 0) | (0x10 if cc is not None else 0)]
    if lang is not None:
        b.append(lang)
    b.append(pty & 0x1F)
    if cc is not None:
        b.append(cc)
    return b


def fig1(ext, ident, label, flag, charset=0, oe=0):
    lab = label.encode("latin1")[:16].ljust(16, b" ")
    body = bytes([(charset << 4) | (oe << 3) | ext]) + bytes(ident) + lab + flag.to_bytes(2, "big")
    return bytes([(1 << 5) | len(body)]) + body


def fig2(ext, ident, data, toggle, seg, rfu=0):
    body = bytes([(toggle << 7) | (seg << 4) | (rfu << 3) | ext]) + bytes(ident) + bytes(data)
    return bytes([(2 << 5) | len(body)]) + body


def pack_fibs(figs, rng=None):
    """FIGs -> 32-byte FIBs (30 data bytes, 0xFF end marker / padding, CRC)"""
    fibs, cur = [], b""
    for f in figs:
        assert len(f) <= 30
        if len(cur) + len(f) > 30:
            fibs.append(cur); cur = b""
        cur += f
    if cur:
        fibs.append(cur)
    out = []
    for d in fibs:
        d = d.ljust(30, b"\xff")
        out.append(d + crc16(d).to_bytes(2, "big"))
    return np.frombuffer(b"".join(out), np.uint8).reshape(-1, 32).copy()


@pytest.fixture(scope="module")
def dumps(ref):
    host = C.CDLL(os.path.join(ROOT, "welle.io_b200", "libwelle_b200_host.so"))

    def run(fibs):
        fibs = np.ascontiguousarray(fibs, np.uint8)
        buf = C.create_string_buffer(1 << 18)
        n = host.welle_b200_figdb_dump(fibs.ctypes.data_as(C.c_void_p), len(fibs), buf, len(buf))
        assert n >= 0
        return buf.value.decode("latin1"), ref.fib_dump(fibs)
    return run


def build_ensemble(rng, n_services=5):
    eid = int(rng.integers(1, 0xFFFF))
    figs = [fig0_0(eid), fig0_9(int(rng.integers(0, 2)), int(rng.integers(0, 12)), int(rng.integers(0, 2)), int(rng.integers(0, 256)))]
    sub_entries, start = [], 0
    subch_ids = rng.permutation(64)[: 2 * n_services + 2].tolist()
    for k, sc in enumerate(subch_ids):
        if k % 3 == 0:
            ti = int(rng.integers(0, 64)); sub_entries.append(subch_short(sc, start, ti)); start += 40
        else:
            sub_entries.append(subch_long(sc, start, int(rng.integers(0, 2)), int(rng.integers(1, 5)), int(rng.integers(6, 120)))); start += 50
    for i in range(0, len(sub_entries), 6):
        figs.append(fig0(1, sum(sub_entries[i: i + 6], []), pd=int(rng.integers(0, 2))))
    services = []
    for s in range(n_services):
        pd = int(s % 3 == 2)
        sid = int(rng.integers(0x1000, 0xFFFF)) if not pd else int(rng.integers(0xE0100000, 0xE01FFFFF))
        comps = []
        for c in range(int(rng.integers(1, 4))):
            tm = [0, 0, 1, 3][int(rng.integers(0, 4))]
            if tm == 3:
                comps.append(dict(tmid=3, scid=int(rng.integers(1, 4095)), ps=int(c == 0), ca=int(rng.integers(0, 2))))
            else:
                comps.append(dict(tmid=tm, ty=int(rng.choice([0, 63, 5, 60])), subch=int(subch_ids[(2 * s + c) % len(subch_ids)]), ps=int(c == 0)))
        services.append((sid, comps, pd))
        figs.append(fig0(2, service_entry(sid, comps, pd), pd=pd))
    # packet component details, languages, FEC, programme types
    for sid, comps, pd in services:
        for c in comps:
            if c["tmid"] == 3:
                figs.append(fig0(3, fig0_3_entry(c["scid"], int(rng.integers(0, 2)), int(rng.integers(0, 64)), int(rng.choice(subch_ids)), int(rng.integers(0, 1024)))))
    figs.append(fig0(5, sum([[sc & 0x3F, int(rng.integers(0, 128))] for sc in subch_ids[:5]], []) + [0x80 | 0x01, 0x23, 0x09]))
    figs.append(fig0(14, [(sc << 2) | int(rng.integers(0, 4)) for sc in subch_ids[:6]]))
    figs.append(fig0(17, sum([fig0_17_entry(sid & 0xFFFF, int(rng.integers(0, 100)) if k % 2 else None, int(rng.integers(0, 32)), 0x05 if k % 3 == 0 else None)
                              for k, (sid, _, pd) in enumerate(services) if not pd], [])))
    figs.append(fig0_10(int(rng.integers(50000, 62000)), int(rng.integers(0, 24)), int(rng.integers(0, 60)), int(rng.integers(0, 60)) if rng.integers(0, 2) else None))
    # labels
    figs.append(fig1(0, eid.to_bytes(2, "big"), "Ensemble %04X" % eid, 0xFF00))
    for k, (sid, comps, pd) in enumerate(services):
        if pd:
            figs.append(fig1(5, sid.to_bytes(4, "big"), "Data %d" % k, 0xF000))
        else:
            figs.append(fig1(1, sid.to_bytes(2, "big"), "Service %d \xe4\xf6" % k, 0x0FF0, charset=int(rng.choice([0, 0, 15]))))
        if len(comps) > 1:
            ident = [(pd << 7) | 1] + list(sid.to_bytes(4 if pd else 2, "big"))
            figs.append(fig1(4, ident, "Comp %d/1" % k, 0x00F0))
    # FIG 2 extended labels: ensemble in two segments, one service, one component
    txt = "Erweitertes Label äöü".encode("utf8")
    figs.append(fig2(0, eid.to_bytes(2, "big"), bytes([0x10, 0xFF, 0x00]) + txt[:10], 0, 0))
    figs.append(fig2(0, eid.to_bytes(2, "big"), txt[10:], 0, 1))
    sid0 = next(s for s, _, pd in services if not pd)
    figs.append(fig2(1, sid0.to_bytes(2, "big"), bytes([0x00, 0x80, 0x00]) + b"FIG2 service", 1, 0))
    figs.append(fig2(1, sid0.to_bytes(2, "big"), bytes([0x80]) + "ucs2".encode("utf-16-be"), 0, 0, rfu=1))
    return figs


@pytest.mark.parametrize("seed", range(8))
def test_ensemble_database_matches_reference(dumps, seed):
    rng = np.random.default_rng(seed)
    figs = build_ensemble(rng)
    # every FIG twice (services are listed from their second sighting), in two differently shuffled passes, then labels again
    seq = [figs[i] for i in rng.permutation(len(figs))] + figs + [figs[i] for i in rng.permutation(len(figs))]
    mine, theirs = dumps(pack_fibs(seq))
    assert mine == theirs
    assert mine.count("\nS ") >= 4 and "cb serviceDetected" in mine and "cb dateTime" in mine and "\nXE " in mine


def test_ensemble_change_and_restart(dumps):
    rng = np.random.default_rng(99)
    a = build_ensemble(rng, 3)
    b = [fig0_0(0x4242, change=1, occ=7)] + build_ensemble(rng, 2)
    mine, theirs = dumps(pack_fibs(a + a + b + b + [fig0_0(0x4242, change=3, occ=1)]))
    assert mine == theirs and "cb restartService" in mine and mine.count("cb newEnsemble") >= 2


def test_random_fig_bodies(dumps):
    """well-formed FIG framing with random bodies (types 0-2, every extension): the two parsers must walk them identically"""
    rng = np.random.default_rng(2024)
    base = build_ensemble(rng, 4)
    for trial in range(40):
        figs = list(base) + list(base)
        for _ in range(60):
            t = int(rng.integers(0, 3)); ln = int(rng.integers(2, 28))
            body = rng.integers(0, 256, ln).astype(np.uint8).tolist()
            if t == 2 and (body[0] & 0x70) == 0 and ln < 10:
                continue                      # a too-short first FIG 2 segment makes the reference throw; the glue ignores the FIG
            if t == 0 and (body[0] & 0x1F) in (1, 13):
                continue                      # FIG 0/1: strides past the FIB in both; FIG 0/13: the reference's 16-bit bit offset overflows on a
                                              # malformed application list and it reads far out of bounds (crash)
            figs.append(bytes([(t << 5) | ln]) + bytes(body))
        mine, theirs = dumps(pack_fibs(figs))
        if "exception" in theirs:
            continue
        assert mine == theirs, trial


def test_tii_analysis_matches_reference(oracle, ref):
    """welle.io_b200/host/tii.h (pattern analysis of the glue) against the unmodified TIIDecoder (tii-decoder.cpp) frame by frame: two
    transmitters (different comb / pattern / delay) in the null symbol, noise, 12 frames -> the same measurements (comb, pattern, delay in
    samples, error sum) in the same order.  The glue's analyser starts from the two spectra - here made with the oracle's FFT, which is
    bit-identical to the reference's fft::Forward (tests/test_oracle_vs_ref.py); on the GPU they are tap 4 (tests/test_gpu_glue.py)."""
    import ctypes as C
    import dabtx
    lib = C.CDLL(os.path.join(ROOT, "welle.io_b200", "libwelle_b200_host.so"))
    lib.welle_b200_tii_run.restype = C.c_int
    tx = dabtx.DabTx(seed=0x711)
    tx.tii = [(4, 17, 23, 0.5), (11, 52, 140, 0.35)]
    sig = dabtx.add_awgn(tx.frames(13), 25.0, seed=4)
    TF, TU, TNULL = 196608, 2048, 2656
    nulls, prss = [], []
    for f in range(1, 13):
        base = f * TF
        nulls.append(sig[base: base + TNULL]); prss.append(sig[base + TNULL + 504: base + TNULL + 504 + TU])     # aligned PRS (useful part)
    # the reference pairs the PRS of frame n with the null symbol that FOLLOWS it
    nulls, prss = np.stack(nulls[1:]), np.stack(prss[:-1])
    want = ref.tii_run(nulls, prss)
    assert len(want) >= 2 and {(int(w[0]), int(w[1])) for w in want} == {(4, 17), (11, 52)}
    assert {(4, 23), (11, 140)} <= {(int(w[0]), int(w[2])) for w in want}, want          # the delays come out
    nspec = np.stack([oracle.fft(x[TNULL - TU:]) for x in nulls]); pspec = np.stack([oracle.fft(x) for x in prss])
    out = np.zeros(4 * 64, np.float32)
    k = lib.welle_b200_tii_run(nspec.ctypes.data_as(C.c_void_p), pspec.ctypes.data_as(C.c_void_p), len(nulls), out.ctypes.data_as(C.c_void_p), 64)
    got = [tuple(out[4 * i: 4 * i + 4].tolist()) for i in range(k)]
    assert got == want, (got, want)
