"""Pins the C oracle (oracle/dab_oracle.c) against the UNMODIFIED reference (oracle/_ref/libwelle_ref.so, KISS-FFT build, compiled
from the reference's sources by oracle/Makefile).  Integer stages and - because the oracle keeps the reference's float operation
order - the float stages too must be bit-identical.  Where the reference build is not available, its results recorded in
tests/golden/ref_calls.npz stand in for it (tests/refcalls.py)."""
import numpy as np
import pytest

import dabtx
from refcalls import same

TU, TS, TF, TNULL = 2048, 2552, 196608, 2656


@pytest.fixture(scope="module")
def sig():
    tx = dabtx.DabTx(seed=0xDAB)
    return tx, tx.frames(14)


def test_tables(oracle, ref):
    assert np.array_equal(oracle.perm_table(), ref.perm_table())
    assert np.array_equal(dabtx.perm_table(), ref.perm_table())
    assert np.array_equal(oracle.prs_table().view(np.uint32), ref.prs_table().view(np.uint32))
    assert np.abs(dabtx.prs_spectrum() - ref.prs_table()).max() < 1e-6
    assert np.array_equal(oracle.pcodes(), ref.pcodes()) and np.array_equal(dabtx.pcodes(), ref.pcodes())
    # KATs printed by the reference's classes (SURVEY.md §9)
    assert list(ref.perm_table()[:12]) == [-513, -14, 329, 692, -733, 13, 680, 273, -36, 43, 85, -432] and ref.perm_table()[1535] == 197
    assert "".join(map(str, oracle.prbs(32))) == "00000111101111100010111001100100"


def test_fft_bit_exact(oracle, ref):
    rng = np.random.default_rng(1)
    for _ in range(3):
        x = (rng.standard_normal(2048) + 1j * rng.standard_normal(2048)).astype(np.complex64)
        assert same(oracle.fft(x), ref.fft(x))
        assert same(oracle.ifft_scaled(x), ref.fft(x, True))


def test_find_index_and_demod(oracle, ref, sig):
    tx, iq = sig
    base = 3 * TF + TNULL
    for off in (199, 100, 350, -3000):
        v = iq[base - off: base - off + TU]
        i1, c1 = oracle.find_index(v); i2, c2 = ref.find_index(v)
        assert i1 == i2 and same(c1, c2)
    st = base + 305
    prs, syms = iq[st: st + TU], iq[st + TU: st + TU + 75 * TS]
    s1, r1 = oracle.demod_frame(prs, syms, True); s2, r2 = ref.demod_frame(prs, syms, True)
    assert same(s1, s2) and same(r1, r2)
    # (s1 == s2: both FIC decoders get the same softbits)
    fb1, ok1 = oracle.fic_decode(s1[:3].reshape(-1)); fb2, ok2 = ref.fic_decode(s1[:3].reshape(-1))
    assert np.array_equal(fb1, fb2) and np.array_equal(ok1, ok2) and ok1.all()
    assert np.array_equal(np.packbits(fb1[0]), dabtx.fib_bytes(tx))


def test_viterbi(oracle, ref):
    rng = np.random.default_rng(5)
    for nb in (768, 2304, 192, 24 * 64):
        soft = rng.integers(-128, 128, (nb + 6) * 4).astype(np.int8)
        assert np.array_equal(oracle.viterbi(soft, nb), ref.viterbi(soft, nb))
        bits = rng.integers(0, 2, nb).astype(np.uint8)
        enc = oracle.conv_encode(bits)
        assert np.array_equal(enc, dabtx.conv_encode(bits))
        s = np.clip((enc.astype(np.float32) * 2 - 1) * 40 + rng.standard_normal(enc.size) * 45, -127, 127).astype(np.int8)
        d1, d2 = oracle.viterbi(s, nb), ref.viterbi(s, nb)
        assert np.array_equal(d1, d2)


@pytest.mark.parametrize("cfg", [(96, 1, 3), (64, 1, 1), (8, 1, 2), (32, 1, 2), (128, 1, 4), (32, 0, 1), (64, 0, 2), (96, 0, 3), (128, 0, 4)])
def test_eep(oracle, ref, cfg):
    br, pa, lv = cfg
    rng = np.random.default_rng(br * 10 + lv)
    p = oracle.prot_eep(br, pa, lv)
    assert p.in_bits == dabtx.eep_cu(br, bool(pa), lv) * 64
    soft = rng.integers(-127, 128, p.in_bits).astype(np.int8)
    assert same(oracle.msc_deconvolve(p, soft, True), ref.eep_deconvolve(br, pa, lv, soft, True))


@pytest.mark.parametrize("cfg", [(32, 5), (48, 3), (128, 1), (192, 2), (384, 1), (80, 1), (64, 4), (56, 2), (320, 4)])
def test_uep(oracle, ref, cfg):
    br, lv = cfg
    rng = np.random.default_rng(br * 10 + lv)
    p = oracle.prot_uep(br, lv)
    soft = rng.integers(-127, 128, p.in_bits).astype(np.int8)
    assert same(oracle.msc_deconvolve(p, soft, True), ref.uep_deconvolve(br, lv, soft, True))


def test_rs_and_crc(oracle, ref):
    rng = np.random.default_rng(7)
    d = np.arange(110, dtype=np.uint8)
    assert " ".join("%02X" % x for x in oracle.rs_encode(d)) == "A2 8A 69 0C EA 30 BD D4 A3 5C"      # reference KAT (SURVEY §9)
    assert np.array_equal(oracle.rs_encode(d), ref.rs_encode(d)) and np.array_equal(dabtx.rs_parity(d), ref.rs_encode(d))
    received = []
    for trial in range(1500):
        data = rng.integers(0, 256, 110).astype(np.uint8)
        cw = np.concatenate([data, oracle.rs_encode(data)])
        ne = int(rng.integers(0, 9)); pos = rng.choice(120, ne, replace=False)
        e = cw.copy(); e[pos] ^= rng.integers(1, 256, ne).astype(np.uint8)
        if trial % 10 == 0:
            e = rng.integers(0, 256, 120).astype(np.uint8)
        received.append(e)
    received = np.stack(received)
    b_res, b_cw, b_pos = ref.rs_decode_codewords(received)
    a_cw = []
    for trial, e in enumerate(received):
        a = oracle.rs_decode_codeword(e)
        assert a[0] == b_res[trial], trial
        if a[0] > 0:
            assert np.array_equal(a[2][:a[0]], b_pos[trial][:a[0]]), trial
        a_cw.append(a[1])
    assert same(np.stack(a_cw), b_cw)
    assert oracle.crc_fire(np.arange(9, dtype=np.uint8)) == ref.crc_fire(np.arange(9, dtype=np.uint8)) == 0x3F9E
    k = np.frombuffer(b"123456789", np.uint8)
    assert oracle.crc_ccitt(k) == ref.crc_ccitt(k) == 0xD64E
    z = np.zeros(256, np.uint8)
    assert oracle.check_crc_bits(z) == ref.check_crc_bits(z) == 0


def test_superframe_filter(oracle, ref):
    rng = np.random.default_rng(8)
    tx = dabtx.DabTx(seed=3)
    stream = np.concatenate([tx.superframe() for _ in range(6)])
    bad = stream.copy(); idx = rng.choice(len(bad), 300, replace=False); bad[idx] ^= rng.integers(1, 256, 300).astype(np.uint8)
    for s in (stream, bad):
        fr = np.concatenate([rng.integers(0, 256, (2, 288)).astype(np.uint8), s.reshape(-1, 288)])
        ev, outs = oracle.superframe_filter(fr); fec, auerr, good = ref.superframe_filter(fr)
        assert np.array_equal(np.array([[e["uncorr"], e["corr"]] for e in ev]), fec)
        assert auerr == sum(e["num_aus"] - bin(e["au_ok"]).count("1") for e in ev if e["sync"])
        a = oracle.rs_decode_superframe(s[:1440]); b = ref.rs_decode_superframe(s[:1440])
        assert np.array_equal(a[0], b[0]) and a[1:] == b[1:]


def test_dabaudio_chain(oracle, ref, tmp_path):
    """time de-interleaver + EEP + Viterbi + dispersal + byte pack through the reference's DabAudio thread"""
    rng = np.random.default_rng(11)
    p = oracle.prot_eep(96, 1, 3)
    cifs = rng.integers(-127, 128, (24, 72 * 64)).astype(np.int8)
    data, rs = ref.dabaudio_chain(cifs, 96, True, 3, dabplus=True, dump_path=str(tmp_path / "chain.msc"))
    de = oracle.deinterleave(cifs)
    mine = np.concatenate([oracle.pack_bits(oracle.msc_deconvolve(p, d, True)) for d in de])
    n = min(len(mine), len(data))
    assert n >= 7 * 288 and np.array_equal(mine[:n], data[:n])


def test_closed_loop_receiver(oracle, ref, sig, tmp_path):
    """oracle.rx_run == reference RadioReceiver (flow-controlled input) on the same stream: FIBs, logical frames, RS events"""
    tx, iq = sig
    e = ref.e2e(iq, disable_coarse=True, select_at_fib=24, dump_path=str(tmp_path / "e2e.msc"))
    p = oracle.prot_eep(96, 1, 3)
    m = oracle.rx_run(iq, prot=p, start_cu=0, len_cu=72, select_after_frames=1, disable_coarse=True)
    assert e["select_ok"] == 1 and len(e["fibs"]) >= 12 * 11
    assert np.array_equal(m["fibs"][:len(e["fibs"])], e["fibs"]) and e["fibs"][:, 0].all()
    n = min(len(m["msc"]), len(e["msc"]))
    assert n >= 288 * 20 and np.array_equal(m["msc"][:n], e["msc"][:n])
    k = min(len(m["rs"]), len(e["rs"]))
    assert k >= 3 and np.array_equal(m["rs"][:k], e["rs"][:k])
    lf = np.concatenate(tx.logical)
    assert np.array_equal(e["msc"], lf[8 * 288: 8 * 288 + len(e["msc"])])      # first logical frame = CIF of selection + 16
    assert all(i["start_index"] == 504 for i in m["info"][1:]) and all(i["fine"] == 0 for i in m["info"])


def test_closed_loop_with_noise(oracle, ref, tmp_path):
    tx = dabtx.DabTx(seed=0x77)
    s = tx.frames(16)
    iq = dabtx.add_awgn(s, 9.0, seed=5, signal_power=float(np.mean(np.abs(s[3000:190000]) ** 2)))
    e = ref.e2e(iq, disable_coarse=True, select_at_fib=24, dump_path=str(tmp_path / "n.msc"))
    p = oracle.prot_eep(96, 1, 3)
    m = oracle.rx_run(iq, prot=p, start_cu=0, len_cu=72, select_after_frames=1, disable_coarse=True)
    assert np.array_equal(m["fibs"][:len(e["fibs"])], e["fibs"])
    n = min(len(m["msc"]), len(e["msc"]))
    assert n > 0 and np.array_equal(m["msc"][:n], e["msc"][:n])


@pytest.mark.parametrize("placement", [1, 2])
def test_find_index_other_placements(oracle, ref, sig, placement):
    """StrongestPeak / EarliestPeakWithBinning (phasereference.cpp:93-211): index and CIR, on aligned, shifted, noisy,
    signal-free and all-zero windows"""
    tx, iq = sig
    base = 3 * TF + TNULL
    rng = np.random.default_rng(placement)
    wins = [iq[base - off: base - off + TU] for off in (199, 100, 350, 700, -3000)]
    wins.append(dabtx.add_awgn(iq, 3.0, seed=3)[base - 250: base - 250 + TU])
    wins.append((rng.standard_normal(TU) + 1j * rng.standard_normal(TU)).astype(np.complex64) * 0.05)      # no PRS at all
    wins.append(np.zeros(TU, np.complex64))
    echo = iq[base - 300: base - 300 + TU] + 0.7 * iq[base - 300 - 180: base - 300 - 180 + TU]            # pre-echo 180 samples earlier
    wins.append(echo.astype(np.complex64))
    for k, v in enumerate(wins):
        i1, c1 = oracle.find_index(v, placement)
        i2, c2 = ref.find_index(v, {1: 0, 2: 1}[placement])
        assert i1 == i2, (k, i1, i2)
        # (the binning variant never looks at the last 8 samples: both leave them at the zero they were allocated with)
        assert same(c1, c2), k


@pytest.mark.parametrize("method,shift_hz", [(0, 2000), (1, 2000), (2, 2000), (2, -3000), (0, 0)])
def test_closed_loop_coarse_corrector(oracle, ref, tmp_path, method, shift_hz):
    """coarse frequency corrector on (welle-cli default): PatternOfZeros / GetMiddle / CorrelatePRS (ofdm-processor.cpp:537-644)
    in the closed loop - identical FIB stream (flags and payloads) and identical final correctors"""
    tx = dabtx.DabTx(seed=0x51 + method)
    iq = dabtx.freq_shift(tx.frames(12), shift_hz)
    e = ref.e2e(iq, disable_coarse=False, select_at_fib=10 ** 9, dump_path=str(tmp_path / "c.msc"), freqsync_method=method)
    m = oracle.rx_run(iq, disable_coarse=False, freqsync_method=method)
    assert len(e["fibs"]) >= 12 * 8
    n = min(len(m["fibs"]), len(e["fibs"]))
    assert np.array_equal(m["fibs"][:n], e["fibs"][:n])
    if len(e["corr"]):
        # onFrequencyCorrectorChange samples the state every 0.2 s of input, i.e. also between the coarse update of a frame and
        # its fine update: (fine of frame k-1, coarse of frame k) is as legitimate as the end-of-frame pair
        inf = m["info"]
        pairs = [(i["fine"], i["coarse"]) for i in inf] + [(inf[k - 1]["fine"], inf[k]["coarse"]) for k in range(1, len(inf))] + [(0, inf[0]["coarse"])]
        assert tuple(int(x) for x in e["corr"][-1]) in pairs


@pytest.mark.parametrize("placement", [1, 2])
def test_closed_loop_other_placements(oracle, ref, tmp_path, placement):
    tx = dabtx.DabTx(seed=0x61)
    iq = tx.frames(10)
    e = ref.e2e(iq, disable_coarse=True, select_at_fib=10 ** 9, dump_path=str(tmp_path / "p.msc"), fft_placement=placement)
    m = oracle.rx_run(iq, disable_coarse=True, fft_placement=placement)
    n = min(len(m["fibs"]), len(e["fibs"]))
    assert n >= 12 * 7 and np.array_equal(m["fibs"][:n], e["fibs"][:n])


def test_all_uep_profiles(oracle, ref):
    """every (bitrate, protection level) pair of the reference's UEP table (uep-protection.cpp:38-118)"""
    n = 0
    for br in (32, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320, 384):
        for lv in range(1, 6):
            from oracle.bind import ProtT
            import ctypes as C
            p = ProtT()
            if oracle.lib.orc_prot_uep(br, lv, C.byref(p)) != 0:
                continue
            rng = np.random.default_rng(br * 7 + lv)
            soft = rng.integers(-127, 128, p.in_bits).astype(np.int8)
            assert same(oracle.msc_deconvolve(p, soft, True), ref.uep_deconvolve(br, lv, soft, True)), (br, lv)
            n += 1
    assert n >= 60


def test_all_eep_profiles(oracle, ref):
    """EEP-A at every multiple of 8 kbit/s up to 192 and EEP-B at every multiple of 32 kbit/s up to 192, all four levels
    (eep-protection.cpp:32-113)"""
    n = 0
    for pa, step in ((1, 8), (0, 32)):
        for br in range(step, 193, step):
            for lv in (1, 2, 3, 4):
                p = oracle.prot_eep(br, pa, lv)
                rng = np.random.default_rng(br * 11 + lv + pa)
                soft = rng.integers(-127, 128, p.in_bits).astype(np.int8)
                assert same(oracle.msc_deconvolve(p, soft, False), ref.eep_deconvolve(br, pa, lv, soft, False)), (br, pa, lv)
                n += 1
    assert n == 4 * 24 + 4 * 6


def test_closed_loop_multipath_offset_noise(oracle, ref, tmp_path):
    """a harder channel: two echoes (60 and 210 samples, the second 6 dB down with a phase turn), +137 Hz carrier offset, 13 dB SNR, a
    start offset of 1234 samples - FIBs, logical frames and RS events of the whole run like the reference's"""
    tx = dabtx.DabTx(seed=0x99)
    s = tx.frames(16)
    ch = s.copy()
    ch[60:] += 0.7 * s[:-60]
    ch[210:] += (0.5 * np.exp(1j * 1.1)) * s[:-210]
    ch = dabtx.freq_shift(ch.astype(np.complex64), 137.0)
    iq = np.concatenate([np.zeros(1234, np.complex64), dabtx.add_awgn(ch, 13.0, seed=7, signal_power=float(np.mean(np.abs(ch[3000:190000]) ** 2)))])
    e = ref.e2e(iq, disable_coarse=True, select_at_fib=24, dump_path=str(tmp_path / "mp.msc"))
    p = oracle.prot_eep(96, 1, 3)
    # the harness tunes from inside the first FIB callback (>= the 24th) at which the service is listed, i.e. the second CRC-ok FIB
    # (two sightings): during the pull-in of the fine corrector the first FIBs fail, so the selection frame is read off the FIB flags
    ok = np.nonzero(e["fibs"][:, 0])[0]
    assert len(ok) >= 2
    sel_fib = max(int(ok[1]), 23)
    m = oracle.rx_run(iq, prot=p, start_cu=0, len_cu=72, select_after_frames=sel_fib // 12, disable_coarse=True)
    n = min(len(m["fibs"]), len(e["fibs"]))
    assert n >= 12 * 10 and np.array_equal(m["fibs"][:n], e["fibs"][:n])
    assert e["fibs"][-36:, 0].all()                   # the receiver does lock on this channel once the fine corrector has pulled in
    k = min(len(m["msc"]), len(e["msc"]))
    # (the reference's dump file is only flushed in 4 KiB blocks: the harness leaks the receiver instead of tearing it down)
    assert k >= 288 * 10 and np.array_equal(m["msc"][:k], e["msc"][:k])
    r = min(len(m["rs"]), len(e["rs"]))
    assert r >= 2 and np.array_equal(m["rs"][:r], e["rs"][:r])


def test_snr_estimate(oracle, ref, tmp_path):
    """OfdmDecoder::get_snr (ofdm-decoder.cpp:240-265) through the only tap the reference has for it: onSNR, the value
    snr = 0.7 snr + 0.3 get_snr(PRS spectrum) reported after every 11th frame (:144-160).  Replaying that recursion over the oracle's
    per-frame values must give the reference's floats."""
    tx = dabtx.DabTx(seed=0x5A)
    s = tx.frames(36)
    sp = float(np.mean(np.abs(s[3000:190000]) ** 2))
    iq = s.copy()
    for k, db in enumerate((24.0, 9.0, 16.0, 6.0, 12.0, 20.0)):          # the noise level changes every six frames
        seg = slice(6 * k * TF, 6 * (k + 1) * TF)
        iq[seg] = dabtx.add_awgn(s[seg], db, seed=30 + k, signal_power=sp)
    e = ref.e2e(iq, disable_coarse=True, select_at_fib=24, dump_path=str(tmp_path / "snr.msc"))
    m = oracle.rx_run(iq, disable_coarse=True)
    raw = [i["snr_raw"] for i in m["info"]]
    assert len(set(raw)) >= 4 and all(0 <= r <= 40 for r in raw), raw
    snr, count, rep = np.float32(0), 0, []
    for r in raw:
        snr = np.float32(0.7 * float(snr) + 0.3 * r)
        count += 1
        if count > 10:
            rep.append(snr); count = 0
    k = min(len(rep), len(e["snr"]))
    assert k >= 2 and np.array_equal(np.array(rep[:k], np.float32), e["snr"][:k]), (rep, e["snr"])


def test_reacquisition_after_gap(oracle, ref, tmp_path):
    """a recording with a hole (signal, 1.3 frames of near-silence, signal at an unrelated timing): SyncOnPhase fails, the null search
    runs again from the running signal level (ofdm-processor.cpp:166,215,347-350) - FIBs like the reference's over the whole run"""
    tx = dabtx.DabTx(seed=0x6B)
    s = tx.frames(22)
    a, b = s[:9 * TF + 40000], s[11 * TF - 777:]
    iq = np.concatenate([a, np.full(int(1.3 * TF), 1e-5 + 0j, np.complex64), b]).astype(np.complex64)
    e = ref.e2e(iq, disable_coarse=True, select_at_fib=1 << 30, dump_path=str(tmp_path / "gap.msc"))
    m = oracle.rx_run(iq, disable_coarse=True)
    n = min(len(m["fibs"]), len(e["fibs"]))
    assert n >= 12 * 14 and np.array_equal(m["fibs"][:n], e["fibs"][:n])
    ok = m["fibs"][:n, 0]
    assert ok[:12 * 6].all() and ok[-24:].all() and not ok.all()          # locked, lost, locked again
