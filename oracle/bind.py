"""ctypes bindings for the two CHECKERS (test infrastructure only — never imported by the product):

  Oracle  -> oracle/liboracle.so        our plain-C restatement (oracle/dab_oracle.c)
  Ref     -> oracle/_ref/libwelle_ref.so the unmodified reference backend + oracle/ref_shim.cpp

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
"""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libwelle_ref.so")

L, K, TU, TS, TG, TNULL, TF = 76, 1536, 2048, 2552, 504, 2656, 196608


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])


def build_ref():
    """Only possible where /root/reference exists (this container); the GPU box uses the prebuilt .so."""
    if os.path.isdir("/root/reference/src"):
        subprocess.check_call(["make", "-s", "-j8", "-C", HERE, "ref"])


def _p(a, t=None):
    return a.ctypes.data_as(C.c_void_p)


class ProtT(C.Structure):
    _fields_ = [("bitrate", C.c_int), ("nblk", C.c_int), ("L", C.c_int * 4), ("PI", C.c_int * 4), ("in_bits", C.c_int)]


class RxCfg(C.Structure):
    _fields_ = [("disable_coarse", C.c_int), ("fft_placement", C.c_int), ("freqsync_method", C.c_int), ("subch_start_cu", C.c_int), ("subch_len_cu", C.c_int),
                ("prot", ProtT), ("dabplus", C.c_int), ("select_after_frames", C.c_int), ("select_after_symbol", C.c_int)]


class FrameInfo(C.Structure):
    _fields_ = [("start_index", C.c_int), ("fine", C.c_int), ("coarse", C.c_int), ("snr_raw", C.c_int), ("frame_pos", C.c_long)]


class SffResult(C.Structure):
    _fields_ = [("attempted", C.c_int), ("corr", C.c_int), ("uncorr", C.c_int), ("sync_ok", C.c_int),
                ("num_aus", C.c_int), ("au_crc_ok_mask", C.c_int)]


class Oracle:
    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        self.lib = C.CDLL(ORACLE_SO)
        l = self.lib
        l.orc_find_index.restype = C.c_int
        l.orc_coarse_pattern_of_zeros.restype = C.c_int
        l.orc_rs_decode_codeword.restype = C.c_int
        for f in (l.orc_crc_fire, l.orc_crc_ccitt, l.orc_crc16):
            f.restype = C.c_uint
        l.orc_deint_new.restype = C.c_void_p
        l.orc_sff_new.restype = C.c_void_p
        l.orc_rx_new.restype = C.c_void_p
        l.orc_rx_run.restype = C.c_long

    # ---- tables
    def perm_table(self):
        o = np.zeros(K, np.int16); self.lib.orc_perm_table(_p(o)); return o

    def prs_table(self):
        o = np.zeros(2 * TU, np.float32); self.lib.orc_prs_table(_p(o)); return o.view(np.complex64)

    def pcodes(self):
        o = np.zeros(24 * 32, np.int8); self.lib.orc_pcodes(_p(o)); return o.reshape(24, 32)

    def prbs(self, n):
        o = np.zeros(n, np.uint8); self.lib.orc_prbs(_p(o), n); return o

    # ---- fft / sync / demod
    def fft(self, x, inverse=False):
        x = np.ascontiguousarray(x, np.complex64); o = np.empty_like(x)
        self.lib.orc_fft(len(x), _p(x), _p(o), int(inverse)); return o

    def ifft_scaled(self, x):
        x = np.ascontiguousarray(x, np.complex64); o = np.empty_like(x)
        self.lib.orc_ifft_scaled(len(x), _p(x), _p(o)); return o

    def find_index(self, v, placement=0):
        """placement: 0 ThresholdBeforePeak, 1 StrongestPeak, 2 EarliestPeakWithBinning"""
        v = np.ascontiguousarray(v, np.complex64); cir = np.zeros(TU, np.float32)
        return self.lib.orc_find_index_m(_p(v), _p(cir), int(placement)), cir

    def coarse(self, prs, method=0):
        """method: 0 PatternOfZeros, 1 GetMiddle, 2 CorrelatePRS"""
        prs = np.ascontiguousarray(prs, np.complex64)
        return self.lib.orc_coarse(_p(prs), int(method))

    def demod_frame(self, prs, syms, want_r1=False):
        prs = np.ascontiguousarray(prs, np.complex64); syms = np.ascontiguousarray(syms, np.complex64)
        soft = np.zeros(75 * 3072, np.int8)
        r1 = np.zeros(75 * K, np.complex64) if want_r1 else None
        self.lib.orc_ofdm_demod_frame(_p(prs), _p(syms), _p(soft), _p(r1) if want_r1 else None)
        return (soft.reshape(75, 3072), r1.reshape(75, K)) if want_r1 else soft.reshape(75, 3072)

    # ---- viterbi / fic / msc
    def viterbi(self, soft, nbits):
        soft = np.ascontiguousarray(soft, np.int8); assert soft.size == (nbits + 6) * 4
        o = np.zeros(nbits, np.uint8); self.lib.orc_viterbi(nbits, _p(soft), _p(o)); return o

    def conv_encode(self, bits):
        bits = np.ascontiguousarray(bits, np.uint8); o = np.zeros((len(bits) + 6) * 4, np.uint8)
        self.lib.orc_conv_encode(_p(bits), len(bits), _p(o)); return o

    def fic_decode(self, soft9216):
        s = np.ascontiguousarray(soft9216, np.int8); assert s.size == 9216
        fb = np.zeros(12 * 256, np.uint8); ok = np.zeros(12, np.uint8)
        self.lib.orc_fic_decode(_p(s), _p(fb), _p(ok)); return fb.reshape(12, 256), ok

    def check_crc_bits(self, bits):
        b = np.ascontiguousarray(bits, np.uint8); return self.lib.orc_check_crc_bits(_p(b), len(b))

    def prot_eep(self, bitrate, profile_a, level):
        p = ProtT(); r = self.lib.orc_prot_eep(bitrate, int(profile_a), level, C.byref(p)); assert r == 0; return p

    def prot_uep(self, bitrate, level):
        p = ProtT(); r = self.lib.orc_prot_uep(bitrate, level, C.byref(p)); assert r == 0; return p

    def msc_deconvolve(self, prot, soft, dedisperse=False):
        s = np.ascontiguousarray(soft, np.int8); assert s.size == prot.in_bits, (s.size, prot.in_bits)
        o = np.zeros(24 * prot.bitrate, np.uint8); self.lib.orc_msc_deconvolve(C.byref(prot), _p(s), _p(o))
        if dedisperse:
            self.lib.orc_dedisperse(_p(o), len(o))
        return o

    def pack_bits(self, bits):
        b = np.ascontiguousarray(bits, np.uint8); o = np.zeros(len(b) // 8, np.uint8)
        self.lib.orc_pack_bits(_p(b), len(o), _p(o)); return o

    def deinterleave(self, cifs):
        """cifs: [ncif, fragment] int8 -> [ncif-16, fragment] (output valid after the 16-CIF warm-up)"""
        cifs = np.ascontiguousarray(cifs, np.int8); n, frag = cifs.shape
        d = C.c_void_p(self.lib.orc_deint_new(frag)); out = []
        tmp = np.zeros(frag, np.int8)
        for t in range(n):
            if self.lib.orc_deint_push(d, _p(cifs[t]), _p(tmp)):
                out.append(tmp.copy())
        self.lib.orc_deint_free(d)
        return np.array(out, np.int8).reshape(-1, frag)

    # ---- RS / CRC
    def rs_encode(self, data110):
        d = np.ascontiguousarray(data110, np.uint8); p = np.zeros(10, np.uint8)
        self.lib.orc_rs_encode(_p(d), _p(p)); return p

    def rs_decode_codeword(self, cw120):
        cw = np.array(cw120, np.uint8).copy(); pos = np.zeros(10, np.int32)
        r = self.lib.orc_rs_decode_codeword(_p(cw), _p(pos)); return r, cw, pos

    def rs_decode_superframe(self, sf):
        sf = np.array(sf, np.uint8).copy(); c = C.c_int(); u = C.c_int()
        self.lib.orc_rs_decode_superframe(_p(sf), len(sf), C.byref(c), C.byref(u)); return sf, c.value, u.value

    def crc_fire(self, d):
        d = np.ascontiguousarray(d, np.uint8); return self.lib.orc_crc_fire(_p(d), len(d))

    def crc_ccitt(self, d):
        d = np.ascontiguousarray(d, np.uint8); return self.lib.orc_crc_ccitt(_p(d), len(d))

    def superframe_filter(self, frames):
        """frames [n, flen] uint8 -> list of dict per attempted RS decode, plus synced superframes"""
        frames = np.ascontiguousarray(frames, np.uint8); n, flen = frames.shape
        f = C.c_void_p(self.lib.orc_sff_new()); res = SffResult(); sfbuf = np.zeros(5 * flen, np.uint8)
        ev, sfs = [], []
        for i in range(n):
            self.lib.orc_sff_feed(f, _p(frames[i]), flen, C.byref(res), _p(sfbuf))
            if res.attempted:
                ev.append(dict(frame=i, corr=res.corr, uncorr=res.uncorr, sync=res.sync_ok, num_aus=res.num_aus, au_ok=res.au_crc_ok_mask))
                if res.sync_ok:
                    sfs.append(sfbuf.copy())
        self.lib.orc_sff_free(f)
        return ev, sfs

    # ---- closed-loop receiver
    def rx_run(self, iq, prot=None, start_cu=0, len_cu=0, dabplus=True, select_after_frames=1, disable_coarse=True,
               want_soft=0, fft_placement=0, freqsync_method=0):
        iq = np.ascontiguousarray(iq, np.complex64)
        cfg = RxCfg(); cfg.disable_coarse = int(disable_coarse); cfg.subch_start_cu = start_cu; cfg.subch_len_cu = len_cu
        cfg.fft_placement = int(fft_placement); cfg.freqsync_method = int(freqsync_method)
        if prot is not None:
            cfg.prot = prot
        cfg.dabplus = int(dabplus); cfg.select_after_frames = select_after_frames
        rx = C.c_void_p(self.lib.orc_rx_new(C.byref(cfg)))
        nfr = len(iq) // TF + 2
        fibs = np.zeros(33 * 12 * nfr, np.uint8); msc = np.zeros(4 * nfr * 3 * 384, np.uint8)
        rs = np.zeros(2 * 4 * nfr, np.int32); fi = (FrameInfo * nfr)()
        soft = np.zeros(want_soft * 75 * 3072, np.int8) if want_soft else None
        nf_, nm_, nr_ = C.c_long(), C.c_long(), C.c_long()
        n = self.lib.orc_rx_run(rx, _p(iq), C.c_long(len(iq)), _p(fibs), C.c_long(12 * nfr), C.byref(nf_), _p(msc), C.c_long(len(msc)), C.byref(nm_),
                                _p(rs), C.c_long(4 * nfr), C.byref(nr_), fi, C.c_long(nfr), _p(soft) if want_soft else None, C.c_long(want_soft))
        self.lib.orc_rx_free(rx)
        info = [dict(start_index=fi[i].start_index, fine=fi[i].fine, coarse=fi[i].coarse, pos=fi[i].frame_pos, snr_raw=fi[i].snr_raw) for i in range(n)]
        out = dict(frames=n, fibs=fibs[:33 * nf_.value].reshape(-1, 33), msc=msc[:nm_.value], rs=rs[:2 * nr_.value].reshape(-1, 2), info=info)
        if want_soft:
            out["soft"] = soft.reshape(want_soft, 75, 3072)[:min(n, want_soft)]
        return out


class Ref:
    """The unmodified reference (KISS-FFT build) behind oracle/ref_shim.cpp."""

    def __init__(self):
        if not os.path.exists(REF_SO):
            build_ref()
        self.lib = C.CDLL(REF_SO)
        l = self.lib
        l.ref_find_index.restype = C.c_int
        l.ref_fic_decode.restype = C.c_int
        l.ref_dabaudio_chain.restype = C.c_long
        l.ref_rs_decode_codeword.restype = C.c_int
        l.ref_crc_fire.restype = C.c_uint
        l.ref_crc_ccitt.restype = C.c_uint
        l.ref_e2e_get.restype = C.c_long
        l.ref_subchannel_bitrate.restype = C.c_int

    @staticmethod
    def available():
        return os.path.exists(REF_SO)

    def perm_table(self):
        o = np.zeros(K, np.int16); self.lib.ref_perm_table(1, _p(o)); return o

    def prs_table(self):
        o = np.zeros(2 * TU, np.float32); self.lib.ref_prs_table(1, _p(o)); return o.view(np.complex64)

    def pcodes(self):
        o = np.zeros(24 * 32, np.int8); self.lib.ref_pcodes(_p(o)); return o.reshape(24, 32)

    def fft(self, x, inverse=False):
        b = np.array(x, np.complex64).copy()
        (self.lib.ref_fft_backward if inverse else self.lib.ref_fft_forward)(len(b), _p(b)); return b

    def process_prs(self, prs, method=0):
        """OFDMProcessor::processPRS; method in this repository's numbering (0 PatternOfZeros, 1 GetMiddle, 2 CorrelatePRS)"""
        prs = np.ascontiguousarray(prs, np.complex64)
        return self.lib.ref_process_prs(_p(prs), {0: 2, 1: 0, 2: 1}[int(method)])

    def find_index(self, v, method=2):
        # method in the reference's enum order: 0 StrongestPeak, 1 EarliestPeakWithBinning, 2 ThresholdBeforePeak
        v = np.ascontiguousarray(v, np.complex64); cir = np.zeros(TU, np.float32)
        return self.lib.ref_find_index(1, method, _p(v), _p(cir)), cir

    def demod_frame(self, prs, syms, want_r1=False):
        prs = np.ascontiguousarray(prs, np.complex64); syms = np.ascontiguousarray(syms, np.complex64)
        soft = np.zeros(75 * 3072, np.int8); r1 = np.zeros(75 * K, np.complex64) if want_r1 else None
        self.lib.ref_ofdm_demod_frame(1, _p(prs), _p(syms), _p(soft), _p(r1) if want_r1 else None, None)
        return (soft.reshape(75, 3072), r1.reshape(75, K)) if want_r1 else soft.reshape(75, 3072)

    def viterbi(self, soft, nbits):
        soft = np.ascontiguousarray(soft, np.int8); o = np.zeros(nbits, np.uint8)
        self.lib.ref_viterbi(nbits, _p(soft), _p(o)); return o

    def fic_decode(self, soft9216):
        s = np.ascontiguousarray(soft9216, np.int8); fb = np.zeros(12 * 256, np.uint8); ok = np.zeros(12, np.uint8)
        n = self.lib.ref_fic_decode(_p(s), _p(fb), _p(ok)); assert n == 12; return fb.reshape(12, 256), ok

    def eep_deconvolve(self, bitrate, profile_a, level, soft, dedisperse=False):
        s = np.ascontiguousarray(soft, np.int8); o = np.zeros(24 * bitrate, np.uint8)
        self.lib.ref_eep_deconvolve(bitrate, int(profile_a), level, _p(s), _p(o), int(dedisperse)); return o

    def uep_deconvolve(self, bitrate, level, soft, dedisperse=False):
        s = np.ascontiguousarray(soft, np.int8); o = np.zeros(24 * bitrate, np.uint8)
        self.lib.ref_uep_deconvolve(bitrate, level, _p(s), _p(o), int(dedisperse)); return o

    def dabaudio_chain(self, cifs, bitrate, profile_a=True, level=3, dabplus=True, dump_path="/tmp/ref_chain.msc",
                       short_form=False, uep_level=0):
        cifs = np.ascontiguousarray(cifs, np.int8); n, frag = cifs.shape
        rs = np.zeros(2 * (n + 8), np.int32); nrs = C.c_int()
        sz = self.lib.ref_dabaudio_chain(_p(cifs), n, frag, bitrate, int(short_form), uep_level, int(profile_a), level, int(dabplus),
                                         dump_path.encode(), _p(rs), n + 8, C.byref(nrs))
        data = np.fromfile(dump_path, np.uint8) if sz > 0 else np.zeros(0, np.uint8)
        return data, rs[:2 * nrs.value].reshape(-1, 2)

    def rs_encode(self, d):
        d = np.ascontiguousarray(d, np.uint8); p = np.zeros(10, np.uint8); self.lib.ref_rs_encode(_p(d), _p(p)); return p

    def rs_decode_codeword(self, cw):
        cw = np.array(cw, np.uint8).copy(); pos = np.zeros(10, np.int32)
        r = self.lib.ref_rs_decode_codeword(_p(cw), _p(pos)); return r, cw, pos

    def rs_decode_codewords(self, cws):
        """rs_decode_codeword over the rows of cws [n, 120] -> (results [n], corrected codewords [n, 120], positions [n, 10])"""
        res = [self.rs_decode_codeword(cw) for cw in np.asarray(cws, np.uint8)]
        return np.array([r[0] for r in res], np.int32), np.stack([r[1] for r in res]), np.stack([r[2] for r in res])

    def rs_decode_superframe(self, sf):
        sf = np.array(sf, np.uint8).copy(); c = C.c_int(); u = C.c_int()
        self.lib.ref_rs_decode_superframe(_p(sf), len(sf), C.byref(c), C.byref(u)); return sf, c.value, u.value

    def crc_fire(self, d):
        d = np.ascontiguousarray(d, np.uint8); return self.lib.ref_crc_fire(_p(d), len(d))

    def crc_ccitt(self, d):
        d = np.ascontiguousarray(d, np.uint8); return self.lib.ref_crc_ccitt(_p(d), len(d))

    def check_crc_bits(self, bits):
        b = np.ascontiguousarray(bits, np.uint8); return self.lib.ref_check_crc_bits(_p(b), len(b))

    def superframe_filter(self, frames):
        frames = np.ascontiguousarray(frames, np.uint8); n, flen = frames.shape
        fec = np.zeros(2 * (n + 1), np.int32); au_err = C.c_int(); good = C.c_int()
        k = self.lib.ref_superframe_filter(_p(frames), n, flen, _p(fec), n + 1, C.byref(au_err), C.byref(good))
        return fec[:2 * k].reshape(-1, 2), au_err.value, good.value

    def fib_dump(self, fibs):
        """FIBProcessor fed the 32-byte FIBs in order -> its text dump of the database and of the FIG-derived callbacks"""
        fibs = np.ascontiguousarray(fibs, np.uint8)
        buf = C.create_string_buffer(1 << 18)
        n = self.lib.ref_fib_dump(_p(fibs), len(fibs), buf, len(buf))
        assert n >= 0
        return buf.value.decode("latin1")

    def tii_run(self, nulls, prss):
        """the unmodified TIIDecoder fed frame by frame: nulls [n, 2656], prss [n, 2048] complex64 -> [(comb, pattern, delay_samples, error), ...]"""
        nulls = np.ascontiguousarray(nulls, np.complex64); prss = np.ascontiguousarray(prss, np.complex64)
        n = nulls.shape[0]
        out = np.zeros(4 * 256, np.float32)
        self.lib.ref_tii_run.restype = C.c_int
        k = self.lib.ref_tii_run(_p(nulls), _p(prss), n, _p(out), 256)
        return [tuple(out[4 * i: 4 * i + 4].tolist()) for i in range(min(k, 256))]

    def e2e(self, iq, disable_coarse=True, select_at_fib=24, dump_path="/tmp/ref_e2e.msc", keep_cir=False, fft_placement=0, freqsync_method=0):
        """fft_placement / freqsync_method use this repository's numbering (0 = the reference's defaults), see Oracle.find_index / coarse"""
        iq = np.ascontiguousarray(iq, np.complex64)
        if os.path.exists(dump_path):
            os.remove(dump_path)
        n = self.lib.ref_e2e_run2(_p(iq), C.c_long(len(iq)), int(disable_coarse), select_at_fib, dump_path.encode(), int(keep_cir),
                                  {0: 2, 1: 0, 2: 1}[int(fft_placement)], {0: 2, 1: 0, 2: 1}[int(freqsync_method)])

        def get(what, dt):
            sz = self.lib.ref_e2e_get(what, None, C.c_long(0))
            buf = np.zeros(sz, np.uint8)
            if sz:
                self.lib.ref_e2e_get(what, _p(buf), C.c_long(sz))
            return buf.view(dt)
        st = np.zeros(6, np.float64); self.lib.ref_e2e_stats(_p(st))
        msc = np.fromfile(dump_path, np.uint8) if os.path.exists(dump_path) else np.zeros(0, np.uint8)
        return dict(nfib=n, fibs=get(0, np.uint8).reshape(-1, 33), rs=get(1, np.int32).reshape(-1, 2), corr=get(2, np.int32).reshape(-1, 2),
                    snr=get(3, np.float32), cir=get(4, np.float32).reshape(-1, TU), msc=msc,
                    sync_true=int(st[0]), sync_false=int(st[1]), select_ok=int(st[2]), frames_done=int(st[3]), seconds=st[4])
