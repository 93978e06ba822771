"""ctypes binding of libsw_whisper.so (include/sw_whisper.h) for the tests and bench.py.

This is NOT the product's host layer (that is C++: csrc/stt_engine.*, mirroring the reference's
SttEngine); it only lets Python test code call the C ABI. There is no CPU fallback: loading fails
loudly if the CUDA library is missing, and every compute call fails without an sm_100 device.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SW_LIB_PATH") or os.path.join(HERE, "libsw_whisper.so")  # SW_LIB_PATH: A/B a development build


class CtxParams(C.Structure):
    _fields_ = [("device", C.c_int), ("max_batch", C.c_int), ("max_beams", C.c_int),
                ("flash_attn", C.c_int), ("n_lanes", C.c_int), ("reserved", C.c_int * 11)]


class ModelInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "n_vocab", "n_audio_ctx", "n_audio_state", "n_audio_head", "n_audio_layer", "n_text_ctx",
        "n_text_state", "n_text_head", "n_text_layer", "n_mels", "ftype", "is_multilingual",
        "token_eot", "token_sot", "token_translate", "token_transcribe", "token_solm", "token_prev",
        "token_nosp", "token_not", "token_beg")]


ABORT_CB = C.CFUNCTYPE(C.c_int, C.c_void_p)


class FullParams(C.Structure):
    _fields_ = [
        ("strategy", C.c_int), ("beam_size", C.c_int), ("best_of", C.c_int),
        ("temperature", C.c_float), ("temperature_inc", C.c_float), ("entropy_thold", C.c_float),
        ("logprob_thold", C.c_float), ("no_speech_thold", C.c_float),
        ("translate", C.c_int), ("tdrz_enable", C.c_int), ("suppress_nst", C.c_int),
        ("suppress_blank", C.c_int), ("token_timestamps", C.c_int), ("no_timestamps", C.c_int),
        ("single_segment", C.c_int), ("no_context", C.c_int),
        ("max_initial_ts", C.c_float), ("length_penalty", C.c_float),
        ("language", C.c_char_p), ("initial_prompt", C.c_char_p),
        ("prompt_tokens", C.POINTER(C.c_int32)), ("prompt_n_tokens", C.c_int),
        ("abort_callback", ABORT_CB), ("abort_callback_user_data", C.c_void_p),
        ("n_threads", C.c_int), ("reserved", C.c_int * 8)]


class TokenData(C.Structure):
    _fields_ = [("id", C.c_int32), ("tid", C.c_int32), ("p", C.c_float), ("plog", C.c_float),
                ("pt", C.c_float), ("ptsum", C.c_float), ("t0", C.c_int64), ("t1", C.c_int64),
                ("t_dtw", C.c_int64), ("vlen", C.c_float)]


class Stats(C.Structure):
    _fields_ = [("ms_mel", C.c_double), ("ms_encode", C.c_double), ("ms_decode", C.c_double),
                ("n_windows", C.c_long), ("n_steps", C.c_long), ("n_launches", C.c_long),
                ("decode_bytes", C.c_double), ("decoder_weight_bytes", C.c_double),
                ("h2d_bytes", C.c_double), ("d2h_bytes", C.c_double), ("ms_xattn", C.c_double),
                ("n_xattn", C.c_long), ("xattn_bytes", C.c_double), ("n_lanes", C.c_long)]


class ProsodyOpts(C.Structure):
    _fields_ = [("lpf_alpha", C.c_float), ("gender_threshold", C.c_float), ("min_pitch", C.c_float),
                ("max_pitch", C.c_float)]


class Prosody(C.Structure):
    _fields_ = [("gender", C.c_char), ("emotion", C.c_int), ("arousal", C.c_float), ("valence", C.c_float),
                ("pitch_mean", C.c_float), ("pitch_std", C.c_float), ("energy_mean", C.c_float),
                ("energy_std", C.c_float), ("spectral_centroid", C.c_float), ("zero_crossing_rate", C.c_float),
                ("speaker_vec", C.c_float * 8)]


EMOTIONS = ["neutral", "excited", "sad", "angry"]
PROSODY_FLOATS = ["arousal", "valence", "pitch_mean", "pitch_std", "energy_mean", "energy_std",
                  "spectral_centroid", "zero_crossing_rate"]

EXPORTS = [
    "sw_last_error", "sw_version", "sw_device_count", "sw_log_set", "sw_ctx_default_params",
    "sw_ctx_create", "sw_ctx_destroy", "sw_ctx_model_info", "sw_token_to_str", "sw_token_eot",
    "sw_lang_id", "sw_full_default_params", "sw_full", "sw_full_pcm16", "sw_full_batch_pcm16",
    "sw_full_batch_f32", "sw_full_batch_pcm16_lang", "sw_full_batch_f32_lang", "sw_host_alloc", "sw_host_free", "sw_result_n_segments",
    "sw_result_segment_text", "sw_result_segment_t0", "sw_result_segment_t1",
    "sw_result_segment_speaker_turn_next", "sw_result_n_tokens", "sw_result_token_data",
    "sw_result_lang_id", "sw_result_n_decode_steps", "sw_result_n_windows", "sw_result_free",
    "sw_ctx_get_stats", "sw_ctx_set_kernel_timing", "sw_mel_pcm16", "sw_mel_f32", "sw_encode", "sw_decode_logits",
    "sw_prosody_default_opts", "sw_prosody_segments_f32", "sw_prosody_segments_pcm16",
    "sw_resample_out_len", "sw_resample_f32",
    "sw_dev_gemm_bf16", "sw_dev_skinny_gemm", "sw_dev_skinny_split", "sw_dev_layer_norm", "sw_dev_occupy",
    "sw_dev_skinny_gemm_k", "sw_dev_skinny_split_k", "sw_dev_encoder_attention", "sw_dev_cross_attention_ws_floats",
    "sw_dev_cross_attention", "sw_dev_self_attention"]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libsw_whisper.so is not built (run __graft_entry__.build()); "
                           "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, ci, fp = C.c_void_p, C.c_int, C.POINTER(C.c_float)
    L.sw_last_error.restype = C.c_char_p
    L.sw_version.restype = C.c_char_p
    L.sw_ctx_default_params.restype = CtxParams
    L.sw_ctx_create.restype = vp
    L.sw_ctx_create.argtypes = [C.c_char_p, C.POINTER(CtxParams)]
    L.sw_ctx_destroy.argtypes = [vp]
    L.sw_ctx_model_info.argtypes = [vp, C.POINTER(ModelInfo)]
    L.sw_token_to_str.restype = C.c_char_p
    L.sw_token_to_str.argtypes = [vp, ci]
    L.sw_token_eot.argtypes = [vp]
    L.sw_lang_id.argtypes = [C.c_char_p]
    L.sw_full_default_params.restype = FullParams
    L.sw_full_default_params.argtypes = [ci]
    L.sw_full.argtypes = [vp, C.POINTER(FullParams), fp, ci, C.POINTER(vp)]
    L.sw_full_pcm16.argtypes = [vp, C.POINTER(FullParams), C.POINTER(C.c_int16), ci, C.POINTER(vp)]
    L.sw_full_batch_pcm16.argtypes = [vp, C.POINTER(FullParams), C.POINTER(C.POINTER(C.c_int16)),
                                      C.POINTER(ci), ci, C.POINTER(vp)]
    L.sw_full_batch_f32.argtypes = [vp, C.POINTER(FullParams), C.POINTER(fp), C.POINTER(ci), ci,
                                    C.POINTER(vp)]
    L.sw_full_batch_pcm16_lang.argtypes = [vp, C.POINTER(FullParams), C.POINTER(C.POINTER(C.c_int16)),
                                           C.POINTER(ci), ci, C.POINTER(C.c_char_p), C.POINTER(vp)]
    L.sw_full_batch_f32_lang.argtypes = [vp, C.POINTER(FullParams), C.POINTER(fp), C.POINTER(ci), ci,
                                         C.POINTER(C.c_char_p), C.POINTER(vp)]
    L.sw_host_alloc.restype = vp
    L.sw_host_alloc.argtypes = [C.c_size_t]
    L.sw_host_free.argtypes = [vp]
    L.sw_result_n_segments.argtypes = [vp]
    L.sw_result_segment_text.restype = C.c_char_p
    L.sw_result_segment_text.argtypes = [vp, ci]
    L.sw_result_segment_t0.restype = C.c_int64
    L.sw_result_segment_t0.argtypes = [vp, ci]
    L.sw_result_segment_t1.restype = C.c_int64
    L.sw_result_segment_t1.argtypes = [vp, ci]
    L.sw_result_segment_speaker_turn_next.argtypes = [vp, ci]
    L.sw_result_n_tokens.argtypes = [vp, ci]
    L.sw_result_token_data.restype = TokenData
    L.sw_result_token_data.argtypes = [vp, ci, ci]
    for n in ("lang_id", "n_decode_steps", "n_windows"):
        getattr(L, "sw_result_" + n).argtypes = [vp]
    L.sw_result_free.argtypes = [vp]
    L.sw_ctx_get_stats.argtypes = [vp, C.POINTER(Stats), ci]
    L.sw_ctx_set_kernel_timing.argtypes = [vp, ci]
    L.sw_mel_pcm16.argtypes = [vp, C.POINTER(C.c_int16), ci, fp, C.POINTER(ci)]
    L.sw_mel_f32.argtypes = [vp, fp, ci, fp, C.POINTER(ci)]
    L.sw_encode.argtypes = [vp, fp, ci, fp]
    L.sw_decode_logits.argtypes = [vp, C.POINTER(C.c_int32), ci, ci, fp]
    _lib = L
    return L


def last_error():
    return lib().sw_last_error().decode(errors="replace")


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _tok(t):
    return dict(id=t.id, tid=t.tid, p=t.p, plog=t.plog, pt=t.pt, ptsum=t.ptsum, t0=t.t0, t1=t.t1,
                vlen=t.vlen)


class Engine:
    def __init__(self, model_path, device=0, max_batch=64, max_beams=5, n_lanes=0):
        self.L = lib()
        p = self.L.sw_ctx_default_params()
        p.device, p.max_batch, p.max_beams, p.n_lanes = device, max_batch, max_beams, n_lanes
        self.h = self.L.sw_ctx_create(model_path.encode(), C.byref(p))
        if not self.h:
            raise RuntimeError("sw_ctx_create: " + last_error())
        self.info = ModelInfo()
        self.L.sw_ctx_model_info(self.h, C.byref(self.info))
        self._keep = []

    def close(self):
        if self.h:
            self.L.sw_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def token_str(self, i):
        return self.L.sw_token_to_str(self.h, i)

    def default_params(self, strategy=0, **kw):
        p = self.L.sw_full_default_params(strategy)
        for k, v in kw.items():
            if isinstance(v, str):
                v = v.encode()
                self._keep.append(v)
            setattr(p, k, v)
        return p

    def _collect(self, r):
        L = self.L
        segs = []
        for i in range(L.sw_result_n_segments(r)):
            toks = [_tok(L.sw_result_token_data(r, i, j)) for j in range(L.sw_result_n_tokens(r, i))]
            segs.append(dict(text=L.sw_result_segment_text(r, i), t0=L.sw_result_segment_t0(r, i),
                             t1=L.sw_result_segment_t1(r, i),
                             speaker_turn_next=bool(L.sw_result_segment_speaker_turn_next(r, i)),
                             tokens=toks))
        out = dict(segments=segs, lang_id=L.sw_result_lang_id(r),
                   n_decode_steps=L.sw_result_n_decode_steps(r), n_windows=L.sw_result_n_windows(r))
        L.sw_result_free(r)
        return out

    def full_batch_pcm16(self, pcms, params, collect=True, languages=None):
        n = len(pcms)
        pcms = [np.ascontiguousarray(a, np.int16) for a in pcms]
        ptrs = (C.POINTER(C.c_int16) * n)(*[a.ctypes.data_as(C.POINTER(C.c_int16)) for a in pcms])
        lens = (C.c_int * n)(*[len(a) for a in pcms])
        res = (C.c_void_p * n)()
        if languages is not None:
            lg = (C.c_char_p * n)(*[None if x is None else x.encode() for x in languages])
            rc = self.L.sw_full_batch_pcm16_lang(self.h, C.byref(params), ptrs, lens, n, lg, res)
        else:
            rc = self.L.sw_full_batch_pcm16(self.h, C.byref(params), ptrs, lens, n, res)
        if rc:
            raise RuntimeError("sw_full_batch_pcm16 rc=%d: %s" % (rc, last_error()))
        if not collect:
            for r in res:
                self.L.sw_result_free(r)
            return None
        return [self._collect(r) for r in res]

    def full_batch_ptrs(self, ptrs, lens, n, params, languages=None):
        """bench path: ptrs/lens are prebuilt ctypes arrays (pinned host buffers); returns handles"""
        res = (C.c_void_p * n)()
        if languages is not None:
            rc = self.L.sw_full_batch_pcm16_lang(self.h, C.byref(params), ptrs, lens, n, languages, res)
        else:
            rc = self.L.sw_full_batch_pcm16(self.h, C.byref(params), ptrs, lens, n, res)
        if rc:
            raise RuntimeError("sw_full_batch_pcm16 rc=%d: %s" % (rc, last_error()))
        return res

    def full_f32(self, pcm, params):
        pcm = np.ascontiguousarray(pcm, np.float32)
        r = C.c_void_p()
        rc = self.L.sw_full(self.h, C.byref(params), _fp(pcm), len(pcm), C.byref(r))
        if rc:
            raise RuntimeError("sw_full rc=%d: %s" % (rc, last_error()))
        return self._collect(r)

    def mel_pcm16(self, pcm16):
        a = np.ascontiguousarray(pcm16, np.int16)
        n_len = C.c_int()
        if self.L.sw_mel_pcm16(self.h, a.ctypes.data_as(C.POINTER(C.c_int16)), len(a), None, C.byref(n_len)):
            raise RuntimeError(last_error())
        out = np.empty((self.info.n_mels, n_len.value), np.float32)
        if self.L.sw_mel_pcm16(self.h, a.ctypes.data_as(C.POINTER(C.c_int16)), len(a), _fp(out), C.byref(n_len)):
            raise RuntimeError(last_error())
        return out

    def mel_f32(self, pcm):
        a = np.ascontiguousarray(pcm, np.float32)
        n_len = C.c_int()
        if self.L.sw_mel_f32(self.h, _fp(a), len(a), None, C.byref(n_len)):
            raise RuntimeError(last_error())
        out = np.empty((self.info.n_mels, n_len.value), np.float32)
        if self.L.sw_mel_f32(self.h, _fp(a), len(a), _fp(out), C.byref(n_len)):
            raise RuntimeError(last_error())
        return out

    def encode(self, mel_windows, want_output=True):
        m = np.ascontiguousarray(mel_windows, np.float32)
        n = m.shape[0]
        assert m.shape[1:] == (self.info.n_mels, 3000)
        out = np.empty((n, 1500, self.info.n_audio_state), np.float32) if want_output else None
        if self.L.sw_encode(self.h, _fp(m), n, _fp(out) if want_output else None):
            raise RuntimeError(last_error())
        return out

    def decode_logits(self, tokens):
        t = np.ascontiguousarray(tokens, np.int32)
        n, k = t.shape
        out = np.empty((n, k, self.info.n_vocab), np.float32)
        if self.L.sw_decode_logits(self.h, t.ctypes.data_as(C.POINTER(C.c_int32)), n, k, _fp(out)):
            raise RuntimeError(last_error())
        return out

    def prosody_segments(self, pcm, segments, sample_rate=16000, **opts):
        """pcm: float32 or int16 samples of one utterance; segments: [(begin, end)] in samples."""
        a = np.ascontiguousarray(pcm)
        assert a.dtype in (np.float32, np.int16)
        n = len(segments)
        b = (C.c_int64 * n)(*[int(s[0]) for s in segments])
        e = (C.c_int64 * n)(*[int(s[1]) for s in segments])
        self.L.sw_prosody_default_opts.restype = ProsodyOpts
        o = self.L.sw_prosody_default_opts()
        for k, v in opts.items():
            setattr(o, k, v)
        out = (Prosody * n)()
        if a.dtype == np.float32:
            fn, ptr = self.L.sw_prosody_segments_f32, a.ctypes.data_as(C.POINTER(C.c_float))
        else:
            fn, ptr = self.L.sw_prosody_segments_pcm16, a.ctypes.data_as(C.POINTER(C.c_int16))
        fn.argtypes = [C.c_void_p, type(ptr), C.c_int64, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                       C.c_int, C.POINTER(ProsodyOpts), C.POINTER(Prosody)]
        if fn(self.h, ptr, len(a), sample_rate, b, e, n, C.byref(o), out):
            raise RuntimeError(last_error())
        res = []
        for p in out:
            d = dict(gender=p.gender.decode(), emotion=EMOTIONS[p.emotion],
                     speaker_vec=[float(x) for x in p.speaker_vec])
            for f in PROSODY_FLOATS:
                d[f] = float(getattr(p, f))
            res.append(d)
        return res

    def resample(self, pcm, sr_in, sr_out=16000):
        a = np.ascontiguousarray(pcm, np.float32)
        self.L.sw_resample_out_len.restype = C.c_int64
        self.L.sw_resample_out_len.argtypes = [C.c_int64, C.c_int, C.c_int]
        out = np.empty(self.L.sw_resample_out_len(len(a), sr_in, sr_out), np.float32)
        self.L.sw_resample_f32.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_int64, C.c_int, C.c_int,
                                           C.POINTER(C.c_float)]
        if len(a) and self.L.sw_resample_f32(self.h, _fp(a), len(a), sr_in, sr_out, _fp(out)):
            raise RuntimeError(last_error())
        return out

    def set_kernel_timing(self, on):
        self.L.sw_ctx_set_kernel_timing(self.h, int(on))

    def stats(self, reset=False):
        s = Stats()
        self.L.sw_ctx_get_stats(self.h, C.byref(s), int(reset))
        return {n: getattr(s, n) for n, _ in Stats._fields_}
