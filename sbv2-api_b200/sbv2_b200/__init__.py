"""ctypes binding of libsbv2_b200.so (include/sbv2_b200.h) plus a thin Python twin of the
reference's ``sbv2_bindings`` surface (crates/sbv2_bindings/src/sbv2.rs:19-166), used by the tests
and the benchmark.  There is no Python/torch compute path here: every call goes through the C ABI
into the CUDA library, and importing the module fails loudly when the library is missing.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsbv2_b200.so")


class Sbv2Error(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"[sbv2 status {status}] {message}")
        self.status = status
        self.message = message


OK, ERR_INVALID_ARGUMENT, ERR_PARSE, ERR_MODEL_NOT_FOUND, ERR_CUDA, ERR_UNSUPPORTED, ERR_INTERNAL = range(7)


class Utterance(C.Structure):
    _fields_ = [("bert", C.POINTER(C.c_float)), ("x_tst", C.POINTER(C.c_int64)), ("tones", C.POINTER(C.c_int64)),
                ("lang_ids", C.POINTER(C.c_int64)), ("t_x", C.c_int64), ("sid", C.c_int64),
                ("style_vec", C.POINTER(C.c_float)), ("sdp_ratio", C.c_float), ("length_scale", C.c_float),
                ("noise_scale", C.c_float), ("noise_scale_w", C.c_float), ("noise_sdp", C.POINTER(C.c_float)),
                ("noise_zp", C.POINTER(C.c_float)), ("noise_zp_frames", C.c_int64)]


class TokenUtterance(C.Structure):
    _fields_ = [("input_ids", C.POINTER(C.c_int64)), ("attention_mask", C.POINTER(C.c_int64)), ("t_tok", C.c_int64),
                ("word2ph", C.POINTER(C.c_int32)), ("x_tst", C.POINTER(C.c_int64)), ("tones", C.POINTER(C.c_int64)),
                ("lang_ids", C.POINTER(C.c_int64)), ("t_x", C.c_int64), ("sid", C.c_int64), ("style_vec", C.POINTER(C.c_float)),
                ("sdp_ratio", C.c_float), ("length_scale", C.c_float), ("noise_scale", C.c_float), ("noise_scale_w", C.c_float)]


class TokenSentence(C.Structure):
    _fields_ = [("token_ids", C.POINTER(C.c_int64)), ("attention_mask", C.POINTER(C.c_int64)), ("word2ph", C.POINTER(C.c_int32)),
                ("t_tok", C.c_int64), ("phones", C.POINTER(C.c_int64)), ("tones", C.POINTER(C.c_int64)),
                ("lang_ids", C.POINTER(C.c_int64)), ("t_x", C.c_int64), ("line_index", C.c_int64)]


class Sentence(C.Structure):
    _fields_ = [("bert", C.POINTER(C.c_float)), ("phones", C.POINTER(C.c_int64)), ("tones", C.POINTER(C.c_int64)),
                ("lang_ids", C.POINTER(C.c_int64)), ("t_x", C.c_int64), ("line_index", C.c_int64)]


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python sbv2-api_b200/build.py` "
                          "(there is no fallback implementation)")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i64, i32, f32 = C.c_void_p, C.c_size_t, C.c_int64, C.c_int32, C.c_float
    pf, pi64, pi32 = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_int32)
    sig = {
        "sbv2_last_error": (C.c_char_p, []),
        "sbv2_free": (None, [vp]),
        "sbv2_alloc": (vp, [sz]),
        "sbv2_alloc_pinned": (vp, [sz]),
        "sbv2_set_last_error": (None, [C.c_char_p]),
        "sbv2_version": (C.c_char_p, []),
        "sbv2_device_count": (C.c_int, []),
        "sbv2_model_create": (C.c_int, [vp, sz, C.c_int, C.c_int, C.POINTER(vp)]),
        "sbv2_model_destroy": (None, [vp]),
        "sbv2_model_metadata": (C.c_int, [vp, C.c_char_p, C.POINTER(vp), C.POINTER(sz)]),
        "sbv2_model_describe": (C.c_int, [vp, C.POINTER(C.c_char_p)]),
        "sbv2_bert_predict": (C.c_int, [vp, pi64, pi64, i64, pf]),
        "sbv2_bert_predict_batch": (C.c_int, [vp, pi64, pi64, C.c_int, i64, pf]),
        "sbv2_bert_hidden_size": (C.c_int, [vp, C.POINTER(C.c_int)]),
        "sbv2_synthesize": (C.c_int, [vp, pf, pi64, pi64, pi64, i64, i64, pf, f32, f32, f32, f32, C.POINTER(pf), pi64]),
        "sbv2_synthesize_from_tokens": (C.c_int, [vp, vp, pi64, pi64, i64, pi32, pi64, pi64, pi64, i64, i64, pf, f32, f32, f32, f32,
                                                  C.POINTER(pf), pi64]),
        "sbv2_synthesize_from_tokens_batch": (C.c_int, [vp, vp, C.POINTER(TokenUtterance), C.c_int, pi64, C.POINTER(pf), pi64, pi64]),
        "sbv2_holder_easy_synthesize_tokens": (C.c_int, [vp, C.c_char_p, C.POINTER(TokenSentence), C.c_int, i64, i32, i64, f32, f32, f32,
                                                         C.POINTER(vp), C.POINTER(sz)]),
        "sbv2_onnx_bind_report": (C.c_int, [vp, sz, C.c_int, C.POINTER(vp)]),
        "sbv2_model_seed": (C.c_int, [vp, C.c_uint64]),
        "sbv2_synthesize_with_noise": (C.c_int, [vp, pf, pi64, pi64, pi64, i64, i64, pf, f32, f32, f32, f32, pf, pf, i64,
                                                 C.POINTER(pf), pi64, pi32, C.POINTER(pi32), pi64]),
        "sbv2_synthesize_batch": (C.c_int, [vp, C.POINTER(Utterance), C.c_int, C.POINTER(pf), pi64, C.POINTER(pi32),
                                            C.POINTER(pi32)]),
        "sbv2_batch_upload": (C.c_int, [vp, C.POINTER(Utterance), C.c_int, C.POINTER(vp)]),
        "sbv2_batch_run": (C.c_int, [vp, vp, pi64]),
        "sbv2_batch_download": (C.c_int, [vp, vp, C.POINTER(pf), pi64]),
        "sbv2_batch_free": (None, [vp]),
        "sbv2_model_launch_count": (i64, [vp]),
        "sbv2_model_stream": (vp, [vp]),
        "sbv2_decode_batch": (C.c_int, [vp, C.POINTER(pf), pi64, pi64, C.c_int, C.POINTER(pf), pi64]),
        "sbv2_debug_fetch": (C.c_int, [vp, C.c_char_p, C.POINTER(pf), pi64, pi64]),
        "sbv2_model_enable_timing": (C.c_int, [vp, C.c_int]),
        "sbv2_model_region_ms": (C.c_int, [vp, C.c_char_p, pf]),
        "sbv2_parse_sbv2file": (C.c_int, [vp, sz, C.POINTER(vp), C.POINTER(sz), C.POINTER(vp), C.POINTER(sz)]),
        "sbv2_load_style": (C.c_int, [vp, sz, C.POINTER(pf), pi64, pi64]),
        "sbv2_load_style_npy_base64": (C.c_int, [C.c_char_p, sz, C.POINTER(pf), pi64, pi64]),
        "sbv2_get_style_vector": (C.c_int, [pf, i64, i64, i32, f32, pf]),
        "sbv2_wav_from_f32": (C.c_int, [pf, i64, C.POINTER(vp), C.POINTER(sz)]),
        "sbv2_wav_pcm16_from_f32": (C.c_int, [pf, i64, C.POINTER(vp), C.POINTER(sz)]),
        "sbv2_holder_new": (C.c_int, [vp, sz, vp, sz, i64, C.c_int, C.POINTER(vp)]),
        "sbv2_holder_free": (None, [vp]),
        "sbv2_holder_load_sbv2file": (C.c_int, [vp, C.c_char_p, vp, sz]),
        "sbv2_holder_load": (C.c_int, [vp, C.c_char_p, vp, sz, vp, sz]),
        "sbv2_holder_load_aivmx": (C.c_int, [vp, C.c_char_p, vp, sz]),
        "sbv2_holder_unload": (C.c_int, [vp, C.c_char_p, C.POINTER(C.c_int)]),
        "sbv2_holder_models": (C.c_int, [vp, C.POINTER(vp)]),
        "sbv2_holder_loaded_count": (C.c_int, [vp, C.POINTER(C.c_int)]),
        "sbv2_holder_bert_hidden_size": (C.c_int, [vp, C.POINTER(C.c_int)]),
        "sbv2_holder_get_style_vector": (C.c_int, [vp, C.c_char_p, i32, f32, pf]),
        "sbv2_holder_bert_features": (C.c_int, [vp, pi64, pi64, i64, pi32, C.POINTER(pf), pi64]),
        "sbv2_holder_easy_synthesize": (C.c_int, [vp, C.c_char_p, C.POINTER(Sentence), C.c_int, i64, i32, i64, f32, f32, f32,
                                                  C.POINTER(vp), C.POINTER(sz)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    lib._sbv2_signatures = sig
    return lib


lib = _load()
EXPORTED_SYMBOLS = sorted(lib._sbv2_signatures)

_debug_lib = None


def debug_lib() -> C.CDLL:
    """libsbv2_b200_debug.so: the same objects plus the kernel unit-test / tracing hooks (sbv2_debug_conv_compare,
    _conv_trace, _pair_compare, _attn_trace, _mma_rate*, _flow_attention, _rel_attention, _convflow_spline, _durations,
    _umma_layer, _dec_post, _bert_bucket_table, _deberta_attention), which the product library does not export."""
    global _debug_lib
    if _debug_lib is None:
        path = os.path.join(_HERE, "libsbv2_b200_debug.so")
        if not os.path.exists(path):
            raise ImportError(f"{path} is missing: build it with `python sbv2-api_b200/build.py`")
        _debug_lib = C.CDLL(path)
        _debug_lib.sbv2_last_error.restype = C.c_char_p
    return _debug_lib


def _debug_check(status: int) -> None:
    if status != OK:
        raise Sbv2Error(status, debug_lib().sbv2_last_error().decode("utf-8", "replace"))


def debug_bert_bucket_table(span: int) -> np.ndarray:
    """The DeBERTa relative-position bucket table of `span` position buckets as the model builds it at load: entry
    d + R for d = -R..R, R = (len - 1) // 2 being the bound beyond which every distance reads the row of +-R."""
    D = debug_lib()
    r = C.c_int(0)
    _debug_check(D.sbv2_debug_bert_bucket_table(C.c_int(span), C.byref(r), None))
    out = np.zeros(2 * r.value + 1, np.int32)
    _debug_check(D.sbv2_debug_bert_bucket_table(C.c_int(span), C.byref(r), out.ctypes.data_as(C.POINTER(C.c_int))))
    return out


DEBERTA_ATTN_MODES = {"single": 0, "multi": 1, "exact-multi": 2, "simt": 3}


def debug_deberta_attention(qkv: np.ndarray, pos_k: np.ndarray, pos_q: np.ndarray, lens, heads: int, mode: str,
                            far_pairs: bool = True, sc: float = 16.0, reps: int = 0):
    """One DeBERTa attention launch (sbv2_debug_deberta_attention) on a ragged batch: qkv fp16 [terms, sum(lens), 3*heads*64],
    pos_k / pos_q fp16 [terms, 2*span, heads*64]; terms = 2 (the split terms of values scaled by sc) for mode "exact-multi",
    else 1.  Returns the context, fp16 [terms, sum(lens), heads*64] (exact-multi: the two terms of context * sc); with
    reps > 0, (context, mean ms of `reps` more launches timed with CUDA events)."""
    terms = 2 if mode == "exact-multi" else 1
    lens_a = np.ascontiguousarray(lens, dtype=np.int32)
    qkv = np.ascontiguousarray(qkv, dtype=np.float16).reshape(terms, int(lens_a.sum()), 3 * heads * 64)
    pos_k = np.ascontiguousarray(pos_k, dtype=np.float16).reshape(terms, -1, heads * 64)
    pos_q = np.ascontiguousarray(pos_q, dtype=np.float16).reshape(pos_k.shape)
    out = np.zeros((terms, int(lens_a.sum()), heads * 64), np.float16)
    u16, ms = C.POINTER(C.c_uint16), C.c_float(0.0)
    _debug_check(debug_lib().sbv2_debug_deberta_attention(
        qkv.ctypes.data_as(u16), pos_k.ctypes.data_as(u16), pos_q.ctypes.data_as(u16), lens_a.ctypes.data_as(C.POINTER(C.c_int)),
        len(lens_a), heads, pos_k.shape[1] // 2, DEBERTA_ATTN_MODES[mode], int(bool(far_pairs)), C.c_float(sc), reps, C.byref(ms),
        out.ctypes.data_as(u16)))
    return (out, ms.value) if reps > 0 else out


def _check(status: int) -> None:
    if status != OK:
        raise Sbv2Error(status, lib.sbv2_last_error().decode("utf-8", "replace"))


def _pf(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _pi64(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _i64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int64)


class _Owned:
    """Keeps a library-allocated buffer alive for the numpy views cut from it (zero-copy results)."""

    def __init__(self, ptr):
        self.ptr = C.cast(ptr, C.c_void_p)

    def __del__(self):
        try:
            if self.ptr:
                lib.sbv2_free(self.ptr)
        except Exception:
            pass


def _take(ptr, n: int, dtype, copy: bool = True) -> np.ndarray:
    """n elements of a library-allocated buffer: copied out (buffer released) or as a zero-copy
    view that releases the buffer when it is garbage collected."""
    if n == 0:
        lib.sbv2_free(C.cast(ptr, C.c_void_p))
        return np.zeros(0, dtype=dtype)
    if copy:
        arr = np.ctypeslib.as_array(ptr, shape=(n,)).copy()
        lib.sbv2_free(C.cast(ptr, C.c_void_p))
        return arr.astype(dtype, copy=False)
    owner = _Owned(ptr)
    buf = (C.c_byte * (n * np.dtype(dtype).itemsize)).from_address(owner.ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=n)
    _OWNERS[id(buf)] = owner  # tie the owner's lifetime to the ctypes buffer the views reference
    import weakref
    weakref.finalize(buf, _OWNERS.pop, id(buf), None)
    return arr


_OWNERS = {}


def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
    """Uninitialised array in page-locked host memory (sbv2_alloc_pinned): inputs that live here are read by the copy
    engine in place instead of being staged."""
    shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
    n = int(np.prod(shape)) if shape else 1
    p = lib.sbv2_alloc_pinned(max(1, n * np.dtype(dtype).itemsize))
    if not p:
        raise MemoryError("sbv2_alloc_pinned failed")
    return _take(C.cast(p, C.POINTER(C.c_byte)), n * np.dtype(dtype).itemsize, np.uint8, copy=False).view(dtype).reshape(shape)


def pinned_copy(a) -> np.ndarray:
    a = np.asarray(a)
    out = pinned_empty(a.shape, a.dtype)
    out[...] = a
    return out


def onnx_bind_report(onnx_bytes: bytes, bert: bool) -> dict:
    """Which initializer every canonical weight name binds to (structural binding of anonymous exports); CPU only."""
    p = C.c_void_p()
    _check(lib.sbv2_onnx_bind_report(onnx_bytes, len(onnx_bytes), 1 if bert else 0, C.byref(p)))
    s = C.string_at(p).decode()
    lib.sbv2_free(p)
    return json.loads(s)


def device_count() -> int:
    return int(lib.sbv2_device_count())


def version() -> str:
    return lib.sbv2_version().decode()


# ---- asset helpers -----------------------------------------------------------------------------

def parse_sbv2file(data: bytes) -> Tuple[bytes, bytes]:
    """-> (style_vectors_json, model_onnx); crates/sbv2_core/src/sbv2file.rs:15-37."""
    sj, on = C.c_void_p(), C.c_void_p()
    sn, onn = C.c_size_t(), C.c_size_t()
    _check(lib.sbv2_parse_sbv2file(data, len(data), C.byref(sj), C.byref(sn), C.byref(on), C.byref(onn)))
    style = C.string_at(sj, sn.value)
    onnx = C.string_at(on, onn.value)
    lib.sbv2_free(sj)
    lib.sbv2_free(on)
    return style, onnx


def load_style(json_bytes: bytes) -> np.ndarray:
    p = C.POINTER(C.c_float)()
    r, c = C.c_int64(), C.c_int64()
    _check(lib.sbv2_load_style(json_bytes, len(json_bytes), C.byref(p), C.byref(r), C.byref(c)))
    return _take(p, r.value * c.value, np.float32).reshape(r.value, c.value)


def load_style_npy_base64(b64: bytes) -> np.ndarray:
    p = C.POINTER(C.c_float)()
    r, c = C.c_int64(), C.c_int64()
    _check(lib.sbv2_load_style_npy_base64(b64, len(b64), C.byref(p), C.byref(r), C.byref(c)))
    return _take(p, r.value * c.value, np.float32).reshape(r.value, c.value)


def get_style_vector(style_vectors: np.ndarray, style_id: int, weight: float) -> np.ndarray:
    sv = _f32(style_vectors)
    out = np.zeros(sv.shape[1], dtype=np.float32)
    _check(lib.sbv2_get_style_vector(_pf(sv), sv.shape[0], sv.shape[1], style_id, weight, _pf(out)))
    return out


def wav_from_f32(samples: np.ndarray) -> bytes:
    s = _f32(samples).reshape(-1)
    p, n = C.c_void_p(), C.c_size_t()
    _check(lib.sbv2_wav_from_f32(_pf(s), s.size, C.byref(p), C.byref(n)))
    out = C.string_at(p, n.value)
    lib.sbv2_free(p)
    return out


def wav_pcm16_from_f32(samples: np.ndarray) -> bytes:
    s = _f32(samples).reshape(-1)
    p, n = C.c_void_p(), C.c_size_t()
    _check(lib.sbv2_wav_pcm16_from_f32(_pf(s), s.size, C.byref(p), C.byref(n)))
    out = C.string_at(p, n.value)
    lib.sbv2_free(p)
    return out


# ---- model::load_model / synthesize / bert::predict ----------------------------------------------

class Model:
    """One ``ort::Session`` replacement (``model::load_model``, crates/sbv2_core/src/model.rs:6-50)."""

    def __init__(self, onnx_bytes: bytes, bert: bool, device: int = 0):
        self._h = C.c_void_p()
        self.is_bert = bool(bert)
        _check(lib.sbv2_model_create(onnx_bytes, len(onnx_bytes), 1 if bert else 0, device, C.byref(self._h)))

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            lib.sbv2_model_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def describe(self) -> dict:
        s = C.c_char_p()
        _check(lib.sbv2_model_describe(self._h, C.byref(s)))
        return json.loads(s.value.decode())

    def metadata(self, key: str) -> Optional[bytes]:
        v, n = C.c_void_p(), C.c_size_t()
        _check(lib.sbv2_model_metadata(self._h, key.encode(), C.byref(v), C.byref(n)))
        if not v:
            return None
        return C.string_at(v, n.value)

    @property
    def launch_count(self) -> int:
        return int(lib.sbv2_model_launch_count(self._h))

    @property
    def stream(self) -> int:
        return int(lib.sbv2_model_stream(self._h) or 0)

    def enable_timing(self, on: bool = True) -> None:
        _check(lib.sbv2_model_enable_timing(self._h, 1 if on else 0))

    def region_ms(self, region: str) -> float:
        ms = C.c_float()
        _check(lib.sbv2_model_region_ms(self._h, region.encode(), C.byref(ms)))
        return float(ms.value)

    def seed(self, seed: int) -> None:
        _check(lib.sbv2_model_seed(self._h, seed))

    def debug_fetch(self, name: str) -> np.ndarray:
        p = C.POINTER(C.c_float)()
        r, c = C.c_int64(), C.c_int64()
        _check(lib.sbv2_debug_fetch(self._h, name.encode(), C.byref(p), C.byref(r), C.byref(c)))
        return _take(p, r.value * c.value, np.float32).reshape(r.value, c.value)

    # -- bert::predict (crates/sbv2_core/src/bert.rs:6-24)
    def hidden_size(self) -> int:
        h = C.c_int()
        _check(lib.sbv2_bert_hidden_size(self._h, C.byref(h)))
        return h.value

    def predict(self, token_ids: Sequence[int], attention_masks: Sequence[int]) -> np.ndarray:
        ids, mask = _i64(token_ids), _i64(attention_masks)
        if ids.shape != mask.shape or ids.ndim != 1:
            raise Sbv2Error(ERR_INVALID_ARGUMENT, "token_ids and attention_masks must be 1-D and equal length")
        out = np.zeros((ids.size, self.hidden_size()), dtype=np.float32)
        _check(lib.sbv2_bert_predict(self._h, _pi64(ids), _pi64(mask), ids.size, _pf(out)))
        return out

    def predict_batch(self, token_ids: np.ndarray, attention_masks: np.ndarray) -> np.ndarray:
        ids, mask = _i64(token_ids), _i64(attention_masks)
        if ids.shape != mask.shape or ids.ndim != 2:
            raise Sbv2Error(ERR_INVALID_ARGUMENT, "token_ids and attention_masks must be [batch, s]")
        out = np.zeros((ids.shape[0], ids.shape[1], self.hidden_size()), dtype=np.float32)
        _check(lib.sbv2_bert_predict_batch(self._h, _pi64(ids), _pi64(mask), ids.shape[0], ids.shape[1], _pf(out)))
        return out

    # -- model::synthesize (crates/sbv2_core/src/model.rs:53-111)
    def synthesize(self, bert_ori, x_tst, spk_ids, tones, lang_ids, style_vector, sdp_ratio: float, length_scale: float,
                   noise_scale: float, noise_scale_w: float) -> np.ndarray:
        """Returns the reference's ``Array3<f32>`` of shape [1, 1, N]."""
        bert, x, t, l, sv = _f32(bert_ori), _i64(x_tst), _i64(tones), _i64(lang_ids), _f32(style_vector)
        spk = _i64(spk_ids).reshape(-1)
        if bert.ndim != 2 or bert.shape[1] != x.size or t.size != x.size or l.size != x.size or spk.size != 1:
            raise Sbv2Error(ERR_INVALID_ARGUMENT, "inconsistent input shapes")
        p, n = C.POINTER(C.c_float)(), C.c_int64()
        _check(lib.sbv2_synthesize(self._h, _pf(bert), _pi64(x), _pi64(t), _pi64(l), x.size, int(spk[0]), _pf(sv), sdp_ratio,
                                   length_scale, noise_scale, noise_scale_w, C.byref(p), C.byref(n)))
        return _take(p, n.value, np.float32).reshape(1, 1, -1)

    def synthesize_from_tokens(self, bert_model: "Model", token_ids, attention_masks, word2ph, x_tst, sid: int, tones, lang_ids,
                               style_vector, sdp_ratio: float, length_scale: float, noise_scale: float,
                               noise_scale_w: float) -> np.ndarray:
        """bert::predict -> word2ph expansion -> synthesize with the BERT features kept on the device (SURVEY §8f row 1).
        -> audio [N]."""
        ids, mask, w2p = _i64(token_ids), _i64(attention_masks), np.ascontiguousarray(word2ph, dtype=np.int32)
        x, t, l, sv = _i64(x_tst), _i64(tones), _i64(lang_ids), _f32(style_vector)
        if ids.size != mask.size or w2p.size != ids.size or t.size != x.size or l.size != x.size:
            raise Sbv2Error(ERR_INVALID_ARGUMENT, "inconsistent input shapes")
        p, n = C.POINTER(C.c_float)(), C.c_int64()
        _check(lib.sbv2_synthesize_from_tokens(self._h, bert_model._h, _pi64(ids), _pi64(mask), ids.size,
                                               w2p.ctypes.data_as(C.POINTER(C.c_int32)), _pi64(x), _pi64(t), _pi64(l), x.size, sid,
                                               _pf(sv), sdp_ratio, length_scale, noise_scale, noise_scale_w, C.byref(p), C.byref(n)))
        return _take(p, n.value, np.float32)

    def synthesize_from_tokens_batch(self, bert_model: "Model", sentences: Sequence[dict], pause_after: Optional[Sequence[int]] = None):
        """sentences[i]: dict(token_ids, word2ph, x_tst, tones, lang_ids, style_vec[, sid, sdp_ratio, length_scale,
        noise_scale, noise_scale_w]).  -> (audio [total] incl. the pauses, samples per sentence int64 [batch])"""
        B = len(sentences)
        arr = (TokenUtterance * B)()
        keep = []
        for i, u in enumerate(sentences):
            ids, w2p = _i64(u["token_ids"]), np.ascontiguousarray(u["word2ph"], dtype=np.int32)
            mask = _i64(u.get("attention_mask", np.ones_like(ids)))
            x, t, l, sv = _i64(u["x_tst"]), _i64(u["tones"]), _i64(u["lang_ids"]), _f32(u["style_vec"])
            keep += [ids, mask, w2p, x, t, l, sv]
            a = arr[i]
            a.input_ids, a.attention_mask, a.t_tok, a.word2ph = _pi64(ids), _pi64(mask), ids.size, w2p.ctypes.data_as(C.POINTER(C.c_int32))
            a.x_tst, a.tones, a.lang_ids, a.t_x = _pi64(x), _pi64(t), _pi64(l), x.size
            a.sid, a.style_vec = int(u.get("sid", 0)), _pf(sv)
            a.sdp_ratio, a.length_scale = float(u.get("sdp_ratio", 0.0)), float(u.get("length_scale", 1.0))
            a.noise_scale, a.noise_scale_w = float(u.get("noise_scale", 0.677)), float(u.get("noise_scale_w", 0.8))
        pa = _i64(pause_after) if pause_after is not None else None
        p, total = C.POINTER(C.c_float)(), C.c_int64()
        ns = np.zeros(B, dtype=np.int64)
        _check(lib.sbv2_synthesize_from_tokens_batch(self._h, bert_model._h, arr, B, _pi64(pa) if pa is not None else None, C.byref(p),
                                                     C.byref(total), _pi64(ns)))
        return _take(p, total.value, np.float32), ns

    def synthesize_with_noise(self, bert_ori, x_tst, sid: int, tones, lang_ids, style_vector, sdp_ratio, length_scale,
                              noise_scale, noise_scale_w, noise_sdp, noise_zp):
        """-> (audio [N], durations int32 [T_x], frame2ph int32 [T_y])."""
        bert, x, t, l, sv = _f32(bert_ori), _i64(x_tst), _i64(tones), _i64(lang_ids), _f32(style_vector)
        nsdp, nzp = _f32(noise_sdp), _f32(noise_zp)
        if nsdp.shape != (2, x.size) or nzp.ndim != 2:
            raise Sbv2Error(ERR_INVALID_ARGUMENT, "noise_sdp must be [2, t_x] and noise_zp [C, frames]")
        p, n = C.POINTER(C.c_float)(), C.c_int64()
        dur = np.zeros(x.size, dtype=np.int32)
        f2p, ty = C.POINTER(C.c_int32)(), C.c_int64()
        _check(lib.sbv2_synthesize_with_noise(self._h, _pf(bert), _pi64(x), _pi64(t), _pi64(l), x.size, sid, _pf(sv),
                                              sdp_ratio, length_scale, noise_scale, noise_scale_w, _pf(nsdp), _pf(nzp),
                                              nzp.shape[1], C.byref(p), C.byref(n),
                                              dur.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(f2p), C.byref(ty)))
        audio = _take(p, n.value, np.float32)
        frame2ph = _take(f2p, ty.value, np.int32)
        return audio, dur, frame2ph

    def _utterances(self, utts: Sequence[dict]):
        keep = []
        arr = (Utterance * len(utts))()
        for i, u in enumerate(utts):
            bert, x, t, l, sv = _f32(u["bert"]), _i64(u["x_tst"]), _i64(u["tones"]), _i64(u["lang_ids"]), _f32(u["style_vec"])
            if bert.ndim != 2 or bert.shape[1] != x.size or t.size != x.size or l.size != x.size:
                raise Sbv2Error(ERR_INVALID_ARGUMENT, f"utterance {i}: inconsistent input shapes")
            keep += [bert, x, t, l, sv]
            a = arr[i]
            a.bert, a.x_tst, a.tones, a.lang_ids, a.style_vec = _pf(bert), _pi64(x), _pi64(t), _pi64(l), _pf(sv)
            a.t_x, a.sid = x.size, int(u.get("sid", 0))
            a.sdp_ratio, a.length_scale = float(u.get("sdp_ratio", 0.0)), float(u.get("length_scale", 1.0))
            a.noise_scale, a.noise_scale_w = float(u.get("noise_scale", 0.677)), float(u.get("noise_scale_w", 0.8))
            if u.get("noise_sdp") is not None:
                ns = _f32(u["noise_sdp"])
                keep.append(ns)
                a.noise_sdp = _pf(ns)
            if u.get("noise_zp") is not None:
                nz = _f32(u["noise_zp"])
                keep.append(nz)
                a.noise_zp = _pf(nz)
                a.noise_zp_frames = nz.shape[1]
        return arr, keep

    def synthesize_batch(self, utts: Sequence[dict], want_alignment: bool = False):
        """Var-len batched extension. -> list of audio arrays (and durations / frame2ph lists)."""
        arr, keep = self._utterances(utts)
        B = len(utts)
        p = C.POINTER(C.c_float)()
        ns = np.zeros(B, dtype=np.int64)
        pd, pf2 = C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)()
        _check(lib.sbv2_synthesize_batch(self._h, arr, B, C.byref(p), _pi64(ns), C.byref(pd) if want_alignment else None,
                                         C.byref(pf2) if want_alignment else None))
        flat = _take(p, int(ns.sum()), np.float32, copy=False)
        offs = np.concatenate([[0], np.cumsum(ns)])
        audios = [flat[offs[i]:offs[i + 1]] for i in range(B)]
        if not want_alignment:
            return audios
        hop = self.describe()["hop"]
        tx = [int(u_.t_x) for u_ in arr]
        d = _take(pd, int(sum(tx)), np.int32)
        f = _take(pf2, int(ns.sum() // hop), np.int32)
        xo = np.concatenate([[0], np.cumsum(tx)])
        yo = offs // hop
        return audios, [d[xo[i]:xo[i + 1]] for i in range(B)], [f[yo[i]:yo[i + 1]] for i in range(B)]

    def decode_batch(self, zs: Sequence[np.ndarray], sids: Optional[Sequence[int]] = None) -> List[np.ndarray]:
        """HiFi-GAN decoder alone: zs[b] float32 [192, T_y[b]]."""
        B = len(zs)
        z = [_f32(a) for a in zs]
        ptrs = (C.POINTER(C.c_float) * B)(*[_pf(a) for a in z])
        ty = _i64([a.shape[1] for a in z])
        sid = _i64(sids if sids is not None else [0] * B)
        p = C.POINTER(C.c_float)()
        ns = np.zeros(B, dtype=np.int64)
        _check(lib.sbv2_decode_batch(self._h, ptrs, _pi64(ty), _pi64(sid), B, C.byref(p), _pi64(ns)))
        flat = _take(p, int(ns.sum()), np.float32)
        offs = np.concatenate([[0], np.cumsum(ns)])
        return [flat[offs[i]:offs[i + 1]] for i in range(B)]


class DeviceBatch:
    """Inputs resident in HBM (sbv2_batch_upload) for kernel-only timing."""

    def __init__(self, model: Model, utts: Sequence[dict]):
        self.model = model
        arr, keep = model._utterances(utts)
        self._h = C.c_void_p()
        self.batch = len(utts)
        _check(lib.sbv2_batch_upload(model._h, arr, len(utts), C.byref(self._h)))

    def run(self) -> int:
        n = C.c_int64()
        _check(lib.sbv2_batch_run(self.model._h, self._h, C.byref(n)))
        return n.value

    def download(self) -> List[np.ndarray]:
        p = C.POINTER(C.c_float)()
        ns = np.zeros(self.batch, dtype=np.int64)
        _check(lib.sbv2_batch_download(self.model._h, self._h, C.byref(p), _pi64(ns)))
        flat = _take(p, int(ns.sum()), np.float32)
        offs = np.concatenate([[0], np.cumsum(ns)])
        return [flat[offs[i]:offs[i + 1]] for i in range(self.batch)]

    def close(self):
        if self._h:
            lib.sbv2_batch_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def load_model(model_file: bytes, bert: bool, device: int = 0) -> Model:
    return Model(model_file, bert, device)


# ---- TTSModelHolder twin (crates/sbv2_core/src/tts.rs:40-349, crates/sbv2_bindings/src/sbv2.rs) ---

class TTSModelHolder:
    def __init__(self, bert_model_bytes: bytes, tokenizer_bytes: bytes = b"", max_loaded_models: Optional[int] = None,
                 device: int = 0):
        self._h = C.c_void_p()
        _check(lib.sbv2_holder_new(bert_model_bytes, len(bert_model_bytes), tokenizer_bytes, len(tokenizer_bytes),
                                   -1 if max_loaded_models is None else int(max_loaded_models), device, C.byref(self._h)))
        h = C.c_int()
        _check(lib.sbv2_holder_bert_hidden_size(self._h, C.byref(h)))
        self._bert_hidden = h.value

    def close(self):
        if self._h:
            lib.sbv2_holder_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def models(self) -> List[str]:
        p = C.c_void_p()
        _check(lib.sbv2_holder_models(self._h, C.byref(p)))
        s = C.string_at(p).decode()
        lib.sbv2_free(p)
        return [x for x in s.split("\n") if x]

    def loaded_count(self) -> int:
        n = C.c_int()
        _check(lib.sbv2_holder_loaded_count(self._h, C.byref(n)))
        return n.value

    def load_sbv2file(self, ident: str, sbv2_bytes: bytes) -> None:
        _check(lib.sbv2_holder_load_sbv2file(self._h, ident.encode(), sbv2_bytes, len(sbv2_bytes)))

    def load(self, ident: str, style_vectors_bytes: bytes, vits2_bytes: bytes) -> None:
        _check(lib.sbv2_holder_load(self._h, ident.encode(), style_vectors_bytes, len(style_vectors_bytes), vits2_bytes,
                                    len(vits2_bytes)))

    def load_aivmx(self, ident: str, aivmx_bytes: bytes) -> None:
        _check(lib.sbv2_holder_load_aivmx(self._h, ident.encode(), aivmx_bytes, len(aivmx_bytes)))

    def unload(self, ident: str) -> bool:
        f = C.c_int()
        _check(lib.sbv2_holder_unload(self._h, ident.encode(), C.byref(f)))
        return bool(f.value)

    def get_style_vector(self, ident: str, style_id: int, weight: float) -> np.ndarray:
        out = np.zeros(256, dtype=np.float32)
        _check(lib.sbv2_holder_get_style_vector(self._h, ident.encode(), style_id, weight, _pf(out)))
        return out

    def bert_features(self, token_ids, attention_masks, word2ph) -> np.ndarray:
        ids, mask = _i64(token_ids), _i64(attention_masks)
        w = np.ascontiguousarray(word2ph, dtype=np.int32)
        p, tx = C.POINTER(C.c_float)(), C.c_int64()
        _check(lib.sbv2_holder_bert_features(self._h, _pi64(ids), _pi64(mask), ids.size,
                                             w.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(p), C.byref(tx)))
        n = C.c_int64()  # rows = hidden size of the holder's DeBERTa: the library returns rows * t_x floats
        rows = self._bert_hidden
        return _take(p, rows * tx.value, np.float32).reshape(rows, tx.value)

    def easy_synthesize_tokens(self, ident: str, lines: Sequence[Optional[dict]], style_id: int, speaker_id: int,
                               sdp_ratio: float = 0.0, length_scale: float = 1.0, style_weight: float = 1.0) -> bytes:
        """``lines[i]`` is None for an empty line, else dict(token_ids, word2ph, phones, tones, lang_ids): the request's
        sentences run through DeBERTa and the synthesizer as one batch each, silences are written on the device."""
        sent = [(i, l) for i, l in enumerate(lines) if l is not None]
        arr = (TokenSentence * max(len(sent), 1))()
        keep = []
        for j, (i, l) in enumerate(sent):
            ids, w2p = _i64(l["token_ids"]), np.ascontiguousarray(l["word2ph"], dtype=np.int32)
            mask = _i64(l.get("attention_mask", np.ones_like(ids)))
            ph, t, lg = _i64(l["phones"]), _i64(l["tones"]), _i64(l["lang_ids"])
            keep += [ids, mask, w2p, ph, t, lg]
            a = arr[j]
            a.token_ids, a.attention_mask, a.word2ph, a.t_tok = _pi64(ids), _pi64(mask), w2p.ctypes.data_as(C.POINTER(C.c_int32)), ids.size
            a.phones, a.tones, a.lang_ids, a.t_x, a.line_index = _pi64(ph), _pi64(t), _pi64(lg), ph.size, i
        p, n = C.c_void_p(), C.c_size_t()
        _check(lib.sbv2_holder_easy_synthesize_tokens(self._h, ident.encode(), arr, len(sent), len(lines), style_id, speaker_id,
                                                      sdp_ratio, length_scale, style_weight, C.byref(p), C.byref(n)))
        out = C.string_at(p, n.value)
        lib.sbv2_free(p)
        return out

    def easy_synthesize(self, ident: str, lines: Sequence[Optional[dict]], style_id: int, speaker_id: int,
                        sdp_ratio: float = 0.0, length_scale: float = 1.0, style_weight: float = 1.0) -> bytes:
        """``lines[i]`` is None for an empty line, else dict(bert, phones, tones, lang_ids)."""
        sent = [(i, l) for i, l in enumerate(lines) if l is not None]
        arr = (Sentence * max(len(sent), 1))()
        keep = []
        for j, (i, l) in enumerate(sent):
            bert, ph, t, lg = _f32(l["bert"]), _i64(l["phones"]), _i64(l["tones"]), _i64(l["lang_ids"])
            keep += [bert, ph, t, lg]
            arr[j].bert, arr[j].phones, arr[j].tones, arr[j].lang_ids = _pf(bert), _pi64(ph), _pi64(t), _pi64(lg)
            arr[j].t_x, arr[j].line_index = ph.size, i
        p, n = C.c_void_p(), C.c_size_t()
        _check(lib.sbv2_holder_easy_synthesize(self._h, ident.encode(), arr, len(sent), len(lines), style_id, speaker_id,
                                               sdp_ratio, length_scale, style_weight, C.byref(p), C.byref(n)))
        out = C.string_at(p, n.value)
        lib.sbv2_free(p)
        return out
