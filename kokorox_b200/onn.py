"""Host-side mirror of the reference's inference seam, over the C ABI of ``include/kkx.h``.

Reference interface mirrored (same names, argument meaning and error behaviour):

* ``kokorox::onn::init_ort(dylib_path)``        /root/reference/kokorox/src/onn/mod.rs:19-49
* ``OrtKoko::new(model_path) -> Result<_, String>``          .../onn/ort_koko.rs:31-35
* ``OrtKoko::infer(tokens: Vec<Vec<i64>>, styles: Vec<Vec<f32>>, speed: f32)
      -> Result<ArrayD<f32>, Box<dyn Error>>``               .../onn/ort_koko.rs:37-91

The host language of the reference is Rust, which this image does not have; the Rust shim a
maintainer would add is in INTEGRATION.md, and this module is the same shim in Python (ctypes).
There is no CPU fallback: if ``libkkx.so`` is missing or no B200 is visible every call raises.
"""
from __future__ import annotations

import ctypes as C
import weakref
import os
import threading
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libkkx.so")

_lib = None
_lib_lock = threading.Lock()


class KkxError(RuntimeError):
    """Err(String) of the reference API (ort_koko.rs:31,42)."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"kkx error {code}: {msg}")
        self.code = code


def load_library(path: Optional[str] = None):
    """dlopen libkkx.so and declare the prototypes of include/kkx.h (and kkx_test.h)."""
    global _lib
    with _lib_lock:
        if _lib is not None and path is None:
            return _lib
        p = path or os.environ.get("KKX_LIB", LIB_PATH)
        if not os.path.exists(p):
            raise KkxError(-4, f"{p} not found: build it with `python -m kokorox_b200.build` "
                               "(there is no CPU fallback)")
        lib = C.CDLL(p)
        vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
        P = C.POINTER
        lib.kkx_version.restype = C.c_char_p
        lib.kkx_init.restype = C.c_int
        lib.kkx_create.argtypes = [C.c_char_p, C.c_int, P(vp)]
        lib.kkx_destroy.argtypes = [vp]
        lib.kkx_destroy.restype = None
        lib.kkx_last_error.argtypes = [vp]
        lib.kkx_last_error.restype = C.c_char_p
        lib.kkx_infer.argtypes = [vp, P(i64), i32, P(f32), f32, P(P(f32)), P(i64), P(i32)]
        lib.kkx_infer_batch.argtypes = [vp, i32, P(i64), P(i32), P(f32), P(f32), P(P(f32)), P(i64), P(i32)]
        lib.kkx_release.argtypes = [vp, P(f32)]
        lib.kkx_release.restype = None
        i16 = C.c_int16
        lib.kkx_load_voices.argtypes = [vp, P(f32), i32]
        lib.kkx_infer_batch_voices.argtypes = [vp, i32, P(i64), P(i32), P(i32), P(i32), P(f32), P(i32), P(f32),
                                               P(P(f32)), P(i64), P(i32)]
        lib.kkx_infer_batch_pcm16.argtypes = [vp, i32, P(i64), P(i32), P(f32), P(f32), P(P(i16)), P(i64), P(i32)]
        lib.kkx_release_pcm16.argtypes = [vp, P(i16)]
        lib.kkx_release_pcm16.restype = None
        u8 = C.c_uint8
        lib.kkx_infer_batch_g711.argtypes = [vp, i32, P(i64), P(i32), P(f32), P(f32), i32, P(P(u8)), P(i64), P(i32)]
        lib.kkx_release_g711.argtypes = [vp, P(u8)]
        lib.kkx_release_g711.restype = None
        lib.kkx_infer_batch_flac.argtypes = [vp, i32, P(i64), P(i32), P(f32), P(f32), P(P(u8)), P(i64), P(i64), P(i32)]
        lib.kkx_release_flac.argtypes = [vp, P(u8)]
        lib.kkx_release_flac.restype = None
        lib.kkx_infer_programs.argtypes = [vp, i32, P(i64), P(i32), P(f32), P(f32), i32, P(i32), i32, P(vp), P(i64),
                                           P(i64), P(i32)]
        lib.kkx_release_programs.argtypes = [vp, vp]
        lib.kkx_release_programs.restype = None
        lib.kkx_wav_header_pcm16.argtypes = [P(C.c_uint8), i64, i32]
        lib.kkx_wav_header_f32_stream.argtypes = [P(C.c_uint8), i32, i32]
        lib.kkx_encode_wav16_base64.argtypes = [P(i16), i64, i32, C.c_char_p, i64]
        lib.kkx_encode_wav16_base64.restype = i64
        lib.kkx_stage_batch.argtypes = [vp, i32, P(i64), P(i32), P(f32), P(f32)]
        lib.kkx_run_staged.argtypes = [vp, P(i64), P(i64)]
        lib.kkx_fetch_staged.argtypes = [vp, P(f32), i64, P(i64), P(i32)]
        lib.kkx_set_option.argtypes = [vp, C.c_char_p, i64]
        lib.kkx_get_stat.argtypes = [vp, C.c_char_p]
        lib.kkx_get_stat.restype = i64
        lib.kkx_set_noise.argtypes = [vp, P(f32), i64]
        lib.kkx_set_inject.argtypes = [vp, C.c_char_p, vp, i64]
        lib.kkx_set_inject_item.argtypes = [vp, i32, C.c_char_p, vp, i64]
        lib.kkx_debug_select.argtypes = [vp, C.c_int, i32]
        lib.kkx_submit.argtypes = [vp, P(i64), i32, P(f32), f32, P(i64)]
        lib.kkx_poll.argtypes = [vp, i64]
        lib.kkx_wait.argtypes = [vp, i64, P(P(f32)), P(i64), P(i32)]
        lib.kkx_convert_model_file.argtypes = [C.c_char_p, C.c_char_p, P(i32)]
        lib.kkx_test_tensor_specs.argtypes = [C.c_char_p, i64]
        lib.kkx_test_tensor_specs.restype = i64
        lib.kkx_test_conv_f16x3.argtypes = [C.c_int, P(f32), C.c_int, C.c_int, P(f32), P(f32), C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.c_int, P(f32)]
        lib.kkx_test_conv_f16x3_k.argtypes = [C.c_int, P(f32), C.c_int, C.c_int, P(f32), P(f32), C.c_int, C.c_int, C.c_int,
                                              C.c_int, C.c_int, C.c_int, P(f32), f32, P(f32)]
        lib.kkx_test_arb_conv_stream.argtypes = [C.c_int, P(f32), C.c_int, P(i32), C.c_int, P(f32), P(f32), P(f32), P(f32),
                                                 P(f32), C.c_int, C.c_int, P(f32), f32, C.c_int, C.c_int, P(f32), P(f32)]
        lib.kkx_test_resample_taps.argtypes = [i32, P(f32), i64]
        lib.kkx_test_resample_taps.restype = i64
        lib.kkx_test_resample.argtypes = [C.c_int, P(f32), i32, P(i64), i32, i32, P(f32), P(i16), P(u8)]
        lib.kkx_last_loudness.argtypes = [vp, i32, P(f32), P(f32), P(f32)]
        lib.kkx_test_loudness_design.argtypes = [C.c_double, P(C.c_double), P(f32), i64]
        lib.kkx_test_loudness_design.restype = i64
        lib.kkx_test_loudness.argtypes = [C.c_int, P(f32), i32, P(i64), i32, i32, P(f32), P(f32), P(f32)]
        lib.kkx_test_flac.argtypes = [C.c_int, P(i16), i32, P(i64), i32, P(u8), i64, P(i64)]
        lib.kkx_test_flac.restype = i64
        lib.kkx_test_attention_batch.argtypes = [C.c_int, P(f32), C.c_int, P(i32), P(i32), C.c_int, C.c_int, P(f32)]
        lib.kkx_debug_stage.argtypes = [vp, C.c_char_p, i32, P(f32), i64, P(i64), P(i64)]
        lib.kkx_debug_stage.restype = i64
        lib.kkx_debug_enable.argtypes = [vp, C.c_int]
        lib.kkx_profile_enable.argtypes = [vp, C.c_int]
        lib.kkx_profile_json.argtypes = [vp, C.c_char_p, i64]
        lib.kkx_profile_json.restype = i64
        if path is None:
            _lib = lib
        return lib


def parse_style_name(style_name: str, voice_ids) -> tuple:
    """The parsing half of TTSKoko::mix_styles (koko.rs:1255-1295): ``"af_sky"`` or ``"af_sky.4+af_nicole.5"`` ->
    ([voice ids], [f32 portions]).  A single voice is one entry with portion 1.0 (the reference copies the row);
    in a mix every ``name.weight`` part contributes ``weight * 0.1`` (f32, not renormalised); parts without a
    numeric weight are skipped like the reference's ``if let Ok(portion)``; unknown voices are errors with the
    reference's messages."""
    if "+" not in style_name:
        if style_name not in voice_ids:
            raise KkxError(-1, f"can not found from styles_map: {style_name}")
        return [voice_ids[style_name]], [np.float32(1.0)]
    vs, ps = [], []
    for part in style_name.split("+"):
        if "." in part:
            name, portion = part.split(".", 1)
            try:
                w = np.float32(float(portion))
            except ValueError:
                continue
            if name not in voice_ids:
                raise KkxError(-1, f"Voice '{name}' not found in available voices")
            vs.append(voice_ids[name])
            ps.append(np.float32(w * np.float32(0.1)))
    if not vs:
        raise KkxError(-1, f"Invalid voice mix format '{style_name}'. Use format: voice1.weight+voice2.weight "
                           "(e.g., jf_alpha.4+am_echo.6)")
    return vs, ps


def encode_audio(pcm: np.ndarray, sample_rate: int = 24000) -> str:
    """``encode_audio`` of the WebSocket server (kokorox-websocket/src/lib.rs:696-736) for a 16-bit PCM result
    (``infer_batch_pcm16``): base64 of a 44-byte PCM WAV header + the samples.  Host-side byte work in libkkx."""
    lib = load_library()
    a = np.ascontiguousarray(np.asarray(pcm, dtype=np.int16).reshape(-1))
    ptr = a.ctypes.data_as(C.POINTER(C.c_int16))
    n = lib.kkx_encode_wav16_base64(ptr, a.size, int(sample_rate), None, 0)
    if n < 0:
        raise KkxError(int(n), "encode_audio: bad argument")
    buf = C.create_string_buffer(int(n) + 1)
    lib.kkx_encode_wav16_base64(ptr, a.size, int(sample_rate), buf, int(n) + 1)
    return buf.raw[:int(n)].decode("ascii")


def wav_header(n_samples: Optional[int] = None, sample_rate: int = 24000, channels: int = 1) -> bytes:
    """44-byte WAV header: ``n_samples`` given -> the sized PCM16 mono header of ``encode_audio``
    (websocket lib.rs:707-731); ``None`` -> the streaming IEEE-float header of utils/wav.rs:19-43 (sizes are
    0xFFFFFFFF placeholders; the f32 result buffer follows as is, wav.rs:45-50)."""
    lib = load_library()
    buf = (C.c_uint8 * 44)()
    rc = (lib.kkx_wav_header_f32_stream(buf, int(channels), int(sample_rate)) if n_samples is None
          else lib.kkx_wav_header_pcm16(buf, int(n_samples), int(sample_rate)))
    if rc != 44:
        raise KkxError(int(rc), "wav_header: bad argument")
    return bytes(buf)


def convert_model_file(src: str, dst: str) -> int:
    """Host-only: read ``src`` the way ``kkx_create`` does (ONNX -- fp32 / fp16 / int8 / 4-bit variants -- or KKXW)
    and write the recovered state dict as a KKXW file.  Returns the tensor count."""
    lib = load_library()
    n = C.c_int32(0)
    rc = lib.kkx_convert_model_file(os.fsencode(src), os.fsencode(dst), C.byref(n))
    if rc != 0:
        raise KkxError(rc, (lib.kkx_last_error(None) or b"").decode())
    return int(n.value)


def library_tensor_specs():
    """[(name, shape)] the C++ loader expects (test hook; compared with weightfile.weight_specs)."""
    lib = load_library()
    n = lib.kkx_test_tensor_specs(None, 0)
    buf = C.create_string_buffer(int(n) + 1)
    lib.kkx_test_tensor_specs(buf, n + 1)
    out = []
    for line in buf.value.decode().splitlines():
        parts = line.split()
        out.append((parts[0], tuple(int(x) for x in parts[1:])))
    return out


def _fp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def init_ort(dylib_path: Optional[str] = None) -> None:
    """mod.rs:19-49.  ``dylib_path`` optionally names libkkx.so (the reference's ORT_DYLIB_PATH)."""
    lib = load_library(dylib_path)
    rc = lib.kkx_init()
    if rc != 0:
        raise KkxError(rc, (lib.kkx_last_error(None) or b"").decode())


class B200Koko:
    """Drop-in for ``OrtKoko`` (ort_koko.rs:13-91): ``new(model_path)`` then ``infer(...)``.

    Send + Sync like the reference type (ort_koko.rs:17-18): one instance may be shared between
    threads; calls serialise inside the library.
    """

    def __init__(self, model_path: str, device: int = 0):
        self._lib = load_library()
        self._ctx = C.c_void_p()
        rc = self._lib.kkx_create(os.fsencode(model_path), int(device), C.byref(self._ctx))
        if rc != 0:
            self._ctx = C.c_void_p()
            raise KkxError(rc, (self._lib.kkx_last_error(None) or b"").decode())
        self.device = device
        self._outstanding = 0
        self._closing = False
        self._count_lock = threading.RLock()   # re-entrant: a GC-run finalizer may fire inside the block

    @classmethod
    def new(cls, model_path: str, device: int = 0) -> "B200Koko":
        return cls(model_path, device)

    # -- lifetime -------------------------------------------------------------------------
    def close(self) -> None:
        """Destroy the session.  If waveforms returned by infer_batch are still alive (they are views into
        library-owned pinned memory), destruction is deferred until the last of them is released."""
        if getattr(self, "_ctx", None) is None or not self._ctx.value:
            return
        if getattr(self, "_outstanding", 0) > 0:
            self._closing = True
            return
        self._lib.kkx_destroy(self._ctx)
        self._ctx = C.c_void_p()

    @staticmethod
    def _release_buffer(session: "B200Koko", addr: int) -> None:
        try:
            if session._ctx.value:
                session._lib.kkx_release(session._ctx, C.cast(C.c_void_p(addr), C.POINTER(C.c_float)))
            with session._count_lock:
                session._outstanding -= 1
            if session._closing and session._outstanding <= 0:
                session._closing = False
                session.close()
        except Exception:
            pass

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc != 0:
            raise KkxError(rc, (self._lib.kkx_last_error(self._ctx) or b"").decode())

    def _require(self):
        if not self._ctx.value:
            raise KkxError(-5, "Session is not initialized.")  # ort_koko.rs:88-90

    @staticmethod
    def _pack(tokens, styles, speeds):
        """A ragged batch as the C ABI takes it: (B, flat int64 tokens, int32 offsets [B + 1], styles [B, 256] -- None
        when ``styles`` is None -- and f32 speeds [B])."""
        B = len(tokens)
        if B == 0:
            raise KkxError(-1, "empty batch")
        offs = np.zeros(B + 1, dtype=np.int32)
        offs[1:] = np.cumsum([len(t) for t in tokens])
        flat = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.int64).reshape(-1) for t in tokens]))
        st = None
        if styles is not None:
            st = np.ascontiguousarray(np.asarray(styles, dtype=np.float32).reshape(-1))
            if st.size != B * 256:
                raise KkxError(-1, f"style must have 256 values, got {st.size / B:g}")
            st = st.reshape(B, 256)
        sp = np.ascontiguousarray(np.asarray(speeds, dtype=np.float32).reshape(B))
        return B, flat, offs, st, sp

    def _adopt(self, ptr, offsets):
        """Zero-copy: item b of a library-owned result buffer as the view [offsets[b], offsets[b + 1]) (the reference
        copies its output twice, ort_koko.rs:85 + koko.rs:1179).  The buffer goes back to the library's pool
        (kkx_release) when the last view is garbage-collected; the views keep this session alive until then."""
        base = np.ctypeslib.as_array(ptr, shape=(max(int(offsets[-1]), 1),))
        with self._count_lock:
            self._outstanding += 1
        weakref.finalize(base, B200Koko._release_buffer, self, C.cast(ptr, C.c_void_p).value)
        return [base[int(offsets[b]):int(offsets[b + 1])] for b in range(len(offsets) - 1)]

    # -- the reference entry point --------------------------------------------------------
    def infer(self, tokens: Sequence[Sequence[int]], styles: Sequence[Sequence[float]],
              speed: float) -> np.ndarray:
        """ort_koko.rs:37-91.  tokens [B][N] (rectangular, incl. the 0 pads), styles [B][256],
        one speed.  Returns the waveform(s) as one flat f32 array -- the caller flattens the
        reference's output the same way (koko.rs:1179)."""
        if len(tokens) == 1:      # the only shape the reference sends (koko.rs:1175): the coalescable entry point
            return self.infer_one(tokens[0], np.asarray(styles, dtype=np.float32).reshape(-1), speed)
        outs = self.infer_batch([list(t) for t in tokens], styles, [speed] * len(tokens))
        return np.concatenate(outs)

    def infer_one(self, tokens: Sequence[int], style, speed: float = 1.0, return_durations: bool = False):
        """One utterance through ``kkx_infer`` -- the call a server thread makes per request.  Safe to call from
        many threads at once; with ``set_option("coalesce", K)`` the concurrent calls are merged into ragged
        batches inside the library (the reference serialises them on its session mutex, ort_koko.rs:77)."""
        self._require()
        tk = np.ascontiguousarray(np.asarray(tokens, dtype=np.int64).reshape(-1))
        st = np.ascontiguousarray(np.asarray(style, dtype=np.float32).reshape(-1))
        if st.size != 256:
            raise KkxError(-1, f"style must have 256 values, got {st.size}")
        audio = C.POINTER(C.c_float)()
        ns = C.c_int64(0)
        dur = np.zeros(max(tk.size, 1), dtype=np.int32)
        rc = self._lib.kkx_infer(self._ctx, tk.ctypes.data_as(C.POINTER(C.c_int64)), int(tk.size), _fp(st),
                                 C.c_float(speed), C.byref(audio), C.byref(ns),
                                 dur.ctypes.data_as(C.POINTER(C.c_int32)))
        self._check(rc)
        out = self._adopt(audio, (0, ns.value))[0]
        return (out, dur[:tk.size]) if return_durations else out

    # -- asynchronous form (kkx_submit / kkx_poll / kkx_wait): sentence k+1 synthesises while k is being sent
    def submit(self, tokens: Sequence[int], style, speed: float = 1.0) -> int:
        """Queue one utterance and return a ticket at once; the inputs are copied by the library."""
        self._require()
        tk = np.ascontiguousarray(np.asarray(tokens, dtype=np.int64).reshape(-1))
        st = np.ascontiguousarray(np.asarray(style, dtype=np.float32).reshape(-1))
        if st.size != 256:
            raise KkxError(-1, f"style must have 256 values, got {st.size}")
        t = C.c_int64(0)
        self._check(self._lib.kkx_submit(self._ctx, tk.ctypes.data_as(C.POINTER(C.c_int64)), int(tk.size), _fp(st),
                                         C.c_float(speed), C.byref(t)))
        with self._count_lock:
            self._tickets = getattr(self, "_tickets", {})
            self._tickets[int(t.value)] = int(tk.size)
        return int(t.value)

    def poll(self, ticket: int) -> bool:
        self._require()
        rc = self._lib.kkx_poll(self._ctx, int(ticket))
        if rc < 0:
            self._check(rc)
        return rc == 1

    def wait(self, ticket: int, return_durations: bool = False):
        """Block until the ticket's request has finished; returns what ``infer_one`` returns."""
        self._require()
        with self._count_lock:
            n = getattr(self, "_tickets", {}).pop(int(ticket), None)
        if n is None:
            raise KkxError(-1, "unknown ticket")
        audio = C.POINTER(C.c_float)()
        ns = C.c_int64(0)
        dur = np.zeros(max(n, 1), dtype=np.int32)
        self._check(self._lib.kkx_wait(self._ctx, int(ticket), C.byref(audio), C.byref(ns),
                                       dur.ctypes.data_as(C.POINTER(C.c_int32))))
        out = self._adopt(audio, (0, ns.value))[0]
        return (out, dur[:n]) if return_durations else out

    def infer_batch(self, tokens: Sequence[Sequence[int]], styles, speeds: Sequence[float],
                    return_durations: bool = False):
        """Ragged batch of independent utterances (kkx_infer_batch).  Returns a list of 1-D f32
        arrays (and the per-item integer frame durations if asked)."""
        self._require()
        B, flat, offs, st, sp = self._pack(tokens, styles, speeds)
        audio = C.POINTER(C.c_float)()
        soff = np.zeros(B + 1, dtype=np.int64)
        dur = np.zeros(int(offs[-1]), dtype=np.int32)
        rc = self._lib.kkx_infer_batch(
            self._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)),
            offs.ctypes.data_as(C.POINTER(C.c_int32)), _fp(st), _fp(sp), C.byref(audio),
            soff.ctypes.data_as(C.POINTER(C.c_int64)), dur.ctypes.data_as(C.POINTER(C.c_int32)))
        self._check(rc)
        outs = self._adopt(audio, soff)
        if return_durations:
            return outs, [dur[int(offs[b]):int(offs[b + 1])].copy() for b in range(B)]
        return outs

    # -- "next" rows (SURVEY 8f): voice table + mix_styles on the device, 16-bit PCM output ------------
    def load_voices(self, voices) -> None:
        """TTSKoko::load_voices (koko.rs:1308-1334): ``voices`` maps name -> array [511,1,256] (or [511,256]);
        the table is uploaded once and addressed by name afterwards."""
        self._require()
        names = sorted(voices)
        table = np.zeros((len(names), 511, 256), dtype=np.float32)
        for i, n in enumerate(names):
            v = np.asarray(voices[n], dtype=np.float32).reshape(-1, 256)
            table[i, :min(511, v.shape[0])] = v[:511]      # koko.rs:1315-1321 copies into a fixed 511-row tensor
        self._check(self._lib.kkx_load_voices(self._ctx, _fp(table), len(names)))
        self._voice_ids = {n: i for i, n in enumerate(names)}
        self._voice_table = table

    def _parse_style(self, style_name: str):
        ids = getattr(self, "_voice_ids", None)
        if ids is None:
            raise KkxError(-5, "no voices loaded")
        return parse_style_name(style_name, ids)

    def mix_styles(self, style_name: str, tokens_len: int) -> np.ndarray:
        """Host mirror of TTSKoko::mix_styles (same f32 arithmetic and order) -> [1,256]; the device path of
        ``infer_batch_voices`` must agree with it bit for bit."""
        vs, ps = self._parse_style(style_name)
        if "+" not in style_name:
            return self._voice_table[vs[0], tokens_len][None, :].copy()
        out = np.zeros(256, dtype=np.float32)
        for v, p in zip(vs, ps):
            out = (out + self._voice_table[v, tokens_len] * p).astype(np.float32)
        return out[None, :]

    def infer_batch_voices(self, tokens: Sequence[Sequence[int]], style_names: Sequence[str],
                           speeds: Sequence[float], return_durations: bool = False):
        """koko.rs:1161-1180 for a ragged batch: item b uses voice / mix ``style_names[b]`` at table row
        ``len(tokens[b]) - 2`` (the un-padded token count); styles are mixed on the device."""
        self._require()
        B, flat, offs, _, sp = self._pack(tokens, None, speeds)
        moff = np.zeros(B + 1, dtype=np.int32)
        vids, pors = [], []
        for b, name in enumerate(style_names):
            v, p = self._parse_style(name)
            vids += v
            pors += p
            moff[b + 1] = len(vids)
        vids = np.asarray(vids, dtype=np.int32)
        pors = np.asarray(pors, dtype=np.float32)
        rows = np.asarray([len(t) - 2 for t in tokens], dtype=np.int32)
        audio = C.POINTER(C.c_float)()
        soff = np.zeros(B + 1, dtype=np.int64)
        dur = np.zeros(int(offs[-1]), dtype=np.int32)
        ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
        self._check(self._lib.kkx_infer_batch_voices(
            self._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)), ip(offs), ip(moff), ip(vids), _fp(pors),
            ip(rows), _fp(sp), C.byref(audio), soff.ctypes.data_as(C.POINTER(C.c_int64)), ip(dur)))
        outs = self._adopt(audio, soff)
        if return_durations:
            return outs, [dur[int(offs[b]):int(offs[b + 1])].copy() for b in range(B)]
        return outs

    def infer_batch_pcm16(self, tokens: Sequence[Sequence[int]], styles, speeds: Sequence[float]):
        """Like infer_batch, but returns int16 PCM (trunc(clamp(s,-1,1)*32767), kokorox-websocket lib.rs:699-703),
        converted inside the iSTFT kernel; the device->host copy is half the size."""
        self._require()
        B, flat, offs, st, sp = self._pack(tokens, styles, speeds)
        pcm = C.POINTER(C.c_int16)()
        soff = np.zeros(B + 1, dtype=np.int64)
        self._check(self._lib.kkx_infer_batch_pcm16(
            self._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)), offs.ctypes.data_as(C.POINTER(C.c_int32)),
            _fp(st), _fp(sp), C.byref(pcm), soff.ctypes.data_as(C.POINTER(C.c_int64)), None))
        return self._adopt(pcm, soff)

    def infer_batch_g711(self, tokens: Sequence[Sequence[int]], styles, speeds: Sequence[float], law: str = "ulaw",
                         return_durations: bool = False):
        """Like infer_batch_pcm16, but every sample comes back as one G.711 byte (``law`` "ulaw" = PCMU or "alaw" =
        PCMA) of that 16-bit value, at the session's ``out_rate`` (set it to 8000 for telephony).  Returns a list of
        uint8 arrays, views into a library-owned buffer released like the pcm16 ones."""
        self._require()
        laws = {"ulaw": 0, "alaw": 1}
        if law not in laws:
            raise KkxError(-1, f"law must be 'ulaw' or 'alaw', got {law!r}")
        B, flat, offs, st, sp = self._pack(tokens, styles, speeds)
        codes = C.POINTER(C.c_uint8)()
        soff = np.zeros(B + 1, dtype=np.int64)
        dur = np.zeros(int(offs[-1]), dtype=np.int32)
        self._check(self._lib.kkx_infer_batch_g711(
            self._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)), offs.ctypes.data_as(C.POINTER(C.c_int32)),
            _fp(st), _fp(sp), laws[law], C.byref(codes), soff.ctypes.data_as(C.POINTER(C.c_int64)),
            dur.ctypes.data_as(C.POINTER(C.c_int32))))
        outs = self._adopt(codes, soff)
        if return_durations:
            return outs, [dur[int(offs[b]):int(offs[b + 1])].copy() for b in range(B)]
        return outs

    def infer_batch_flac(self, tokens: Sequence[Sequence[int]], styles, speeds: Sequence[float],
                         return_durations: bool = False):
        """Like infer_batch_pcm16, but item b comes back as one complete FLAC file (``bytes``, Content-Type
        audio/flac) at the session's ``out_rate``, encoded on the device; decoding it gives exactly the int16 samples
        infer_batch_pcm16 returns.  The files are copied out of the library's buffer, which is released before this
        returns."""
        self._require()
        B, flat, offs, st, sp = self._pack(tokens, styles, speeds)
        buf = C.POINTER(C.c_uint8)()
        boff = np.zeros(B + 1, dtype=np.int64)
        dur = np.zeros(int(offs[-1]), dtype=np.int32)
        self._check(self._lib.kkx_infer_batch_flac(
            self._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)), offs.ctypes.data_as(C.POINTER(C.c_int32)),
            _fp(st), _fp(sp), C.byref(buf), boff.ctypes.data_as(C.POINTER(C.c_int64)), None,
            dur.ctypes.data_as(C.POINTER(C.c_int32))))
        try:
            outs = [C.string_at(C.addressof(buf.contents) + int(boff[b]), int(boff[b + 1] - boff[b])) for b in range(B)]
        finally:
            self._lib.kkx_release_flac(self._ctx, buf)
        if return_durations:
            return outs, [dur[int(offs[b]):int(offs[b + 1])].copy() for b in range(B)]
        return outs

    # encoding name -> (KKX_ENC_* code, element type of the returned arrays; None = one ``bytes`` per program)
    _ENCODINGS = {"f32": (0, C.c_float), "pcm16": (1, C.c_int16), "ulaw": (2, C.c_uint8), "alaw": (3, C.c_uint8),
                  "flac": (4, None)}

    def infer_programs(self, tokens: Sequence[Sequence[int]], styles, speeds: Sequence[float],
                       program_offsets: Sequence[int], encoding: str = "f32", return_durations: bool = False):
        """One output per program (kkx_infer_programs): program k is items [program_offsets[k],
        program_offsets[k + 1]), synthesised as ONE utterance whose 24 kHz waveform is the concatenation of its items'
        -- the chunks of one long request, as koko.rs splits and joins them.  Loudness, resampling and FLAC apply to
        the program as a whole.  ``encoding``: "f32" / "pcm16" / "ulaw" / "alaw" give one float32 / int16 / uint8
        array per program (views into a library-owned buffer, released like infer_batch's), "flac" one ``bytes`` file
        per program."""
        self._require()
        if encoding not in self._ENCODINGS:
            raise KkxError(-1, f"encoding must be one of {sorted(self._ENCODINGS)}, got {encoding!r}")
        code, ctype = self._ENCODINGS[encoding]
        B, flat, offs, st, sp = self._pack(tokens, styles, speeds)
        prog = np.ascontiguousarray(np.asarray(program_offsets, dtype=np.int32).reshape(-1))
        P = max(prog.size - 1, 0)
        buf = C.c_void_p()
        boff = np.zeros(P + 1, dtype=np.int64)
        dur = np.zeros(int(offs[-1]), dtype=np.int32)
        self._check(self._lib.kkx_infer_programs(
            self._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)), offs.ctypes.data_as(C.POINTER(C.c_int32)),
            _fp(st), _fp(sp), P, prog.ctypes.data_as(C.POINTER(C.c_int32)), code, C.byref(buf),
            boff.ctypes.data_as(C.POINTER(C.c_int64)), None, dur.ctypes.data_as(C.POINTER(C.c_int32))))
        if ctype is None:
            try:
                outs = [C.string_at(buf.value + int(boff[k]), int(boff[k + 1] - boff[k])) for k in range(P)]
            finally:
                self._lib.kkx_release_programs(self._ctx, buf)
        else:
            outs = self._adopt(C.cast(buf, C.POINTER(ctype)), boff // C.sizeof(ctype))
        if return_durations:
            return outs, [dur[int(offs[b]):int(offs[b + 1])].copy() for b in range(B)]
        return outs

    def last_loudness(self):
        """What loudness normalisation (option ``loudness_target``) measured and applied in this session's last
        synchronous call: ``(lufs, true_peak_dbtp, gain)``, three float32 arrays in item order -- program order after
        ``infer_programs`` -- (``lufs`` is NaN where
        the loudness is undefined: items under 400 ms, silence).  Raises KkxError when that call ran with the option
        off.  Coalesced and ``submit`` batches are not reported."""
        self._require()
        n = max(int(self._lib.kkx_get_stat(self._ctx, b"loudness_items")), 0)
        lufs, tp, gain = (np.zeros(max(n, 1), np.float32) for _ in range(3))
        self._check(self._lib.kkx_last_loudness(self._ctx, n, _fp(lufs), _fp(tp), _fp(gain)))
        return lufs[:n], tp[:n], gain[:n]

    # -- device-resident path (bench `value`) ---------------------------------------------
    def stage(self, tokens, styles, speeds) -> None:
        self._require()
        B, flat, offs, st, sp = self._pack(tokens, styles, speeds)
        self._check(self._lib.kkx_stage_batch(self._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)),
                                              offs.ctypes.data_as(C.POINTER(C.c_int32)), _fp(st), _fp(sp)))
        self._staged = (B, int(offs[-1]))

    def run_staged(self):
        """Returns (total_samples, kernel_launches)."""
        self._require()
        n, l = C.c_int64(), C.c_int64()
        self._check(self._lib.kkx_run_staged(self._ctx, C.byref(n), C.byref(l)))
        return int(n.value), int(l.value)

    def fetch_staged(self, total_samples: int):
        B, ntok = self._staged
        out = np.empty(max(total_samples, 1), dtype=np.float32)
        soff = np.zeros(B + 1, dtype=np.int64)
        dur = np.zeros(ntok, dtype=np.int32)
        self._check(self._lib.kkx_fetch_staged(self._ctx, _fp(out), total_samples,
                                               soff.ctypes.data_as(C.POINTER(C.c_int64)),
                                               dur.ctypes.data_as(C.POINTER(C.c_int32))))
        return out[:total_samples], soff, dur

    # -- options / test hooks -------------------------------------------------------------
    def set_option(self, key: str, value: int) -> None:
        self._require()
        self._check(self._lib.kkx_set_option(self._ctx, key.encode(), int(value)))

    def get_stat(self, key: str) -> int:
        self._require()
        return int(self._lib.kkx_get_stat(self._ctx, key.encode()))

    def set_noise(self, noise: Optional[np.ndarray]) -> None:
        self._require()
        if noise is None:
            self._check(self._lib.kkx_set_noise(self._ctx, None, 0))
        else:
            a = np.ascontiguousarray(noise, dtype=np.float32).reshape(-1)
            self._check(self._lib.kkx_set_noise(self._ctx, _fp(a), a.size))

    def set_inject(self, name: str, data: Optional[np.ndarray], item: int = 0) -> None:
        """Teacher-force ``pred_dur`` / ``F0`` / ``N`` of batch item ``item`` (test hook, kkx_test.h)."""
        self._require()
        if data is None:
            self._check(self._lib.kkx_set_inject_item(self._ctx, int(item), name.encode(), None, 0))
            return
        a = np.ascontiguousarray(data, dtype=np.int32 if name == "pred_dur" else np.float32).reshape(-1)
        self._check(self._lib.kkx_set_inject_item(self._ctx, int(item), name.encode(), a.ctypes.data_as(C.c_void_p),
                                                  a.size))

    def profile_enable(self, on: bool = True) -> None:
        self._require()
        self._check(self._lib.kkx_profile_enable(self._ctx, 1 if on else 0))

    def profile(self) -> dict:
        """Per-kernel device time of the last run: {"conv_flops", "gpu_us", "kernels": {name: [n, us]}}."""
        import json
        self._require()
        n = self._lib.kkx_profile_json(self._ctx, None, 0)
        buf = C.create_string_buffer(int(n) + 1)
        self._lib.kkx_profile_json(self._ctx, buf, n + 1)
        return json.loads(buf.value.decode())

    def debug_enable(self, on: bool = True, item: Optional[int] = None) -> None:
        """Keep stage tensors of every item (``item`` None) or of one batch item for ``debug_stage``."""
        self._require()
        if item is None:
            self._check(self._lib.kkx_debug_enable(self._ctx, 1 if on else 0))
        else:
            self._check(self._lib.kkx_debug_select(self._ctx, 1 if on else 0, int(item)))

    def debug_stage(self, name: str, item: int = 0) -> Optional[np.ndarray]:
        self._require()
        rows, cols = C.c_int64(), C.c_int64()
        n = self._lib.kkx_debug_stage(self._ctx, name.encode(), item, None, 0, C.byref(rows), C.byref(cols))
        if n < 0:
            return None
        out = np.empty(max(int(n), 1), dtype=np.float32)
        self._lib.kkx_debug_stage(self._ctx, name.encode(), item, _fp(out), n, None, None)
        out = out[:n].reshape(int(rows.value), int(cols.value))
        return out[:, 0] if cols.value == 1 else out
