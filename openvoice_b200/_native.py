"""ctypes binding of libovc_b200.so (C ABI: include/ovc.h).

PyTorch is used for device memory and streams only; every tensor crosses the boundary as a raw
device pointer.  If the library is missing or no sm_100 GPU is present this module raises --
there is no fallback path of any kind.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Iterable, Optional, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libovc_b200.so")

ABI_VERSION = 4
EXPORTS = (
    "ovc_abi_version", "ovc_last_error", "ovc_create", "ovc_destroy", "ovc_load_tensor",
    "ovc_finalize_weights", "ovc_workspace_floats", "ovc_voice_conversion", "ovc_last_launch_count",
    "ovc_profile_enable", "ovc_profile_read", "ovc_profile_detail", "ovc_debug_enable", "ovc_debug_fetch",
    "ovc_spectrogram", "ovc_convert_waveform", "ovc_set_precision", "ovc_reference_encoder",
    "ovc_tts_info", "ovc_tts_encode", "ovc_tts_decode", "ovc_set_option", "ovc_graph_replays",
)


class OvcHParams(C.Structure):
    """struct ovc_hparams of include/ovc.h."""
    _fields_ = [
        ("spec_channels", C.c_int32), ("inter_channels", C.c_int32), ("hidden_channels", C.c_int32),
        ("gin_channels", C.c_int32), ("resblock", C.c_int32), ("n_resblock_kernels", C.c_int32),
        ("resblock_kernel_sizes", C.c_int32 * 4), ("resblock_dilations", (C.c_int32 * 3) * 4),
        ("n_upsamples", C.c_int32), ("upsample_rates", C.c_int32 * 4),
        ("upsample_kernel_sizes", C.c_int32 * 4), ("upsample_initial_channel", C.c_int32),
        ("zero_g", C.c_int32), ("hop_length", C.c_int32),
    ]


PRECISIONS = {"fp32": 0, "f16x3": 1, "f16": 2, "f16s": 3}


class OvcError(RuntimeError):
    pass


_lib = None


def load_library(path: Optional[str] = None):
    """dlopen the CUDA library (once).  Raises OvcError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or os.environ.get("OVC_B200_LIB", LIB_PATH)
    if not os.path.exists(path):
        raise OvcError(
            f"{path} not found: build the sm_100a extension first "
            "(python -c 'import __graft_entry__ as g; g.build()' or make -C openvoice_b200/csrc). "
            "openvoice_b200 has no CPU / PyTorch fallback.")
    lib = C.CDLL(path)
    lib.ovc_abi_version.restype = C.c_int
    lib.ovc_last_error.restype = C.c_char_p
    lib.ovc_create.argtypes = [C.POINTER(OvcHParams), C.c_int, C.POINTER(C.c_void_p)]
    lib.ovc_destroy.argtypes = [C.c_void_p]
    lib.ovc_destroy.restype = None
    lib.ovc_load_tensor.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int]
    lib.ovc_finalize_weights.argtypes = [C.c_void_p]
    lib.ovc_workspace_floats.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.ovc_workspace_floats.restype = C.c_size_t
    lib.ovc_voice_conversion.argtypes = [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_float,
        C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ovc_last_launch_count.argtypes = [C.c_void_p]
    lib.ovc_graph_replays.argtypes = [C.c_void_p]
    lib.ovc_graph_replays.restype = C.c_int
    lib.ovc_set_precision.argtypes = [C.c_void_p, C.c_int]
    lib.ovc_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.ovc_reference_encoder.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.ovc_profile_enable.argtypes = [C.c_void_p, C.c_int]
    lib.ovc_profile_read.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64),
                                     C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.ovc_profile_detail.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                       C.POINTER(C.c_double), C.POINTER(C.c_int)]
    lib.ovc_debug_enable.argtypes = [C.c_void_p, C.c_int]
    lib.ovc_debug_fetch.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int64)]
    lib.ovc_spectrogram.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    lib.ovc_convert_waveform.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_uint64, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ovc_tts_info.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
    lib.ovc_tts_encode.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_float,
                                   C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ovc_tts_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    if lib.ovc_abi_version() != ABI_VERSION:
        raise OvcError(f"ABI mismatch: library {lib.ovc_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


def _check(lib, rc: int, what: str):
    if rc < 0:
        msg = lib.ovc_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise OvcError(f"{what}: {msg} (status {rc})")


def hparams_struct(hps) -> OvcHParams:
    """Build struct ovc_hparams from the reference-style config tree (utils.HParams or dict)."""
    def get(obj, k, default=None):
        if isinstance(obj, dict):
            return obj.get(k, default)
        return getattr(obj, k, default)

    model, data = get(hps, "model"), get(hps, "data")
    s = OvcHParams()
    s.spec_channels = int(get(data, "filter_length")) // 2 + 1
    s.inter_channels = int(get(model, "inter_channels"))
    s.hidden_channels = int(get(model, "hidden_channels"))
    s.gin_channels = int(get(model, "gin_channels", 256))
    rb = str(get(model, "resblock"))
    s.resblock = 1 if rb == "1" else 2
    ks = list(get(model, "resblock_kernel_sizes"))
    ds = [list(d) for d in get(model, "resblock_dilation_sizes")]
    if len(ks) > 4 or any(len(d) != 3 for d in ds) or len(ds) != len(ks):
        raise ValueError("unsupported resblock configuration")
    s.n_resblock_kernels = len(ks)
    for i, k in enumerate(ks):
        s.resblock_kernel_sizes[i] = int(k)
        for j in range(3):
            s.resblock_dilations[i][j] = int(ds[i][j])
    ur, uk = list(get(model, "upsample_rates")), list(get(model, "upsample_kernel_sizes"))
    if len(ur) > 4 or len(ur) != len(uk):
        raise ValueError("unsupported upsample configuration")
    s.n_upsamples = len(ur)
    for i in range(len(ur)):
        s.upsample_rates[i] = int(ur[i])
        s.upsample_kernel_sizes[i] = int(uk[i])
    s.upsample_initial_channel = int(get(model, "upsample_initial_channel"))
    s.zero_g = 1 if get(model, "zero_g", False) else 0
    s.hop_length = int(get(data, "hop_length"))
    return s


class NativeConverter:
    """Owns one ovc_ctx (one per device)."""

    def __init__(self, hps, device_index: int):
        self.lib = load_library()
        self.hp = hparams_struct(hps)
        h = C.c_void_p()
        _check(self.lib, self.lib.ovc_create(C.byref(self.hp), int(device_index), C.byref(h)), "ovc_create")
        self.handle = h
        self.device_index = int(device_index)
        self.finalized = False
        if os.environ.get("OVC_WIDE_VARIANT"):      # tuning experiments: kernel of the 128-column tensor-core layers
            self.set_option("wide_variant", int(os.environ["OVC_WIDE_VARIANT"]))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.ovc_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights ---------------------------------------------------------------------------
    def load_state_dict(self, sd: Dict[str, "object"]) -> Tuple[list, list]:
        """Feed a reference-schema state dict; returns (used_keys, ignored_keys)."""
        import numpy as np
        used, ignored = [], []
        for k, v in sd.items():
            a = v.detach().cpu().float().contiguous().numpy() if hasattr(v, "detach") else np.ascontiguousarray(v, dtype=np.float32)
            if a.ndim == 0 or a.ndim > 4:
                ignored.append(k)
                continue
            shape = (C.c_int64 * a.ndim)(*a.shape)
            rc = self.lib.ovc_load_tensor(self.handle, k.encode(), a.ctypes.data_as(C.c_void_p), shape, a.ndim)
            _check(self.lib, rc, f"ovc_load_tensor({k})")
            (ignored if rc == 1 else used).append(k)
        self.finalized = False
        return used, ignored

    def finalize(self):
        _check(self.lib, self.lib.ovc_finalize_weights(self.handle), "ovc_finalize_weights")
        self.finalized = True

    def set_precision(self, mode: str):
        """'fp32' (CUDA-core FFMA2), 'f16x3' (split-precision fp16 tensor-core convs, fp32-grade), 'f16' (single pass)
        or 'f16s' (as 'f16x3' up to z_hat, then an fp16-storage generator: fp16 activations, one fp16 pass per conv)."""
        m = PRECISIONS[mode]
        _check(self.lib, self.lib.ovc_set_precision(self.handle, m), "ovc_set_precision")
        self.precision = mode

    def set_option(self, key: str, value: int):
        """Tuning switches of include/ovc.h: 'wide_variant' (0/2/3), 'tts_simple', 'graph', 'pdl' (0/1/2), 'branches', 'pair' (0/1)."""
        k = {"wide_variant": 1, "tts_simple": 2, "graph": 3, "pdl": 5, "branches": 7, "pair": 8}[key]
        _check(self.lib, self.lib.ovc_set_option(self.handle, k, int(value)), "ovc_set_option")

    # ---- hot path --------------------------------------------------------------------------
    def voice_conversion(self, spec, lengths, g_src, g_tgt, noise=None, tau: float = 0.3, seed: int = 0,
                         ragged: bool = False, latents: bool = True, stream=None):
        """spec [B,S,T] f32 cuda, lengths [B] i64 cuda, g_* [B,gin(,1)] f32 cuda.
        Returns (o_hat [B,1,hop*T], (z, z_p, z_hat) or None).  Asynchronous on `stream`."""
        import torch
        assert spec.is_cuda and spec.dtype == torch.float32 and spec.is_contiguous()
        assert lengths.is_cuda and lengths.dtype == torch.int64 and lengths.is_contiguous()
        B, S, T = spec.shape
        gs = g_src.reshape(B, -1).contiguous().float()
        gt = g_tgt.reshape(B, -1).contiguous().float()
        if noise is not None:
            noise = noise.contiguous().float()
            assert tuple(noise.shape) == (B, self.hp.inter_channels, T)
        hop = self.hp.hop_length
        o = torch.empty(B, 1, hop * T, device=spec.device, dtype=torch.float32)
        lat = None
        if latents:
            lat = tuple(torch.empty(B, self.hp.inter_channels, T, device=spec.device, dtype=torch.float32)
                        for _ in range(3))
        st = stream if stream is not None else torch.cuda.current_stream(spec.device)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
        rc = self.lib.ovc_voice_conversion(
            self.handle, p(spec), p(lengths), p(gs), p(gt), p(noise), C.c_uint64(seed & (2 ** 64 - 1)),
            C.c_float(tau), B, T, 1 if ragged else 0, p(o),
            p(lat[0]) if lat else None, p(lat[1]) if lat else None, p(lat[2]) if lat else None,
            C.c_void_p(st.cuda_stream))
        _check(self.lib, rc, "ovc_voice_conversion")
        return o, lat

    def spectrogram(self, wav, wav_lengths, stream=None):
        """wav [B, Lmax] f32 cuda (zero padded), wav_lengths [B] i64 cuda (samples) ->
        (spec [B, S, Lmax // hop], frames [B] i64): spectrogram_torch on device, per-item reflect padding."""
        import torch
        assert wav.is_cuda and wav.dtype == torch.float32 and wav.is_contiguous() and wav.dim() == 2
        assert wav_lengths.is_cuda and wav_lengths.dtype == torch.int64
        B, L = wav.shape
        T = L // self.hp.hop_length
        spec = torch.empty(B, self.hp.spec_channels, T, device=wav.device, dtype=torch.float32)
        frames = torch.empty(B, device=wav.device, dtype=torch.int64)
        st = stream if stream is not None else torch.cuda.current_stream(wav.device)
        rc = self.lib.ovc_spectrogram(self.handle, C.c_void_p(wav.data_ptr()), C.c_void_p(wav_lengths.data_ptr()), B, L, T,
                                      C.c_void_p(spec.data_ptr()), C.c_void_p(frames.data_ptr()), C.c_void_p(st.cuda_stream))
        _check(self.lib, rc, "ovc_spectrogram")
        return spec, frames

    def convert_waveform(self, wav, wav_lengths, g_src, g_tgt, noise=None, tau: float = 0.3, seed: int = 0, stream=None,
                         out=None, frames_out=None):
        """The device work of ToneColorConverter.convert for a batch: wav [B, Lmax] f32 cuda ->
        (o_hat [B, hop * (Lmax // hop)], frames [B]).  Asynchronous on `stream`.  ``out`` / ``frames_out`` let the
        caller supply the result buffers: with every buffer at a stable address, a repeated call is replayed from a
        CUDA graph (include/ovc.h: OVC_OPT_GRAPH)."""
        import torch
        assert wav.is_cuda and wav.dtype == torch.float32 and wav.is_contiguous() and wav.dim() == 2
        assert wav_lengths.is_cuda and wav_lengths.dtype == torch.int64
        B, L = wav.shape
        T = L // self.hp.hop_length
        gs = g_src.reshape(B, -1).contiguous().float()
        gt = g_tgt.reshape(B, -1).contiguous().float()
        if noise is not None:
            noise = noise.contiguous().float()
            assert tuple(noise.shape) == (B, self.hp.inter_channels, T)
        if out is not None:
            assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.numel() == B * self.hp.hop_length * T
            o = out.view(B, self.hp.hop_length * T)
        else:
            o = torch.empty(B, self.hp.hop_length * T, device=wav.device, dtype=torch.float32)
        if frames_out is not None:
            assert frames_out.is_cuda and frames_out.dtype == torch.int64 and frames_out.numel() == B
            frames = frames_out
        else:
            frames = torch.empty(B, device=wav.device, dtype=torch.int64)
        st = stream if stream is not None else torch.cuda.current_stream(wav.device)
        rc = self.lib.ovc_convert_waveform(
            self.handle, C.c_void_p(wav.data_ptr()), C.c_void_p(wav_lengths.data_ptr()), B, L, C.c_void_p(gs.data_ptr()),
            C.c_void_p(gt.data_ptr()), C.c_void_p(noise.data_ptr()) if noise is not None else None,
            C.c_uint64(seed & (2 ** 64 - 1)), C.c_float(tau), C.c_void_p(o.data_ptr()), C.c_void_p(frames.data_ptr()),
            C.c_void_p(st.cuda_stream))
        _check(self.lib, rc, "ovc_convert_waveform")
        return o, frames

    def reference_encoder(self, spec, stream=None):
        """spec [N, S, T] f32 cuda (ovc_spectrogram layout) -> tone-colour embedding [N, gin]
        (ReferenceEncoder.forward, openvoice/models.py:339-359)."""
        import torch
        assert spec.is_cuda and spec.dtype == torch.float32 and spec.is_contiguous() and spec.dim() == 3
        N, S, T = spec.shape
        if S != self.hp.spec_channels:
            raise ValueError(f"reference_encoder: spec has {S} channels, the model has spec_channels {self.hp.spec_channels}")
        out = torch.empty(N, self.hp.gin_channels, device=spec.device, dtype=torch.float32)
        st = stream if stream is not None else torch.cuda.current_stream(spec.device)
        rc = self.lib.ovc_reference_encoder(self.handle, C.c_void_p(spec.data_ptr()), N, T, C.c_void_p(out.data_ptr()),
                                            C.c_void_p(st.cuda_stream))
        _check(self.lib, rc, "ovc_reference_encoder")
        return out

    # ---- V1 TTS front half (SynthesizerTrn.infer, openvoice/models.py:467-490) ----------------
    def tts_info(self) -> dict:
        out = (C.c_int32 * 8)()
        _check(self.lib, self.lib.ovc_tts_info(self.handle, out), "ovc_tts_info")
        keys = ("has_tts", "n_vocab", "n_speakers", "n_heads", "n_layers", "window", "filter_channels", "dp_filter")
        return dict(zip(keys, (int(v) for v in out)))

    def tts_encode(self, tokens, x_lengths, sid, noise_w=None, seed: int = 0, noise_scale_w: float = 1.0,
                   length_scale: float = 1.0, sdp_ratio: float = 0.2, stream=None):
        """tokens [B,T] i64 cuda, x_lengths [B] i64 cuda, sid [B] i64 cuda, noise_w [B,2,T] or None (Philox).
        Returns (y_lengths [B] i64, w_ceil [B,T], logw [B,T]), all on the device; asynchronous on `stream`."""
        import torch
        for t in (tokens, x_lengths, sid):
            assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous()
        B, T = tokens.shape
        if noise_w is not None:
            noise_w = noise_w.contiguous().float()
            assert tuple(noise_w.shape) == (B, 2, T)
        y_lengths = torch.empty(B, device=tokens.device, dtype=torch.int64)
        w_ceil = torch.empty(B, T, device=tokens.device, dtype=torch.float32)
        logw = torch.empty(B, T, device=tokens.device, dtype=torch.float32)
        st = stream if stream is not None else torch.cuda.current_stream(tokens.device)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
        rc = self.lib.ovc_tts_encode(self.handle, p(tokens), p(x_lengths), p(sid), p(noise_w), C.c_uint64(seed & (2 ** 64 - 1)),
                                     C.c_float(noise_scale_w), C.c_float(length_scale), C.c_float(sdp_ratio), B, T,
                                     p(y_lengths), p(w_ceil), p(logw), C.c_void_p(st.cuda_stream))
        _check(self.lib, rc, "ovc_tts_encode")
        return y_lengths, w_ceil, logw

    def tts_decode(self, B: int, y_max: int, device, noise=None, seed: int = 0, noise_scale: float = 1.0,
                   ragged: bool = False, latents: bool = False, max_len: Optional[int] = None, stream=None):
        """Second half of infer() for the last tts_encode.  Returns (o [B,1,hop*min(y_max, max_len)], (z, z_p) or None)."""
        import torch
        C_ = self.hp.inter_channels
        if noise is not None:
            noise = noise.contiguous().float()
            assert noise.is_cuda and tuple(noise.shape) == (B, C_, y_max)
        cut = int(max_len) if max_len is not None and 0 < int(max_len) < y_max else 0
        o = torch.empty(B, 1, self.hp.hop_length * (cut or y_max), device=device, dtype=torch.float32)
        lat = tuple(torch.empty(B, C_, y_max, device=device, dtype=torch.float32) for _ in range(2)) if latents else None
        st = stream if stream is not None else torch.cuda.current_stream(device)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
        rc = self.lib.ovc_tts_decode(self.handle, p(noise), C.c_uint64(seed & (2 ** 64 - 1)), C.c_float(noise_scale), B,
                                     int(y_max), cut, 1 if ragged else 0, p(o), p(lat[0]) if lat else None,
                                     p(lat[1]) if lat else None, C.c_void_p(st.cuda_stream))
        _check(self.lib, rc, "ovc_tts_decode")
        return o, lat

    @property
    def last_launch_count(self) -> int:
        return int(self.lib.ovc_last_launch_count(self.handle))

    @property
    def graph_replays(self) -> int:
        """calls served from a captured CUDA graph so far (include/ovc.h: ovc_graph_replays)"""
        return int(self.lib.ovc_graph_replays(self.handle))

    # ---- instrumentation -------------------------------------------------------------------
    def profile_enable(self, on: bool):
        _check(self.lib, self.lib.ovc_profile_enable(self.handle, 1 if on else 0), "ovc_profile_enable")

    def profile_read(self):
        ms, n, fl, by = C.c_double(), C.c_int64(), C.c_double(), C.c_double()
        _check(self.lib, self.lib.ovc_profile_read(self.handle, C.byref(ms), C.byref(n), C.byref(fl), C.byref(by)),
               "ovc_profile_read")
        return dict(ms=ms.value, launches=n.value, flops=fl.value, bytes=by.value)

    def profile_detail(self, max_entries: int = 4096):
        """Per-launch (name, ms, flops, bytes, family) of the conv kernels since the last reset."""
        names = C.create_string_buffer(16 * max_entries)
        ms = (C.c_double * max_entries)()
        fl = (C.c_double * max_entries)()
        by = (C.c_double * max_entries)()
        fam = (C.c_int * max_entries)()
        n = self.lib.ovc_profile_detail(self.handle, max_entries, names, ms, fl, by, fam)
        _check(self.lib, n, "ovc_profile_detail")
        raw = names.raw
        return [(raw[16 * i: 16 * i + 16].split(b"\0")[0].decode(), ms[i], fl[i], by[i], fam[i]) for i in range(n)]

    def debug_enable(self, on: bool):
        _check(self.lib, self.lib.ovc_debug_enable(self.handle, 1 if on else 0), "ovc_debug_enable")

    def debug_fetch(self, name: str):
        """Returns a numpy array [B, C, T] of the named tap of the last call."""
        import numpy as np
        shape = (C.c_int64 * 4)()
        _check(self.lib, self.lib.ovc_debug_fetch(self.handle, name.encode(), None, 0, shape), "ovc_debug_fetch")
        B, Cc, T, pitch = [int(v) for v in shape]
        buf = np.empty((B, Cc, pitch), dtype=np.float32)
        _check(self.lib, self.lib.ovc_debug_fetch(self.handle, name.encode(), buf.ctypes.data_as(C.c_void_p),
                                                  buf.size, shape), "ovc_debug_fetch")
        return buf[:, :, :T]
