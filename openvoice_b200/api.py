"""Drop-in for the tone-colour-converter half of the reference's ``openvoice/api.py``.

Same classes, method names, arguments and return types as ``OpenVoiceBaseClass`` /
``ToneColorConverter`` (openvoice/api.py:14-39, :101-201); ``self.model`` is a
``NativeSynthesizer`` whose ``voice_conversion`` (the seam at openvoice/api.py:154) runs in
libovc_b200.so.  Supersets of the reference: ``convert`` also accepts a NumPy waveform,
``convert_batch`` converts a list of utterances in one launch sequence,
``enable_watermark=False`` works (it raises TypeError in the reference, SURVEY.md section 3.2).
CUDA only: there is no CPU path.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from . import utils
from ._native import NativeConverter
from .ref_enc import ReferenceEncoder
from .schema import hot_path_keys, ref_enc_keys, tts_keys

AudioLike = Union[str, np.ndarray]


def _load_audio(src: AudioLike, sr: int) -> np.ndarray:
    """Stand-in for ``librosa.load(path, sr=sr)`` (openvoice/api.py:144): mono float32 at ``sr``.
    Uses librosa when it is installed; otherwise .npy (already at ``sr``) and PCM/float .wav via
    scipy, with polyphase resampling (not bit-identical to librosa's resampler -- third-party
    arithmetic the reference does not pin, SURVEY.md section 8c)."""
    if isinstance(src, np.ndarray):
        return np.ascontiguousarray(src, dtype=np.float32).reshape(-1)
    if src.endswith(".npy"):
        return np.ascontiguousarray(np.load(src), dtype=np.float32).reshape(-1)
    try:
        import librosa  # type: ignore
        return librosa.load(src, sr=sr)[0].astype(np.float32)
    except ImportError:
        pass
    from scipy.io import wavfile
    from scipy.signal import resample_poly
    file_sr, data = wavfile.read(src)
    if data.dtype.kind == "i":
        data = data.astype(np.float32) / float(np.iinfo(data.dtype).max + 1)
    elif data.dtype.kind == "u":
        data = (data.astype(np.float32) - 128.0) / 128.0
    data = data.astype(np.float32)
    if data.ndim == 2:
        data = data.mean(axis=1)
    if sr is not None and file_sr != sr:   # sr=None keeps the file's rate (librosa.load(sr=None))
        from math import gcd
        g = gcd(int(file_sr), int(sr))
        data = resample_poly(data, sr // g, file_sr // g).astype(np.float32)
    return np.ascontiguousarray(data)


def _write_audio(path: str, audio: np.ndarray, sr: int) -> None:
    """Stand-in for ``soundfile.write`` (openvoice/api.py:160)."""
    if path.endswith(".npy"):
        np.save(path, audio)
        return
    try:
        import soundfile  # type: ignore
        soundfile.write(path, audio, sr)
    except ImportError:
        from scipy.io import wavfile
        wavfile.write(path, sr, audio.astype(np.float32))


_POOL = None


def _pool():
    """Host-side staging threads: copying the utterances into / out of the pinned buffers is plain memcpy work (numpy
    releases the GIL for it) that sits inside every end-to-end call."""
    global _POOL
    if _POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        try:
            n = len(os.sched_getaffinity(0))
        except Exception:
            n = os.cpu_count() or 1
        _POOL = ThreadPoolExecutor(max_workers=max(1, min(8, n)), thread_name_prefix="ovc-stage")
    return _POOL


def _parallel(fn, n, min_items=4):
    if n < min_items:
        return [fn(i) for i in range(n)]
    return list(_pool().map(fn, range(n)))


def watermark_device(audio, payload_bits, model, chunk: int = 16000, stride: int = 32000):
    """On-device chunking of openvoice/api.py:162-184.  ``audio``: 1-D float32 tensor (any device), modified in place;
    ``payload_bits``: flat 0/1 array, 32 per chunk.  Chunk n = samples [n * stride, n * stride + chunk); as in the
    reference the walk stops at the first chunk that does not fit ("Audio too short").  All full chunks are gathered
    by a strided view (no copy), encoded by ONE batched ``model.encode([m, chunk], [m, 32])`` call and scattered back."""
    n_repeat = len(payload_bits) // 32
    L = int(audio.shape[0])
    m = 0
    while m < n_repeat and m * stride + chunk <= L:
        m += 1
    if m < n_repeat:
        print("Audio too short, fail to add watermark")
    if m == 0:
        return audio
    with torch.no_grad():
        view = torch.as_strided(audio, (m, chunk), (stride, 1))
        bits = torch.as_tensor(np.asarray(payload_bits[: 32 * m], dtype=np.float32).reshape(m, 32), device=audio.device)
        enc = model.encode(view.contiguous(), bits).detach().reshape(m, chunk).to(audio.dtype)
        view.copy_(enc)
    return audio


class NativeSynthesizer:
    """Stands where ``SynthesizerTrn`` stands in the reference (``converter.model``) for the
    ``n_speakers == 0`` converter (openvoice/models.py:399-465): ``voice_conversion``,
    ``ref_enc``, ``load_state_dict``, ``eval``, ``zero_g``."""

    def __init__(self, hps, device: str, precision: Optional[str] = None):
        """``precision``: arithmetic of the generator's ResBlock / upsampling convolutions --
        ``"f16x3"`` (default; split-precision fp16 on the tcgen05 tensor cores, fp32-grade),
        ``"fp32"`` (CUDA-core FFMA2 everywhere), ``"f16"`` (single-pass fp16: the 11-bit operand precision the
        reference itself gets on a GPU through cuDNN's allow_tf32 default; ~1e-2) or ``"f16s"`` (fp16 storage:
        z / z_p / z_hat exactly as ``"f16x3"``, then a generator with fp16 activations in memory and one fp16 pass
        per conv -- half its memory traffic and workspace, o_hat SNR >= 50 dB).  Env override: OVC_PRECISION."""
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("openvoice_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        self.device = dev
        self.hps = hps
        self.zero_g = bool(getattr(hps.model, "zero_g", False))
        self.n_speakers = int(getattr(hps.data, "n_speakers", 0))
        index = dev.index if dev.index is not None else torch.cuda.current_device()
        self.native = NativeConverter(hps, index)
        self.precision = precision or os.environ.get("OVC_PRECISION", "f16x3")
        self.native.set_precision(self.precision)
        self.spec_channels = hps.data.filter_length // 2 + 1
        self.ref_enc = ReferenceEncoder(self.native, self.spec_channels, int(getattr(hps.model, "gin_channels", 256)))
        # n_speakers == 0: converter (ReferenceEncoder); > 0: V1 base speaker (enc_p / dp / sdp / emb_g), models.py:451-465
        self._expected = hot_path_keys(hps) + (ref_enc_keys() if self.n_speakers == 0 else tts_keys(hps))

    # nn.Module-ish surface used by callers of the reference
    def eval(self):
        return self

    def to(self, device):
        if torch.device(device) != self.device and torch.device(device).type != "cuda":
            raise RuntimeError("CUDA only")
        return self

    def load_state_dict(self, state_dict, strict: bool = False):
        """Returns (missing_keys, unexpected_keys) like torch with strict=False.  Unlike the
        reference, a checkpoint that lacks hot-path tensors is an error (the reference would
        silently keep random weights)."""
        provided = set(state_dict.keys())
        expected = set(self._expected)
        missing = sorted(expected - provided)
        unexpected = sorted(provided - expected)
        self.native.load_state_dict(state_dict)
        self.native.finalize()          # raises OvcError naming the first missing hot-path key
        self._state_dict = state_dict   # kept (by reference) so that per-stream replicas can be built on demand
        if strict and (missing or unexpected):
            raise RuntimeError(f"missing keys {missing}, unexpected keys {unexpected}")
        return missing, unexpected

    @torch.no_grad()
    def voice_conversion(self, y, y_lengths, sid_src, sid_tgt, tau: float = 1.0, noise=None,
                         ragged: bool = False, seed: Optional[int] = None, latents: bool = True):
        """(o_hat, y_mask, (z, z_p, z_hat)) = SynthesizerTrn.voice_conversion
        (openvoice/models.py:492-499).  ``noise`` ([B,192,T]) replaces the reference's
        ``randn_like``; when None, Philox normals are drawn in-kernel from ``seed`` (default: a
        draw from torch's global CPU generator, so ``torch.manual_seed`` makes runs repeatable).
        ``ragged=True`` converts every item at its exact length (what ``convert`` does)."""
        y = y.to(self.device, torch.float32).contiguous()
        B, _, T = y.shape
        y_lengths = y_lengths.to(self.device, torch.int64).contiguous()
        sid_src = self._expand_se(sid_src, B)
        sid_tgt = self._expand_se(sid_tgt, B)
        if noise is None and seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        if noise is not None:
            noise = noise.to(self.device, torch.float32)
        o, lat = self.native.voice_conversion(y, y_lengths, sid_src, sid_tgt, noise=noise, tau=float(tau),
                                              seed=seed or 0, ragged=ragged, latents=latents)
        y_mask = (torch.arange(T, device=self.device)[None, :] < y_lengths[:, None]).unsqueeze(1).to(torch.float32)
        return o, y_mask, lat

    @torch.no_grad()
    def infer(self, x, x_lengths, sid=None, noise_scale=1, length_scale=1, noise_scale_w=1.0, sdp_ratio=0.2,
              max_len=None, noise_w=None, noise=None, ragged: bool = False, seed: Optional[int] = None,
              latents: bool = True):
        """(o, attn, y_mask, (z, z_p, None, None)) = SynthesizerTrn.infer (openvoice/models.py:467-490) for a V1
        base-speaker checkpoint.  ``x`` [B,T] token ids, ``x_lengths`` [B], ``sid`` [B] speaker ids.
        ``noise_w`` ([B,2,T]) / ``noise`` ([B,192,>=Ty]) replace the two random draws (models.py:173, 487); when None,
        Philox normals are drawn in-kernel from ``seed``.  The expanded m_p / logs_p of the reference's return
        tuple are not materialised (they only feed z_p).  One host sync, where the reference has one too
        (y_lengths sizes every later tensor, models.py:476-478)."""
        info = self.native.tts_info()
        if not info["has_tts"]:
            raise RuntimeError("this checkpoint has no enc_p / dp / sdp / emb_g: infer() needs a V1 base speaker")
        x = x.to(torch.int64)
        if int(x.min()) < 0 or int(x.max()) >= info["n_vocab"]:
            raise ValueError(f"token ids must lie in [0, {info['n_vocab']})")
        x = x.to(self.device).contiguous()
        B, T = x.shape
        x_lengths = x_lengths.to(self.device, torch.int64).contiguous()
        if sid is None:
            raise ValueError("sid is required (n_speakers > 0)")
        sid = sid.to(torch.int64).reshape(-1)
        if int(sid.min()) < 0 or int(sid.max()) >= info["n_speakers"]:
            raise ValueError(f"speaker ids must lie in [0, {info['n_speakers']})")
        sid = sid.to(self.device).contiguous()
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        if noise_w is not None:
            noise_w = noise_w.to(self.device, torch.float32)
        y_lengths, w_ceil, _ = self.native.tts_encode(x, x_lengths, sid, noise_w=noise_w, seed=seed,
                                                      noise_scale_w=float(noise_scale_w), length_scale=float(length_scale),
                                                      sdp_ratio=float(sdp_ratio))
        Ty = int(y_lengths.max().item())                       # the sync
        if noise is not None:
            noise = noise.to(self.device, torch.float32)[:, :, :Ty].contiguous()
        o, lat = self.native.tts_decode(B, Ty, self.device, noise=noise, seed=seed + 1, noise_scale=float(noise_scale),
                                        ragged=ragged, latents=latents, max_len=max_len)
        ar = torch.arange(Ty, device=self.device)
        y_mask = (ar[None, :] < y_lengths[:, None]).unsqueeze(1).to(torch.float32)
        cum = torch.cumsum(w_ceil, 1)                          # commons.generate_path (commons.py:128-142)
        path = (ar[None, :, None] < cum[:, None, :]) & (ar[None, :, None] >= (cum - w_ceil)[:, None, :])
        attn = (path.to(torch.float32) * y_mask.transpose(1, 2)).unsqueeze(1)      # [B,1,Ty,T]
        z, z_p = lat if lat else (None, None)
        return o, attn, y_mask, (z, z_p, None, None)

    def _expand_se(self, se, B):
        se = se.to(self.device, torch.float32).reshape(se.shape[0], -1)
        if se.shape[0] == 1 and B > 1:
            se = se.expand(B, -1)
        if se.shape[0] != B:
            raise ValueError(f"speaker embedding batch {se.shape[0]} does not match batch {B}")
        return se.contiguous()


class OpenVoiceBaseClass(object):
    """openvoice/api.py:14-39."""

    def __init__(self, config_path, device="cuda:0", precision=None):
        if "cuda" in device:
            assert torch.cuda.is_available()
        hps = utils.get_hparams_from_file(config_path)
        self.model = NativeSynthesizer(hps, device, precision=precision).eval()
        self.hps = hps
        self.device = device

    def load_ckpt(self, ckpt_path):
        checkpoint_dict = torch.load(ckpt_path, map_location=torch.device("cpu"))
        a, b = self.model.load_state_dict(checkpoint_dict["model"], strict=False)
        print("Loaded checkpoint '{}'".format(ckpt_path))
        print("missing/unexpected keys:", a, b)


class BaseSpeakerTTS(OpenVoiceBaseClass):
    """openvoice/api.py:42-98: the V1 base speaker.  The acoustic model (``SynthesizerTrn.infer``) runs on the
    CUDA library; the text front end (sentence splitting, cleaners, G2P: openvoice/text/*, utils.split_sentence)
    is host-side string processing outside this build's scope (SURVEY.md section 8), so it is pluggable:
    ``text_frontend(text, language_mark) -> list of token-id lists`` (one per sentence, blanks already
    interspersed).  When the reference package is importable its own front end is used."""

    language_marks = {"english": "EN", "chinese": "ZH"}

    def __init__(self, *args, text_frontend=None, **kwargs):
        super().__init__(*args, **kwargs)
        self.text_frontend = text_frontend

    @staticmethod
    def intersperse(lst, item):
        """commons.intersperse (openvoice/commons.py:22-25): [a, b] -> [item, a, item, b, item]."""
        out = [item] * (len(lst) * 2 + 1)
        out[1::2] = lst
        return out

    @staticmethod
    def audio_numpy_concat(segment_data_list, sr, speed=1.0):
        """openvoice/api.py:56-63: sentences joined with 50 ms / speed of silence after each."""
        gap = np.zeros(int((sr * 0.05) / speed), dtype=np.float32)
        parts = []
        for seg in segment_data_list:
            parts += [np.asarray(seg, dtype=np.float32).reshape(-1), gap]
        return np.concatenate(parts) if parts else np.zeros(0, np.float32)

    def _reference_frontend(self, text, mark):
        try:
            import re
            from openvoice import utils as ref_utils          # type: ignore
            from openvoice.text import text_to_sequence      # type: ignore
        except ImportError as e:
            raise RuntimeError("no text front end: pass text_frontend=... to BaseSpeakerTTS, call tts_from_ids(), or "
                               "install the reference package for its cleaners") from e
        seqs = []
        for t in ref_utils.split_sentence(text, language_str=mark):              # api.py:66-71
            t = re.sub(r"([a-z])([A-Z])", r"\1 \2", t)                           # api.py:81
            ids = text_to_sequence(f"[{mark}]{t}[{mark}]", self.hps.symbols, self.hps.data.text_cleaners)
            if getattr(self.hps.data, "add_blank", False):
                ids = self.intersperse(ids, 0)                                   # api.py:50-52
            seqs.append(ids)
        return seqs

    @torch.no_grad()
    def tts_from_ids(self, sequences, speaker, speed=1.0, noise_scale=0.667, noise_scale_w=0.6, sdp_ratio=0.2,
                     seed: Optional[int] = None) -> List[np.ndarray]:
        """All sentences in ONE batched infer() (the reference loops over them at batch 1, api.py:79-91); every
        sentence gets what its own batch-1 call would give (ragged decode)."""
        speaker_id = self.hps.speakers[speaker] if isinstance(speaker, str) else int(speaker)
        n = len(sequences)
        if n == 0:      # the reference's loop over zero sentences yields no audio (api.py:79-91)
            return []
        T = max(len(q) for q in sequences)
        x = torch.zeros(n, T, dtype=torch.int64)
        for i, q in enumerate(sequences):
            x[i, :len(q)] = torch.as_tensor(q, dtype=torch.int64)
        lens = torch.tensor([len(q) for q in sequences], dtype=torch.int64)
        sid = torch.full((n,), speaker_id, dtype=torch.int64)
        o, _, y_mask, _ = self.model.infer(x, lens, sid=sid, noise_scale=noise_scale, noise_scale_w=noise_scale_w,
                                           length_scale=1.0 / speed, sdp_ratio=sdp_ratio, ragged=True, seed=seed,
                                           latents=False)
        frames = y_mask[:, 0].sum(1).long().cpu()
        o = o[:, 0].float().cpu().numpy()
        hop = self.hps.data.hop_length
        return [o[i, : int(frames[i]) * hop].copy() for i in range(n)]

    def tts(self, text, output_path, speaker, language="English", speed=1.0):
        """openvoice/api.py:73-98."""
        mark = self.language_marks.get(language.lower(), None)
        assert mark is not None, f"language {language} is not supported"
        frontend = self.text_frontend or self._reference_frontend
        sequences = frontend(text, mark)
        audio_list = self.tts_from_ids(sequences, speaker, speed=speed)
        audio = self.audio_numpy_concat(audio_list, sr=self.hps.data.sampling_rate, speed=speed)
        if output_path is None:
            return audio
        _write_audio(output_path, audio, self.hps.data.sampling_rate)


class ToneColorConverter(OpenVoiceBaseClass):
    """openvoice/api.py:101-201.

    ``precision=`` ("f16x3" default, "fp32", "f16" or "f16s") is passed to :class:`NativeSynthesizer`;
    "f16s" is the fp16 configuration: fp16 generator activations, half the generator's memory, o_hat SNR >= 50 dB."""

    def __init__(self, *args, **kwargs):
        enable_watermark = kwargs.pop("enable_watermark", True)
        super().__init__(*args, **kwargs)
        self.watermark_model = None
        if enable_watermark:
            # the reference fails hard at `import wavmark` (openvoice/api.py:105-107); silently returning
            # un-watermarked audio to a caller who asked for the watermark is worse than failing
            try:
                import wavmark  # type: ignore
            except ImportError as e:
                raise ImportError("ToneColorConverter(enable_watermark=True) needs the third-party `wavmark` package "
                                  "(openvoice/api.py:105-107); pass enable_watermark=False to convert without it") from e
            self.watermark_model = wavmark.load_model().to(self.device)
        self.version = getattr(self.hps, "_version_", "v1")

    # ------------------------------------------------------------------ speaker embedding
    def extract_se(self, ref_wav_list, se_save_path=None):
        """openvoice/api.py:114-139: mean ReferenceEncoder embedding over the given clips,
        shape [1, gin, 1]."""
        if isinstance(ref_wav_list, (str, np.ndarray)):
            ref_wav_list = [ref_wav_list]
        hps = self.hps
        gs = []
        for fname in ref_wav_list:
            audio_ref = _load_audio(fname, hps.data.sampling_rate)
            y = torch.from_numpy(audio_ref).to(self.device).unsqueeze(0).contiguous()
            n = torch.tensor([y.shape[1]], dtype=torch.int64, device=self.device)
            y, _ = self.model.native.spectrogram(y, n)          # = spectrogram_torch (api.py:126-128)
            g = self.model.native.reference_encoder(y).unsqueeze(-1)   # = model.ref_enc(y.transpose(1, 2)) (api.py:130)
            gs.append(g.detach())
        gs = torch.stack(gs).mean(0)
        if se_save_path is not None:
            os.makedirs(os.path.dirname(se_save_path), exist_ok=True)
            torch.save(gs.cpu(), se_save_path)
        return gs

    # ------------------------------------------------------------------ conversion
    def convert(self, audio_src_path, src_se, tgt_se, output_path=None, tau=0.3, message="default",
                noise=None):
        """openvoice/api.py:141-160.  Returns float32 samples (256 * (L // 256) of them) or writes
        ``output_path``.  ``noise`` ([1,192,T]) optionally replaces the random draw (tests)."""
        audio = self.convert_batch([audio_src_path], src_se, tgt_se, tau=tau, messages=[message],
                                   noise=None if noise is None else [noise])[0]
        if output_path is None:
            return audio
        _write_audio(output_path, audio, self.hps.data.sampling_rate)

    @torch.no_grad()
    def convert_batch(self, audios: Sequence[AudioLike], src_se, tgt_se, tau: float = 0.3,
                      messages: Optional[Sequence[str]] = None, noise: Optional[Sequence] = None,
                      max_batch: int = 64) -> List[np.ndarray]:
        """Convert a list of utterances (paths or waveforms at the model sampling rate); every item
        gets exactly what ``convert`` would return for it alone.  ``src_se`` / ``tgt_se`` are either
        one [1,gin,1] embedding for all items or a sequence of per-item embeddings."""
        hps = self.hps
        n = len(audios)
        waves = [_load_audio(a, hps.data.sampling_rate) for a in audios]
        src = self._stack_se(src_se, n)
        tgt = self._stack_se(tgt_se, n)
        out: List[Optional[np.ndarray]] = [None] * n
        order = sorted(range(n), key=lambda i: -len(waves[i]))     # similar lengths share a launch
        hop = hps.data.hop_length
        for lo in range(0, n, max_batch):
            idx = order[lo: lo + max_batch]
            res = self._convert_chunk([waves[i] for i in idx], src[idx], tgt[idx], tau,
                                      None if noise is None else [noise[i] for i in idx])
            for i, a in zip(idx, res):
                msg = messages[i] if messages is not None else "default"
                out[i] = self.add_watermark(a, msg)
        return out  # type: ignore[return-value]

    # ------------------------------------------------------------------ one utterance per stream
    @torch.no_grad()
    def convert_concurrent(self, audios: Sequence[AudioLike], src_se, tgt_se, tau: float = 0.3, streams: int = 4,
                           messages: Optional[Sequence[str]] = None) -> List[np.ndarray]:
        """Serve many SMALL independent requests: utterance i runs alone (batch 1, exactly ``convert``) on CUDA
        stream ``i % streams``, each stream with its own converter replica (context + workspace), so the
        latency-bound kernels of different requests overlap on the GPU -- north_star's "one utterance per stream".
        For large batches ``convert_batch`` (one launch sequence for the whole batch) is the faster path."""
        n = len(audios)
        src = self._stack_se(src_se, n)
        tgt = self._stack_se(tgt_se, n)
        reps = self._replicas(max(1, min(streams, n)))
        S, depth = len(reps), 2                       # requests in flight per stream (pinned staging slots)
        out: List[Optional[np.ndarray]] = [None] * n
        for w0 in range(0, n, S * depth):
            wave = list(range(w0, min(n, w0 + S * depth)))
            pending = []
            for j, i in enumerate(wave):
                conv, stream = reps[j % S]
                with torch.cuda.stream(stream):
                    pending.append(conv._enqueue_single(_load_audio(audios[i], self.hps.data.sampling_rate), src[i: i + 1],
                                                        tgt[i: i + 1], tau, j // S))
            for _, stream in reps:
                stream.synchronize()
            for i, (host, n_samples) in zip(wave, pending):
                msg = messages[i] if messages is not None else "default"
                out[i] = self.add_watermark(host[:n_samples].numpy().copy(), msg)
        return out  # type: ignore[return-value]

    def _replicas(self, count):
        """[(converter, stream)]: replica 0 is this object; the others share its hparams and checkpoint."""
        reps = self.__dict__.setdefault("_reps", [(self, torch.cuda.Stream(device=self.device))])
        while len(reps) < count:
            twin = ToneColorConverter.__new__(ToneColorConverter)
            twin.hps, twin.device, twin.watermark_model, twin.version = self.hps, self.device, None, self.version
            twin.model = NativeSynthesizer(self.hps, self.device, precision=self.model.precision)
            twin.model.load_state_dict(self.model._state_dict)
            reps.append((twin, torch.cuda.Stream(device=self.device)))
        return reps[:count]

    def _enqueue_single(self, wave, src, tgt, tau, slot):
        """Asynchronous batch-1 conversion on the current stream, staging through pinned slot ``slot``;
        returns (pinned host buffer, samples).  The caller synchronises the stream before reading / reusing it."""
        hop = self.hps.data.hop_length
        dev = self.device
        L = len(wave)
        if L // hop < 1 or L <= (self.hps.data.filter_length - hop) // 2:
            raise ValueError("audio too short")
        stage = self._pinned(f"cin{slot}", L)
        stage.copy_(torch.from_numpy(wave))
        wav = stage.to(dev, non_blocking=True).view(1, L)
        wlen = torch.tensor([L], dtype=torch.int64, device=dev)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        o, _ = self.model.native.convert_waveform(wav, wlen, src, tgt, tau=float(tau), seed=seed)
        host = self._pinned(f"cout{slot}", o.numel())
        host.copy_(o.view(-1), non_blocking=True)
        return host, (L // hop) * hop

    # receptive field of the whole path in spectrogram frames: enc_q +-32 (16 WN layers of k=5), flow forward and
    # reverse +-32 each (4 couplings x 4 layers), generator +-13.3 (conv_pre 3, transposed convs, ResBlocks up to
    # k=11 d=5) -> 110; 128 leaves margin (SURVEY.md section 5 "long-context": measured ~109)
    HALO_FRAMES = 128

    @torch.no_grad()
    def convert_long(self, audio_src_path, src_se, tgt_se, output_path=None, tau=0.3, message="default",
                     window_frames: int = 2048, noise=None, max_batch: int = 32):
        """Row f4 (time-tiled execution): convert a clip of any length with bounded memory.  The spectrogram is
        cut into windows of ``window_frames`` frames plus a halo of the path's receptive field on both sides; the
        windows run as one ragged batch and only their interiors are kept, so the result equals ``convert`` on the
        whole clip (same noise tensor: drawn once for the whole clip, or passed as ``noise`` [192, T])."""
        hps = self.hps
        hop, dev = hps.data.hop_length, self.device
        wav = torch.from_numpy(_load_audio(audio_src_path, hps.data.sampling_rate)).to(dev)
        L = wav.numel()
        spec, _ = self.model.native.spectrogram(wav[None].contiguous(), torch.tensor([L], dtype=torch.int64, device=dev))
        T = spec.shape[2]
        C = hps.model.inter_channels
        if noise is None:
            gen = torch.Generator(device=dev)
            gen.manual_seed(int(torch.randint(0, 2 ** 62, (1,)).item()))
            noise = torch.randn(C, T, device=dev, generator=gen)
        noise = noise.to(dev, torch.float32).reshape(C, T)
        H = self.HALO_FRAMES
        starts = list(range(0, T, window_frames))
        wins = [(max(0, s - H), min(T, s + window_frames + H), s, min(T, s + window_frames)) for s in starts]
        Wmax = max(hi - lo for lo, hi, _, _ in wins)
        out = torch.empty(T * hop, device=dev, dtype=torch.float32)
        src = self._stack_se(src_se, 1)
        tgt = self._stack_se(tgt_se, 1)
        for i0 in range(0, len(wins), max_batch):
            chunk = wins[i0: i0 + max_batch]
            B = len(chunk)
            sp = torch.zeros(B, spec.shape[1], Wmax, device=dev)
            nz = torch.zeros(B, C, Wmax, device=dev)
            for b, (lo, hi, _, _) in enumerate(chunk):
                sp[b, :, : hi - lo] = spec[0, :, lo:hi]
                nz[b, :, : hi - lo] = noise[:, lo:hi]
            lens = torch.tensor([hi - lo for lo, hi, _, _ in chunk], dtype=torch.int64, device=dev)
            o, _, _ = self.model.voice_conversion(sp, lens, src.expand(B, -1), tgt.expand(B, -1), tau=tau, noise=nz,
                                                  ragged=True, latents=False)
            for b, (lo, hi, s, e) in enumerate(chunk):
                out[s * hop: e * hop] = o[b, 0, (s - lo) * hop: (e - lo) * hop]
        audio = self.add_watermark(out.cpu().numpy(), message)
        if output_path is None:
            return audio
        _write_audio(output_path, audio, hps.data.sampling_rate)

    def _stack_se(self, se, n):
        if isinstance(se, (list, tuple)):
            se = torch.cat([s.reshape(1, -1) for s in se], 0)
        se = se.to(self.device, torch.float32).reshape(se.shape[0], -1)
        if se.shape[0] == 1:
            se = se.expand(n, -1)
        assert se.shape[0] == n, "one speaker embedding per utterance (or a single one for all)"
        return se

    def _enqueue_chunk(self, waves, src, tgt, tau, noise, slot=0):
        """Stage, upload and launch one ragged batch on the current stream WITHOUT synchronising the host.
        Returns (o [B, 256 * Tmax] on the device, frames per item)."""
        hps = self.hps
        hop = hps.data.hop_length
        B = len(waves)
        frames = [len(w) // hop for w in waves]
        if min(frames) < 1:
            raise ValueError("audio shorter than one hop")
        Tmax = max(frames)
        dev = self.device
        if min(len(w) for w in waves) <= (hps.data.filter_length - hop) // 2:
            raise ValueError("audio shorter than the STFT reflect padding")   # torch raises here too
        # host -> device: one pinned staging buffer per slot (cached across calls: cudaHostAlloc is slow), one copy;
        # a slot is restaged only after its previous upload has left it
        # the padded length is rounded up to 16 hops: batches of similar length share one launch signature, so the native
        # library replays their CUDA graph; every item still runs at its own exact length (ragged), so nothing changes
        Lmax = -(-max(len(w) for w in waves) // (16 * hop)) * (16 * hop)
        ev = self.__dict__.setdefault("_h2d_done", {}).get(slot)
        if ev is not None:
            ev.synchronize()
        stage = self._pinned(f"in{slot}", B * Lmax).view(B, Lmax)
        stage_np = stage.numpy()
        lens = np.array([len(w) for w in waves], dtype=np.int64)

        def put(b):
            w = waves[b]
            stage_np[b, : len(w)] = w
            if len(w) < Lmax:
                stage_np[b, len(w):] = 0.0
        _parallel(put, B)
        # device-side buffers are cached per slot too: with every address stable, a repeated (batch, length) call is
        # replayed from a CUDA graph by the native library (include/ovc.h: OVC_OPT_GRAPH)
        wav = self._dev(f"wav{slot}", B * Lmax, torch.float32).view(B, Lmax)
        wav.copy_(stage, non_blocking=True)
        lens_pin = self._pinned_i64(f"len{slot}", B)
        lens_pin.copy_(torch.from_numpy(lens))
        wlen = self._dev(f"len{slot}", B, torch.int64)
        wlen.copy_(lens_pin, non_blocking=True)
        src_d = self._dev(f"src{slot}", src.numel(), torch.float32).view(B, -1)
        src_d.copy_(src.reshape(B, -1), non_blocking=True)
        tgt_d = self._dev(f"tgt{slot}", tgt.numel(), torch.float32).view(B, -1)
        tgt_d.copy_(tgt.reshape(B, -1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        self._h2d_done[slot] = ev
        nz = None
        if noise is not None:
            nz = torch.zeros(B, hps.model.inter_channels, Lmax // hop, device=dev, dtype=torch.float32)
            for b, q in enumerate(noise):
                q = q.reshape(hps.model.inter_channels, -1)
                nz[b, :, : q.shape[1]] = q.to(dev)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        # spectrogram + voice_conversion, every item at its own exact length (api.py:148-154)
        o, _ = self.model.native.convert_waveform(wav, wlen, src_d, tgt_d, noise=nz, tau=float(tau), seed=seed,
                                                  out=self._dev(f"out{slot}", B * (Lmax // hop) * hop, torch.float32),
                                                  frames_out=self._dev(f"fr{slot}", B, torch.int64))
        return o.view(B, -1), frames

    def _convert_chunk(self, waves, src, tgt, tau, noise):
        hop = self.hps.data.hop_length
        o, frames = self._enqueue_chunk(waves, src, tgt, tau, noise)
        host = self._pinned("out", o.numel()).view(o.shape)
        host.copy_(o, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        audio = host.numpy()
        return _parallel(lambda b: audio[b, : frames[b] * hop].copy(), len(waves))

    @torch.no_grad()
    def convert_batch_device(self, audios: Sequence[AudioLike], src_se, tgt_se, tau: float = 0.3, slot: int = 0):
        """``convert_batch`` up to the device: stages and launches ONE ragged batch asynchronously on the current
        stream and returns (o [n, max samples] float32 on the device, samples per item).  No host synchronisation,
        no device -> host copy: the building block of ``distributed.convert_sharded_async`` (waveforms gathered
        GPU-to-GPU over NCCL) and of pipelined serving.  ``slot`` picks the pinned upload buffer (alternate 0 / 1
        between in-flight calls)."""
        waves = [_load_audio(a, self.hps.data.sampling_rate) for a in audios]
        n = len(waves)
        o, frames = self._enqueue_chunk(waves, self._stack_se(src_se, n), self._stack_se(tgt_se, n), tau, None, slot)
        hop = self.hps.data.hop_length
        return o, [f * hop for f in frames]

    def _dev(self, name, numel, dtype):
        """Grow-only device buffers (per upload slot): the result of slot s is overwritten by the next call on slot s."""
        cache = self.__dict__.setdefault("_dev_cache", {})
        buf = cache.get(name)
        if buf is None or buf.numel() < numel or buf.dtype != dtype:
            buf = torch.empty(int(numel * 1.25) + 64, dtype=dtype, device=self.device)
            cache[name] = buf
        return buf[:numel]

    def _pinned_i64(self, name, numel):
        cache = self.__dict__.setdefault("_pin_cache", {})
        buf = cache.get(name)
        if buf is None or buf.numel() < numel:
            buf = torch.empty(int(numel) + 64, dtype=torch.int64).pin_memory()
            cache[name] = buf
        return buf[:numel]

    def _pinned(self, name, numel):
        """Grow-only pinned host staging buffers."""
        cache = self.__dict__.setdefault("_pin_cache", {})
        buf = cache.get(name)
        if buf is None or buf.numel() < numel:
            buf = torch.empty(int(numel * 1.25) + 1024, dtype=torch.float32).pin_memory()
            cache[name] = buf
        return buf[:numel]

    # ------------------------------------------------------------------ watermark (third-party model)
    _WM_CHUNK = 16000      # samples per watermarked chunk
    _WM_STRIDE = 32000     # chunk n starts at n * 32000 (openvoice/api.py:169-171)

    def _wm_chunks(self, audio, count):
        """Yield (index, slice) of the first ``count`` watermark chunks; a short chunk ends the walk."""
        for n in range(count):
            sl = slice(n * self._WM_STRIDE, n * self._WM_STRIDE + self._WM_CHUNK)
            yield n, sl, len(audio[sl]) == self._WM_CHUNK

    def add_watermark(self, audio, message):
        """Embed ``message`` with the wavmark model, 32 bits per 16000-sample chunk, chunks 32000 samples apart
        (behaviour of openvoice/api.py:162-184, incl. the "Audio too short" early stop).  No model -> no-op.
        The chunks are cut, encoded and written back ON THE DEVICE as one batch (``watermark_device``): one upload and
        one download per utterance instead of two host round trips per chunk."""
        if self.watermark_model is None:
            return audio
        dev_audio = torch.as_tensor(audio, dtype=torch.float32).to(self.device)
        watermark_device(dev_audio, utils.string_to_bits(message).reshape(-1), self.watermark_model)
        audio[...] = dev_audio.cpu().numpy()
        return audio

    def detect_watermark(self, audio, n_repeat):
        """Decode ``n_repeat`` chunks back to text (openvoice/api.py:186-201); "Fail" when the audio is too short."""
        if self.watermark_model is None:
            raise RuntimeError("detect_watermark needs the wavmark model: construct with enable_watermark=True")
        rows = []
        for n, sl, full in self._wm_chunks(audio, n_repeat):
            if not full:
                print("Audio too short, fail to detect watermark")
                return "Fail"
            with torch.no_grad():
                sig = torch.as_tensor(audio[sl], dtype=torch.float32, device=self.device)[None]
                rows.append((self.watermark_model.decode(sig) >= 0.5).int().detach().cpu().numpy().squeeze())
        return utils.bits_to_string(np.stack(rows).reshape(-1, 8))
