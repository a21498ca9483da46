"""GPU parity of the V1 TTS front half (SURVEY.md section 8 rows a12 / a13 / f3) through the C ABI
(ovc_tts_encode / ovc_tts_decode) against vectors of the REAL reference's SynthesizerTrn.infer
(tests/golden/tts_*.npz, oracle/make_golden_tts.py) and against the oracle.

Tolerances: durations (w_ceil, y_lengths) are integers -> exact.  Floating point: max|delta| <= 1e-4 * rms(ref)
for the audio (the repo-wide fp32 gate); text-side tensors (x, m_p, logs_p, logw_dp) 1e-4 absolute on O(1) values
(measured 2e-5: the 1x1 projections run as 3xTF32 on the tensor cores); logw_sdp 5e-4 on the goldens (measured 2.7e-4;
the spline inverses amplify, see test_one_token_and_very_long_text for the tail on long texts)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle.golden import Golden

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["tts_b1_t37", "tts_b2_padded", "tts_b1_t121_tails"]


def load(name):
    d = Golden(os.path.join(GOLD, name + ".npz"))
    return d, json.loads(str(d["meta"]))


def inputs(c):
    from oracle import tts_oracle as T
    tokens, lengths, sid, noise_w = T.synthetic_tts_inputs(c["B"], c["T"], c["seed"], c["lengths"])
    noise = torch.randn(c["B"], 192, 40 * c["T"] + 64, generator=torch.Generator().manual_seed(30_000 + c["seed"]))
    return tokens, lengths, sid, noise_w, noise


def rms(a):
    return float(np.sqrt(np.mean(np.square(a, dtype=np.float64))))


@pytest.fixture(scope="module")
def tts():
    from conftest import get_native_tts
    return get_native_tts()


@pytest.mark.parametrize("name", CASES)
def test_text_side_matches_reference(name, tts):
    d, c = load(name)
    tokens, lengths, sid, noise_w, _ = inputs(c)
    nat = tts.native
    nat.debug_enable(True)
    dev = tts.device
    yl, w_ceil, logw = nat.tts_encode(tokens.to(dev), lengths.to(dev), sid.to(dev), noise_w=noise_w.to(dev),
                                      noise_scale_w=c["noise_scale_w"], length_scale=c["length_scale"],
                                      sdp_ratio=c["sdp_ratio"])
    torch.cuda.synchronize()
    mask = (np.arange(c["T"])[None, :] < lengths.numpy()[:, None]).astype(np.float32)
    x = nat.debug_fetch("tts.x")                 # [B, T, H] channels-last
    st = nat.debug_fetch("tts.stats")
    ls, ld = nat.debug_fetch("tts.logw_sdp")[:, 0], nat.debug_fetch("tts.logw_dp")[:, 0]
    nat.debug_enable(False)
    err = {
        "x": np.abs(x * mask[:, :, None] - d["x"].transpose(0, 2, 1)).max(),
        "m_p": np.abs(st[..., :192] * mask[:, :, None] - d["m_p"].transpose(0, 2, 1)).max(),
        "logs_p": np.abs(st[..., 192:] * mask[:, :, None] - d["logs_p"].transpose(0, 2, 1)).max(),
        "logw_dp": np.abs(ld * mask - d["logw_dp"][:, 0]).max(),
        "logw_sdp": np.abs(ls * mask - d["logw_sdp"][:, 0]).max(),
    }
    print(name, {k: float(v) for k, v in err.items()})
    for k in ("x", "m_p", "logs_p", "logw_dp"):
        assert err[k] < 1e-4, (k, err)
    assert err["logw_sdp"] < 1e-4, err          # three spline inverses amplify the conditioning error (measured <= 6e-5)
    assert np.array_equal(w_ceil.cpu().numpy(), d["w_ceil"])
    assert np.array_equal(yl.cpu().numpy(), d["y_lengths"])
    ref_logw = (d["logw_sdp"] * c["sdp_ratio"] + d["logw_dp"] * (1 - c["sdp_ratio"]))[:, 0] * mask
    assert np.abs(logw.cpu().numpy() - ref_logw).max() < 1e-4


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
@pytest.mark.parametrize("name", CASES)
def test_infer_matches_reference(name, precision, tts):
    d, c = load(name)
    tokens, lengths, sid, noise_w, noise = inputs(c)
    tts.native.set_precision(precision)
    try:
        o, attn, y_mask, (z, z_p, _, _) = tts.infer(tokens, lengths, sid=sid, noise_scale=c["noise_scale"],
                                                    length_scale=c["length_scale"], noise_scale_w=c["noise_scale_w"],
                                                    sdp_ratio=c["sdp_ratio"], noise_w=noise_w, noise=noise)
        torch.cuda.synchronize()
    finally:
        tts.native.set_precision(tts.precision)
    yl = d["y_lengths"]
    assert np.array_equal(y_mask[:, 0].sum(1).long().cpu().numpy(), yl)
    assert np.array_equal(attn[:, 0].sum(1).cpu().numpy(), d["w_ceil"])          # frames per token
    assert tuple(o.shape) == d.shape("o")
    ym = y_mask.cpu().numpy()
    e_zp = np.abs(d.pick("z_p", z_p.cpu().numpy()) - d["z_p"] * d.pick("z_p", ym)).max() / d.rms("z_p")
    e_z = np.abs(d.pick("z", z.cpu().numpy() * ym) - d["z"] * d.pick("z", ym)).max() / d.rms("z")
    e_o = np.abs(d.pick("o", o.cpu().numpy()) - d["o"]).max() / d.rms("o")
    print(name, precision, dict(z_p=e_zp, z=e_z, o=e_o))
    assert e_zp < 1e-4 and e_z < 1e-4 and e_o < 1e-4


def test_ragged_batch_equals_solo_and_oracle(tts):
    """ragged=True gives every utterance its own batch-1 result (what BaseSpeakerTTS.tts's loop does, api.py:79-91)."""
    from oracle import tts_oracle as T
    d, c = load("tts_b2_padded")
    tokens, lengths, sid, noise_w, noise = inputs(c)
    kw = dict(noise_scale=c["noise_scale"], length_scale=c["length_scale"], noise_scale_w=c["noise_scale_w"],
              sdp_ratio=c["sdp_ratio"])
    o, _, y_mask, _ = tts.infer(tokens, lengths, sid=sid, noise_w=noise_w, noise=noise, ragged=True, latents=False, **kw)
    n = int(lengths[1])
    o1, _, m1, _ = tts.infer(tokens[1:2, :n], lengths[1:2], sid=sid[1:2], noise_w=noise_w[1:2, :, :n], noise=noise[1:2],
                             latents=False, **kw)
    torch.cuda.synchronize()
    ny = int(m1.sum())
    assert ny == int(d["y_lengths"][1])
    a, b = o[1, 0, :ny * 256].cpu().numpy(), o1[0, 0, :ny * 256].cpu().numpy()
    assert np.abs(a - b).max() <= 1e-5 * rms(b)          # tile boundaries differ between the two launches
    with torch.no_grad():
        r = T.tts_infer(T.synthetic_tts_state_dict(), tokens, lengths, sid, noise_w, noise, ragged=True, **kw)
    ref = r["o"][1, 0, :ny * 256].numpy()
    assert np.abs(a - ref).max() < 1e-4 * rms(ref)


def test_philox_draws_are_repeatable_and_plausible(tts):
    from oracle import tts_oracle as T
    tokens, lengths, sid, _ = T.synthetic_tts_inputs(3, 40, 11, [40, 33, 9])
    a = tts.infer(tokens, lengths, sid=sid, noise_scale=0.667, noise_scale_w=0.6, seed=7, ragged=True)
    b = tts.infer(tokens, lengths, sid=sid, noise_scale=0.667, noise_scale_w=0.6, seed=7, ragged=True)
    c = tts.infer(tokens, lengths, sid=sid, noise_scale=0.667, noise_scale_w=0.6, seed=8, ragged=True)
    torch.cuda.synchronize()
    assert torch.equal(a[0], b[0]) and torch.equal(a[3][1], b[3][1])
    assert not torch.equal(a[3][1], c[3][1])
    yl = a[2].shape[-1]
    assert 40 <= yl <= 40 * 30
    assert torch.isfinite(a[0]).all() and float(a[0].abs().max()) <= 1.0


def test_base_speaker_tts_api(tts, tmp_path):
    """BaseSpeakerTTS over config.json + checkpoint.pth, batched sentences, 50 ms joins (api.py:56-63, 73-98)."""
    import copy
    from oracle import tts_oracle as T
    from oracle import vc_oracle as O
    from openvoice_b200.api import BaseSpeakerTTS
    hp = copy.deepcopy(O.DEFAULT_HPARAMS)
    hp["data"]["n_speakers"] = T.TTS_HPARAMS["n_speakers"]
    hp["data"]["add_blank"] = True
    hp["data"]["text_cleaners"] = []
    hp["symbols"] = [chr(ord("a") + i) for i in range(26)] + list(" .,!?-'\"():;_*")[:14]
    hp["speakers"] = {"default": 1, "whispering": 2}
    (tmp_path / "config.json").write_text(json.dumps(hp))
    torch.save({"model": T.synthetic_tts_state_dict()}, tmp_path / "checkpoint.pth")
    sym = {s: i for i, s in enumerate(hp["symbols"])}

    def frontend(text, mark):
        assert mark == "EN"
        return [BaseSpeakerTTS.intersperse([sym[ch] for ch in s.strip().lower() if ch in sym], 0)
                for s in text.split(".") if s.strip()]

    eng = BaseSpeakerTTS(str(tmp_path / "config.json"), device="cuda:0", text_frontend=frontend)
    eng.load_ckpt(str(tmp_path / "checkpoint.pth"))
    torch.manual_seed(3)
    audio = eng.tts("hello there. general kenobi", None, speaker="default", language="English", speed=1.0)
    assert audio.dtype == np.float32 and np.isfinite(audio).all()
    gap = int(22050 * 0.05)
    seqs = frontend("hello there. general kenobi", "EN")
    parts = eng.tts_from_ids(seqs, "default", seed=5)
    assert len(parts) == 2 and all(len(p) % 256 == 0 and len(p) > 0 for p in parts)
    joined = eng.audio_numpy_concat(parts, 22050, 1.0)
    assert len(joined) == sum(len(p) for p in parts) + 2 * gap
    out = tmp_path / "o.npy"
    eng.tts("hello there", str(out), speaker="whispering", speed=1.2)
    assert os.path.exists(out)
    with pytest.raises(ValueError):
        eng.model.infer(torch.tensor([[99]]), torch.tensor([1]), sid=torch.tensor([0]))


def test_simple_kernels_fallback_matches_reference(tts):
    """OVC_OPT_TTS_SIMPLE runs the one-thread-per-element kernels (the CPU-checked element functions, also the fallback
    for very long texts) instead of the warp LayerNorm / fused attention: same goldens."""
    d, c = load("tts_b2_padded")
    tokens, lengths, sid, noise_w, _ = inputs(c)
    dev = tts.device
    tts.native.set_option("tts_simple", 1)
    try:
        yl, wc, lw = tts.native.tts_encode(tokens.to(dev), lengths.to(dev), sid.to(dev), noise_w=noise_w.to(dev),
                                           noise_scale_w=c["noise_scale_w"], length_scale=c["length_scale"],
                                           sdp_ratio=c["sdp_ratio"])
        torch.cuda.synchronize()
    finally:
        tts.native.set_option("tts_simple", 0)
    assert np.array_equal(wc.cpu().numpy(), d["w_ceil"]) and np.array_equal(yl.cpu().numpy(), d["y_lengths"])


def test_max_len_cuts_the_generator_only(tts):
    """o = dec((z * y_mask)[:, :, :max_len]) (models.py:489): the flow runs on every frame, the generator on the first max_len."""
    from oracle import tts_oracle as T
    d, c = load("tts_b1_t37")
    tokens, lengths, sid, noise_w, noise = inputs(c)
    kw = dict(noise_scale=c["noise_scale"], length_scale=c["length_scale"], noise_scale_w=c["noise_scale_w"],
              sdp_ratio=c["sdp_ratio"])
    o, _, y_mask, (z, _, _, _) = tts.infer(tokens, lengths, sid=sid, noise_w=noise_w, noise=noise, max_len=40, **kw)
    torch.cuda.synchronize()
    assert tuple(o.shape) == (1, 1, 40 * 256) and y_mask.shape[-1] == int(d["y_lengths"][0])
    with torch.no_grad():
        r = T.tts_infer(T.synthetic_tts_state_dict(), tokens, lengths, sid, noise_w, noise, max_len=40, **kw)
    ref = r["o"].numpy()
    assert np.abs(o.cpu().numpy() - ref).max() < 1e-4 * rms(ref)
    assert np.abs(z.cpu().numpy() - d["z"]).max() < 1e-4 * rms(d["z"])        # z is the full-length latent


def test_one_token_and_very_long_text(tts):
    """T = 1 (every conv is all padding) and T = 1500 (8 x T logits exceed 48 KB: the plain attention kernels take over)."""
    from oracle import tts_oracle as T
    from oracle import vc_oracle as V
    sd = T.synthetic_tts_state_dict()
    for B, Tn, lens in ((1, 1, [1]), (2, 1500, [1500, 700])):
        tokens, lengths, sid, noise_w = T.synthetic_tts_inputs(B, Tn, 21, lens)
        dev = tts.device
        yl, w_ceil, logw = tts.native.tts_encode(tokens.to(dev), lengths.to(dev), sid.to(dev), noise_w=noise_w.to(dev),
                                                 noise_scale_w=0.6, length_scale=1.0, sdp_ratio=0.2)
        torch.cuda.synchronize()
        with torch.no_grad():
            x, _, _, mask = T.text_encoder(sd, tokens, lengths)
            g = sd["emb_g.weight"][sid].unsqueeze(-1)
            lw = T.sdp_reverse(sd, x, mask, g, noise_w, 0.6) * 0.2 + T.duration_predictor(sd, x, mask, g) * 0.8
            ref = torch.ceil(torch.exp(lw) * mask)[:, 0].numpy()
        got = w_ceil.cpu().numpy()
        e_logw = np.abs(logw.cpu().numpy() - (lw * mask)[:, 0].numpy())
        print("long text", (B, Tn), "logw err max", float(e_logw.max()), "n > 5e-4:", int((e_logw > 5e-4).sum()))
        # The whole duration chain (SDP pre / DDSConv 1x1 / proj, DP convs) runs in plain fp32 on the CUDA cores, the
        # text encoder's projections in split-precision fp16: x agrees with the oracle to ~5e-6, so even where the spline
        # inverse is ill-conditioned (a bin's derivative at its 1e-3 floor: inverse slope up to 1e3) logw stays within
        # 5e-4 (measured 1.4e-4 at T = 1500; the fp32 oracle itself sits 5e-4 from an fp64 evaluation there) and the
        # INTEGER durations are exact.
        assert e_logw.max() < 5e-4, (B, Tn, float(e_logw.max()))
        assert np.array_equal(got, ref), (B, Tn, int((got != ref).sum()))
        if Tn == 1:
            o, _, y_mask, _ = tts.infer(tokens, lengths, sid=sid, noise_w=noise_w, noise_scale=0.5, noise_scale_w=0.6, seed=1)
            torch.cuda.synchronize()
            assert o.shape[-1] == int(got.sum()) * 256 and torch.isfinite(o).all()


def test_decode_needs_a_matching_encode(tts):
    from oracle import tts_oracle as T
    from openvoice_b200._native import OvcError
    from conftest import get_native
    conv = get_native(False)                                      # converter checkpoint: no TTS members
    assert conv.native.tts_info()["has_tts"] == 0
    with pytest.raises(OvcError):
        conv.native.tts_decode(1, 10, conv.device)
    with pytest.raises(RuntimeError):
        conv.infer(torch.zeros(1, 3, dtype=torch.int64), torch.tensor([3]), sid=torch.tensor([0]))
    tokens, lengths, sid, noise_w = T.synthetic_tts_inputs(2, 9, 5)
    dev = tts.device
    tts.native.tts_encode(tokens.to(dev), lengths.to(dev), sid.to(dev), noise_w=noise_w.to(dev))
    with pytest.raises(ValueError):
        tts.native.tts_decode(3, 40, dev)                         # B differs from the pending encode
    o, _ = tts.native.tts_decode(2, 40, dev, seed=3, noise_scale=0.3)
    torch.cuda.synchronize()
    assert torch.isfinite(o).all()
