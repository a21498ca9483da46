"""-m gpu: precision "f16s" (mode 3), the generator with fp16 activations in memory.

Gate: o_hat SNR >= 50 dB against the fp32 reference (the CPU emulation of the rounding contract,
oracle/f16_storage.py, gives ~58.5 dB on the goldens).  Everything before the generator runs as in "f16x3",
so z / z_p / z_hat must be bit-identical to that mode."""
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import f16_storage as H
from oracle import vc_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
GATE_DB = 50.0


def load(name):
    d = np.load(os.path.join(GOLD, name + ".npz"))
    return d, json.loads(str(d["meta"]))


def run(model, mode, spec, lengths, gs, gt, noise, tau, ragged=False, debug=False):
    nat = model.native
    nat.set_precision(mode)
    nat.debug_enable(debug)
    try:
        o, _, lat = model.voice_conversion(spec.cuda(), lengths.cuda(), gs.cuda(), gt.cuda(), tau=tau,
                                           noise=None if noise is None else noise.cuda(), ragged=ragged)
        torch.cuda.synchronize()
    finally:
        nat.debug_enable(False)
        nat.set_precision(model.precision)
    return o.cpu(), tuple(t.cpu() for t in lat)


@pytest.fixture(scope="module")
def model():
    from conftest import get_native
    return get_native(False)


@pytest.mark.parametrize("name", ["vc_b1_t24", "vc_b1_t67", "vc_b2_padded", "vc_b1_t24_tau0", "vc_b1_t24_v2"])
def test_golden_snr_and_latents(name):
    from conftest import get_native
    d, c = load(name)
    m = get_native(c["zero_g"])
    spec, lengths, gs, gt, noise = O.synthetic_inputs(c["B"], c["T"], c["seed"], lengths=c["lengths"])
    o, lat = run(m, "f16s", spec, lengths, gs, gt, noise, c["tau"])
    _, lat3 = run(m, "f16x3", spec, lengths, gs, gt, noise, c["tau"])
    snr = H.snr_db(o, torch.from_numpy(d["o_hat"]))
    print(name, f"o_hat SNR {snr:.1f} dB")
    assert snr >= GATE_DB, snr
    for k, a, b in zip(("z", "z_p", "z_hat"), lat, lat3):
        assert torch.equal(a, b), k
    if c["lengths"]:   # per-utterance (ragged) semantics: nothing is written past an utterance's end
        o, _ = run(m, "f16s", spec, lengths, gs, gt, noise, c["tau"], ragged=True)
        for b, L in enumerate(c["lengths"]):
            assert float(o[b, 0, 256 * L:].abs().max()) == 0.0 if L < c["T"] else True


def test_rounding_points_match_the_emulation(model, synthetic_sd):
    """On vc_b1_t67 the GPU's SNR against the fp32 oracle is within 2 dB of the CPU emulation's: the kernels round
    where the contract says (an extra or a missing rounding moves the SNR by more)."""
    d, c = load("vc_b1_t67")
    spec, lengths, gs, gt, noise = O.synthetic_inputs(c["B"], c["T"], c["seed"], lengths=c["lengths"])
    o, _ = run(model, "f16s", spec, lengths, gs, gt, noise, c["tau"])
    ref = torch.from_numpy(d["o_hat"])
    with torch.no_grad():
        emu = H.generator_f16s(synthetic_sd, torch.from_numpy(d["z_hat"]) * torch.from_numpy(d["mask"]), gt)
    s_gpu, s_emu = H.snr_db(o, ref), H.snr_db(emu, ref)
    print(f"GPU {s_gpu:.2f} dB, emulation {s_emu:.2f} dB, GPU vs emulation {H.snr_db(o, emu):.1f} dB")
    assert abs(s_gpu - s_emu) <= 2.0, (s_gpu, s_emu)


def test_benched_config_snr(model, synthetic_sd):
    """32 x 10 s (T = 861), ragged, two full clips and a shorter one against the oracle run on each clip alone;
    nothing is written past a clip's end."""
    B, T = 32, 861
    lens = [T] * B
    lens[5], lens[17] = 640, 258
    spec, lengths, gs, gt, noise = O.synthetic_inputs(B, T, 861, lengths=lens)
    o, _ = run(model, "f16s", spec, lengths, gs, gt, noise, 0.3, ragged=True)
    assert o.shape == (B, 1, 256 * T)
    for b in (0, 31, 5):
        L = lens[b]
        with torch.no_grad():
            ro, _, _ = O.voice_conversion(synthetic_sd, spec[b:b + 1, :, :L].contiguous(), lengths[b:b + 1], gs[b:b + 1],
                                          gt[b:b + 1], noise[b:b + 1, :, :L].contiguous(), 0.3)
        snr = H.snr_db(o[b, 0, : 256 * L], ro[0, 0])
        print(b, f"{snr:.1f} dB")
        assert snr >= GATE_DB, (b, snr)
        if L < T:
            assert float(o[b, 0, 256 * L:].abs().max()) == 0.0


def test_bit_identities(model):
    """Ragged batch items equal their solo calls; a graph replay equals the direct launch; a small call is the same
    with the concurrent-branch schedule on and off."""
    nat = model.native
    spec, lengths, gs, gt, noise = O.synthetic_inputs(3, 70, 5, lengths=[70, 41, 64])
    o, lat = run(model, "f16s", spec, lengths, gs, gt, noise, 0.3, ragged=True)
    for b in range(3):
        L = int(lengths[b])
        ob, latb = run(model, "f16s", spec[b:b + 1, :, :L].contiguous(), lengths[b:b + 1], gs[b:b + 1], gt[b:b + 1],
                       noise[b:b + 1, :, :L].contiguous(), 0.3, ragged=True)
        assert torch.equal(ob[0, 0], o[b, 0, : 256 * L]), b
        assert torch.equal(latb[2][0], lat[2][b, :, :L]), b

    B, L = 2, 22050   # 86 frames per clip: B * T <= 512, the concurrent-branch schedule
    wav = (torch.rand(B, L, generator=torch.Generator().manual_seed(3)) - 0.5).cuda()
    wlen = torch.tensor([L, L - 3000], dtype=torch.int64, device="cuda")
    g1 = 0.1 * torch.randn(B, 256, generator=torch.Generator().manual_seed(4)).cuda()
    g2 = 0.1 * torch.randn(B, 256, generator=torch.Generator().manual_seed(5)).cuda()
    out = torch.empty(B, (L // 256) * 256, device="cuda")

    def call():
        o, _ = nat.convert_waveform(wav, wlen, g1, g2, tau=0.3, seed=7, out=out)
        torch.cuda.synchronize()
        return o.clone()

    nat.set_precision("f16s")
    try:
        nat.set_option("graph", 0)
        direct = call()
        nat.set_option("branches", 0)
        seq = call()
        nat.set_option("branches", 1)
        nat.set_option("graph", 1)
        before = nat.graph_replays
        replayed = [call() for _ in range(3)][-1]
        assert nat.graph_replays - before >= 1
        assert torch.equal(direct, seq) and torch.equal(direct, replayed)
    finally:
        nat.set_option("graph", 1)
        nat.set_option("branches", 1)
        nat.set_precision(model.precision)


def _profile(model, mode, spec, lengths, gs, gt, noise):
    nat = model.native
    nat.set_precision(mode)
    nat.profile_enable(True)
    try:
        model.voice_conversion(spec.cuda(), lengths.cuda(), gs.cuda(), gt.cuda(), tau=0.3, noise=noise.cuda(), ragged=True)
        torch.cuda.synchronize()
        return nat.profile_detail()
    finally:
        nat.profile_enable(False)
        nat.set_precision(model.precision)


def test_launches(model):
    """Every generator conv launches an fp16-storage variant (H<TN>c<Cin>k<k>d<d>), no pair kernel appears, and the
    other tensor-core launches are those of f16x3."""
    spec, lengths, gs, gt, noise = O.synthetic_inputs(3, 300, 9, lengths=[300, 211, 37])   # > 512 frames: sequential MRF
    rows16 = _profile(model, "f16s", spec, lengths, gs, gt, noise)
    rows3 = _profile(model, "f16x3", spec, lengths, gs, gt, noise)
    gen16 = [r[0] for r in rows16 if re.fullmatch(r"H\d+c\d+k\d+d\d+", r[0])]
    assert len(gen16) == 1 + 4 + 4 * 18, len(gen16)    # conv_pre, 4 upsamplers, 4 x 3 ResBlocks x 6 convs
    assert gen16[0] == "H128c192k7d1"
    assert all(r[0].startswith("H") for r in rows16 if r[4] == 1)   # every MRF conv
    assert not any(r[0].startswith("P") for r in rows16)
    assert any(r[0].startswith("P") for r in rows3)                  # this batch does fuse pairs in f16x3
    # the WaveNet stacks of enc_q and the flows (192 channels, k 5 and the 1x1 res/skip) are f16x3's launches
    other16 = [r[0] for r in rows16 if re.fullmatch(r"T\d+c\d+k\d+d\d+", r[0])]
    other3 = [r[0] for r in rows3 if re.fullmatch(r"T\d+c192k[15]d1", r[0])]
    assert other16 == other3 and len(other3) > 0


def test_workspace_is_about_half(model):
    nat = model.native
    try:
        nat.set_precision("f16x3")
        w3 = nat.lib.ovc_workspace_floats(nat.handle, 32, 861)
        nat.set_precision("f16s")
        w16 = nat.lib.ovc_workspace_floats(nat.handle, 32, 861)
    finally:
        nat.set_precision(model.precision)
    print(f"workspace 32 x 861: f16x3 {w3 * 4e-9:.2f} GB, f16s {w16 * 4e-9:.2f} GB")
    assert 0 < w16 <= 0.55 * w3


def test_tts_decode():
    from conftest import get_native_tts
    from oracle.golden import Golden
    tts = get_native_tts()
    d = Golden(os.path.join(GOLD, "tts_b1_t37.npz"))
    c = json.loads(str(d["meta"]))
    from oracle import tts_oracle as T
    tokens, lengths, sid, noise_w = T.synthetic_tts_inputs(c["B"], c["T"], c["seed"], c["lengths"])
    noise = torch.randn(c["B"], 192, 40 * c["T"] + 64, generator=torch.Generator().manual_seed(30_000 + c["seed"]))
    kw = dict(sid=sid, noise_scale=c["noise_scale"], length_scale=c["length_scale"], noise_scale_w=c["noise_scale_w"],
              sdp_ratio=c["sdp_ratio"], noise_w=noise_w, noise=noise)
    res = {}
    for mode in ("f16x3", "f16s"):
        tts.native.set_precision(mode)
        try:
            o, attn, y_mask, (z, _, _, _) = tts.infer(tokens, lengths, **kw)
            torch.cuda.synchronize()
        finally:
            tts.native.set_precision(tts.precision)
        res[mode] = (o.cpu(), attn.cpu(), y_mask.cpu(), z.cpu())
    o, attn, y_mask, z = res["f16s"]
    assert torch.equal(y_mask, res["f16x3"][2]) and torch.equal(attn, res["f16x3"][1])
    assert torch.equal(z, res["f16x3"][3])
    assert np.array_equal(attn[:, 0].sum(1).numpy(), d["w_ceil"])
    snr = H.snr_db(o, torch.from_numpy(d["o"]))
    print(f"tts_b1_t37 f16s o SNR {snr:.1f} dB")
    assert snr >= GATE_DB, snr


def test_debug_taps(model, synthetic_sd):
    d, c = load("vc_b1_t24")
    spec, lengths, gs, gt, noise = O.synthetic_inputs(c["B"], c["T"], c["seed"], lengths=c["lengths"])
    taps = {}
    with torch.no_grad():
        H.generator_f16s(synthetic_sd, torch.from_numpy(d["z_hat"]), gt, taps=taps)
    run(model, "f16s", spec, lengths, gs, gt, noise, c["tau"], debug=True)
    for i in range(4):
        name = f"dec.stage{i}"
        got = model.native.debug_fetch(name)
        assert got.shape == tuple(taps[name].shape), (name, got.shape)
        assert np.isfinite(got).all(), name
        print(name, f"{H.snr_db(torch.from_numpy(got), taps[name]):.1f} dB vs emulation")


def test_tone_color_converter_api(tmp_path, synthetic_sd):
    from openvoice_b200.api import ToneColorConverter
    cfg = tmp_path / "config.json"
    cfg.write_text(json.dumps(O.DEFAULT_HPARAMS))
    rng = np.random.default_rng(11)
    wavs = [(0.5 * (2 * rng.random(n, dtype=np.float32) - 1)).astype(np.float32) for n in (66150, 40000)]
    gen = torch.Generator().manual_seed(5)
    src = 0.1 * torch.randn(1, 256, 1, generator=gen)
    tgt = 0.1 * torch.randn(1, 256, 1, generator=gen)
    out = {}
    for mode in ("f16x3", "f16s"):
        conv = ToneColorConverter(str(cfg), device="cuda:0", enable_watermark=False, precision=mode)
        conv.model.load_state_dict(synthetic_sd)
        torch.manual_seed(321)
        out[mode] = conv.convert_batch(wavs, src, tgt, tau=0.3)
    for a, b in zip(out["f16s"], out["f16x3"]):
        assert a.shape == b.shape
        snr = H.snr_db(torch.from_numpy(a), torch.from_numpy(b))
        print(f"convert_batch f16s vs f16x3: {snr:.1f} dB")
        assert snr >= GATE_DB, snr
