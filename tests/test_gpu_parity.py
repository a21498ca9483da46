"""-m gpu: the CUDA path (through the C ABI) against the CPU oracle and the committed golden
vectors of the real reference.

Tolerance (north_star: "within a stated fp32 tolerance"): per tensor,
    max|cuda - ref| <= 1e-4 * rms(ref)
which is ~20-100x the reference's own fp32-vs-fp64 noise floor (8e-7 on latents of rms 0.4,
1.7e-7 on audio of rms 0.03; tests/golden/REPORT.json).  Both arithmetic paths are fp32 with
fp32 accumulation; they differ only in summation order.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import vc_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
REL = 1e-4


def rel_err(got, ref):
    ref = np.asarray(ref, dtype=np.float64)
    got = np.asarray(got, dtype=np.float64)
    rms = np.sqrt((ref ** 2).mean()) + 1e-30
    return float(np.abs(got - ref).max() / rms)


def run_native(native, spec, lengths, gs, gt, noise, tau, ragged=False, debug=False):
    native.native.debug_enable(debug)
    o, mask, lat = native.voice_conversion(spec.cuda(), lengths.cuda(), gs.cuda(), gt.cuda(), tau=tau,
                                           noise=None if noise is None else noise.cuda(), ragged=ragged)
    torch.cuda.synchronize()
    return o.cpu(), mask.cpu(), tuple(t.cpu() for t in lat)


def report_taps(native, sd, spec, lengths, gs, gt, noise, tau, zero_g=False):
    """Per-stage errors (debug taps) -- printed when a parity assertion fails."""
    taps = {}
    with torch.no_grad():
        O.voice_conversion(sd, spec, lengths, gs, gt, noise, tau, zero_g, taps=taps)
    lines = []
    for name in ["dec.pre", "dec.ups0", "dec.stage0", "dec.ups1", "dec.stage1", "dec.ups2", "dec.stage2",
                 "dec.ups3", "dec.stage3"]:
        try:
            got = native.native.debug_fetch(name)
            lines.append(f"{name}: rel_err={rel_err(got, taps[name].numpy()):.3e}")
        except Exception as e:  # noqa: BLE001
            lines.append(f"{name}: {e}")
    return "\n".join(lines)


@pytest.mark.parametrize("name", ["vc_b1_t24", "vc_b1_t67", "vc_b2_padded", "vc_b1_t24_tau0"])
def test_golden_reference_vectors(name, native, synthetic_sd):
    d = np.load(os.path.join(GOLD, name + ".npz"))
    c = json.loads(str(d["meta"]))
    spec, lengths, gs, gt, noise = O.synthetic_inputs(c["B"], c["T"], c["seed"], lengths=c["lengths"])
    o, mask, (z, zp, zh) = run_native(native, spec, lengths, gs, gt, noise, c["tau"], debug=True)
    errs = {k: rel_err(v.numpy(), d[g]) for k, v, g in
            (("z", z, "z"), ("z_p", zp, "z_p"), ("z_hat", zh, "z_hat"), ("o_hat", o, "o_hat"))}
    print(name, errs)
    if max(errs.values()) > REL:
        print(report_taps(native, synthetic_sd, spec, lengths, gs, gt, noise, c["tau"]))
    native.native.debug_enable(False)
    assert np.array_equal(mask.numpy(), d["mask"])
    for k, e in errs.items():
        assert e <= REL, (k, e, errs)


def test_golden_v2_zero_g(native_v2, synthetic_sd):
    d = np.load(os.path.join(GOLD, "vc_b1_t24_v2.npz"))
    c = json.loads(str(d["meta"]))
    spec, lengths, gs, gt, noise = O.synthetic_inputs(c["B"], c["T"], c["seed"], lengths=c["lengths"])
    o, _, (z, zp, zh) = run_native(native_v2, spec, lengths, gs, gt, noise, c["tau"])
    for got, key in ((z, "z"), (zp, "z_p"), (zh, "z_hat"), (o, "o_hat")):
        assert rel_err(got.numpy(), d[key]) <= REL, key


@pytest.mark.parametrize("B,T,lens", [(3, 150, [150, 97, 1]), (2, 131, [131, 130]), (1, 5, [5]), (4, 33, [33, 20, 12, 7])])
def test_oracle_padded_and_ragged(B, T, lens, native, synthetic_sd):
    """Ragged / odd sizes: padded-batch semantics vs the oracle, and per-utterance (convert)
    semantics vs the oracle's solo runs."""
    spec, lengths, gs, gt, noise = O.synthetic_inputs(B, T, 100 + T, lengths=lens)
    with torch.no_grad():
        ro, _, (rz, rzp, rzh) = O.voice_conversion(synthetic_sd, spec, lengths, gs, gt, noise, 0.3)
        qo, _, (qz, qzp, qzh) = O.voice_conversion_ragged(synthetic_sd, spec, lengths, gs, gt, noise, 0.3)
    o, _, (z, zp, zh) = run_native(native, spec, lengths, gs, gt, noise, 0.3, ragged=False)
    for got, ref, k in ((z, rz, "z"), (zp, rzp, "z_p"), (zh, rzh, "z_hat"), (o, ro, "o_hat")):
        assert rel_err(got.numpy(), ref.numpy()) <= REL, ("padded", k)
    o, _, (z, zp, zh) = run_native(native, spec, lengths, gs, gt, noise, 0.3, ragged=True)
    for got, ref, k in ((z, qz, "z"), (zp, qzp, "z_p"), (zh, qzh, "z_hat"), (o, qo, "o_hat")):
        assert rel_err(got.numpy(), ref.numpy()) <= REL, ("ragged", k)
    for b, L in enumerate(lens):   # nothing leaks past an utterance's end
        assert float(o[b, 0, 256 * L:].abs().max()) == 0.0 if L < T else True


def test_batch_items_are_independent(native):
    """Solo-vs-batched equality (bitwise): item b of a ragged batch == the same item alone."""
    spec, lengths, gs, gt, noise = O.synthetic_inputs(3, 70, 5, lengths=[70, 41, 64])
    o, _, lat = run_native(native, spec, lengths, gs, gt, noise, 0.3, ragged=True)
    for b in range(3):
        L = int(lengths[b])
        ob, _, latb = run_native(native, spec[b:b + 1, :, :L].contiguous(), lengths[b:b + 1], gs[b:b + 1], gt[b:b + 1],
                                 noise[b:b + 1, :, :L].contiguous(), 0.3, ragged=True)
        assert torch.equal(ob[0, 0], o[b, 0, : 256 * L])
        assert torch.equal(latb[2][0], lat[2][b, :, :L])


def test_graph_replay_is_bit_identical(native):
    """OVC_OPT_GRAPH: a repeated (shapes, buffers) call is captured on its second sighting and replayed afterwards.
    Replays must equal the directly launched sequence bit for bit, follow a new Philox seed, and stop when the
    option is switched off."""
    nat = native.native
    nat.set_precision("f16x3")       # the default mode: tensor-core kernels, PDL on the WaveNet stacks, concurrent branches
    B, L = 2, 22050
    wav = (torch.rand(B, L, generator=torch.Generator().manual_seed(3)) - 0.5).cuda()
    wlen = torch.tensor([L, L - 3000], dtype=torch.int64, device="cuda")
    g1 = 0.1 * torch.randn(B, 256, generator=torch.Generator().manual_seed(4)).cuda()
    g2 = 0.1 * torch.randn(B, 256, generator=torch.Generator().manual_seed(5)).cuda()
    out = torch.empty(B, (L // 256) * 256, device="cuda")

    def call(seed):
        o, _ = nat.convert_waveform(wav, wlen, g1, g2, tau=0.3, seed=seed, out=out)
        torch.cuda.synchronize()
        return o.clone()

    nat.set_option("graph", 0)
    ref7, ref9 = call(7), call(9)
    assert not torch.equal(ref7, ref9)
    nat.set_option("graph", 1)
    before = nat.graph_replays
    a = call(7)                      # first sighting: direct
    b = call(7)                      # second: captured, then launched as a graph
    c = call(9)                      # replay with another seed
    d = call(7)
    assert nat.graph_replays - before >= 2, "the repeated call was not served from a graph"
    assert torch.equal(a, ref7) and torch.equal(b, ref7) and torch.equal(d, ref7)
    assert torch.equal(c, ref9)
    launches = nat.last_launch_count
    nat.set_option("graph", 0)
    e = call(9)
    assert torch.equal(e, ref9) and nat.last_launch_count == launches
    # the concurrent-branch schedule of small calls (three streams, a third of the SMs per kernel) keeps the MRF
    # accumulation order: same bits as the sequential schedule, directly launched and replayed
    nat.set_option("branches", 0)
    seq = call(9)
    nat.set_option("graph", 1)
    seq_g = [call(9) for _ in range(3)][-1]
    nat.set_option("branches", 1)
    assert torch.equal(seq, ref9) and torch.equal(seq_g, ref9)


def test_fused_conv_pair_equals_two_launches(native):
    """OVC_OPT_PAIR: the fused ResBlock conv-pair kernel of the C = 32 stage (intermediate activation kept in shared memory)
    performs the same arithmetic in the same order as two conv launches: bit-identical audio on a ragged batch whose
    lengths put tile boundaries, utterance ends and the 118 / 126-step tiling in different places; both tensor-core modes.
    The batch is small enough for the concurrent-branch schedule, which never fuses: the sequential one is forced."""
    import re
    nat = native.native
    spec, lengths, gs, gt, noise = O.synthetic_inputs(3, 131, 17, lengths=[131, 64, 7])
    outs = {}
    nat.set_option("branches", 0)
    try:
        for mode in ("f16x3", "f16"):
            nat.set_precision(mode)
            for pair in (0, 1):
                nat.set_option("pair", pair)
                o, _, _ = run_native(native, spec, lengths, gs, gt, noise, 0.3, ragged=True)
                outs[(mode, pair)] = o
            assert torch.equal(outs[(mode, 0)], outs[(mode, 1)]), mode
        pairs = {}
        for pair in (0, 1):                       # what ran: the profile names of the pair kernel, P<C>k<k>d<d>
            nat.set_option("pair", pair)
            nat.profile_enable(True)
            try:
                run_native(native, spec, lengths, gs, gt, noise, 0.3, ragged=True)
                pairs[pair] = {int(m[1]) for m in (re.fullmatch(r"P(\d+)k\d+d\d+", r[0]) for r in nat.profile_detail()) if m}
            finally:
                nat.profile_enable(False)
        assert 32 in pairs[1] and not pairs[0], pairs
    finally:
        nat.set_option("branches", 1)
        nat.set_precision("f16x3")
        nat.set_option("pair", 1)


def test_flow_roundtrip_property_full_size(native):
    """Size-independent property at the BASELINE size (10 s clips, T=861): with g_src == g_tgt the
    reverse flow undoes the forward flow, so z_hat == z up to rounding."""
    B, T = 4, 861
    spec, lengths, gs, gt, noise = O.synthetic_inputs(B, T, 77)
    o, _, (z, zp, zh) = run_native(native, spec, lengths, gs, gs, noise, 0.3)
    assert rel_err(zh.numpy(), z.numpy()) < 2e-5
    assert float((zp - z).abs().max()) > 1e-2          # the flow is not a no-op
    assert torch.isfinite(o).all() and float(o.abs().max()) <= 1.0
    assert o.shape == (B, 1, 256 * T)


def _oracle_solo(sd, spec, lengths, gs, gt, noise, b, tau, zero_g=False):
    L = int(lengths[b])
    with torch.no_grad():
        return O.voice_conversion(sd, spec[b:b + 1, :, :L].contiguous(), lengths[b:b + 1], gs[b:b + 1], gt[b:b + 1],
                                  noise[b:b + 1, :, :L].contiguous(), tau, zero_g)


def test_benched_config_vs_oracle(native, synthetic_sd):
    """The BENCHED configuration (BASELINE configs[1]: 32 x 10 s clips, T = 861, ragged = convert semantics) against
    the CPU oracle: two full-length clips and one shorter clip taken out of the batch of 32, every tensor of
    voice_conversion (models.py:492-499) within the stated 1e-4 * rms, in both arithmetic modes."""
    B, T = 32, 861
    lens = [T] * B
    lens[5], lens[17] = 640, 258
    spec, lengths, gs, gt, noise = O.synthetic_inputs(B, T, 861, lengths=lens)
    o, mask, (z, zp, zh) = run_native(native, spec, lengths, gs, gt, noise, 0.3, ragged=True)
    assert o.shape == (B, 1, 256 * T)
    worst = {}
    for b in (0, 31, 5):
        L = lens[b]
        ro, _, (rz, rzp, rzh) = _oracle_solo(synthetic_sd, spec, lengths, gs, gt, noise, b, 0.3)
        for k, got, ref in (("z", z[b, :, :L], rz[0]), ("z_p", zp[b, :, :L], rzp[0]), ("z_hat", zh[b, :, :L], rzh[0]),
                            ("o_hat", o[b, 0, : 256 * L], ro[0, 0])):
            e = rel_err(got.numpy(), ref.numpy())
            worst[k] = max(worst.get(k, 0.0), e)
            assert e <= REL, (b, k, e)
        assert float(o[b, 0, 256 * L:].abs().max()) == 0.0 if L < T else True
    print("benched-config parity (max over 3 clips):", worst)


def test_thirty_second_clip_vs_oracle(native, synthetic_sd):
    """One 30 s clip (T = 2583, BASELINE configs[4]'s longest) against the oracle."""
    T = 2583
    spec, lengths, gs, gt, noise = O.synthetic_inputs(1, T, 2583)
    o, _, (z, zp, zh) = run_native(native, spec, lengths, gs, gt, noise, 0.3, ragged=True)
    ro, _, (rz, rzp, rzh) = _oracle_solo(synthetic_sd, spec, lengths, gs, gt, noise, 0, 0.3)
    for k, got, ref in (("z", z, rz), ("z_p", zp, rzp), ("z_hat", zh, rzh), ("o_hat", o, ro)):
        assert rel_err(got.numpy(), ref.numpy()) <= REL, k


def test_v2_zero_g_full_size_vs_oracle(native_v2, synthetic_sd):
    """V2 converter semantics (zero_g, models.py:495,498) at T = 861 (BASELINE configs[3] clip size), default mode."""
    T = 861
    spec, lengths, gs, gt, noise = O.synthetic_inputs(2, T, 8612, lengths=[T, 700])
    o, _, (z, zp, zh) = run_native(native_v2, spec, lengths, gs, gt, noise, 0.3, ragged=True)
    for b, L in ((0, T), (1, 700)):
        ro, _, (rz, rzp, rzh) = _oracle_solo(synthetic_sd, spec, lengths, gs, gt, noise, b, 0.3, zero_g=True)
        for k, got, ref in (("z", z[b, :, :L], rz[0]), ("z_p", zp[b, :, :L], rzp[0]), ("z_hat", zh[b, :, :L], rzh[0]),
                            ("o_hat", o[b, 0, : 256 * L], ro[0, 0])):
            assert rel_err(got.numpy(), ref.numpy()) <= REL, (b, k)


def test_in_kernel_noise_statistics(native):
    """noise=None draws Philox normals in-kernel: (z - m)/(tau*exp(logs)) must look N(0,1) and be
    reproducible from the seed.  tau=0 run gives m; a second tau gives the scaled noise."""
    B, T = 2, 400
    spec, lengths, gs, gt, _ = O.synthetic_inputs(B, T, 9)
    args = (spec.cuda(), lengths.cuda(), gs.cuda(), gt.cuda())
    m = native.voice_conversion(*args, tau=0.0, noise=torch.zeros(B, 192, T).cuda())[2][0]
    ones = native.voice_conversion(*args, tau=1.0, noise=torch.ones(B, 192, T).cuda())[2][0]
    scale = (ones - m)                                   # exp(logs)
    z1 = native.voice_conversion(*args, tau=1.0, seed=1234)[2][0]
    z2 = native.voice_conversion(*args, tau=1.0, seed=1234)[2][0]
    z3 = native.voice_conversion(*args, tau=1.0, seed=99)[2][0]
    assert torch.equal(z1, z2) and not torch.equal(z1, z3)
    eps = ((z1 - m) / scale).flatten().double().cpu()
    assert abs(float(eps.mean())) < 0.02 and abs(float(eps.std()) - 1.0) < 0.02
    assert abs(float((eps ** 3).mean())) < 0.05 and abs(float((eps ** 4).mean()) - 3.0) < 0.15


def test_single_pass_f16_mode_has_its_own_gate(synthetic_sd):
    """precision="f16" = one fp16 pass per conv on the tensor cores: 11-bit operands, the precision class the reference
    itself runs on a GPU (cuDNN allow_tf32 defaults to True).  Stated gate for this mode: waveform SNR >= 30 dB against
    the fp32 oracle and latents within 2e-2 * rms; the default modes are held to 1e-4 * rms elsewhere in this file."""
    from conftest import get_native
    m = get_native(False)
    spec, lengths, gs, gt, noise = O.synthetic_inputs(2, 90, 21, lengths=[90, 57])
    with torch.no_grad():
        ro, _, (rz, rzp, rzh) = O.voice_conversion(synthetic_sd, spec, lengths, gs, gt, noise, 0.3)
    m.native.set_precision("f16")
    try:
        o, _, (z, zp, zh) = run_native(m, spec, lengths, gs, gt, noise, 0.3)
    finally:
        m.native.set_precision(m.precision)
    err = (o - ro).double()
    snr = 10 * np.log10(float(ro.double().pow(2).mean() / err.pow(2).mean()))
    print("f16 single-pass SNR dB:", snr, "z_hat rel", rel_err(zh.numpy(), rzh.numpy()))
    assert snr >= 30.0
    assert rel_err(zh.numpy(), rzh.numpy()) <= 2e-2


def test_reference_encoder_kernels(synthetic_sd):
    """ovc_reference_encoder (extract_se's ReferenceEncoder, row f2) vs the real reference's output (golden) and
    through the reference-shaped ``model.ref_enc(spec.transpose(1, 2))`` call."""
    from conftest import get_native
    m = get_native(False)
    d = np.load(os.path.join(GOLD, "ref_enc.npz"))
    spec = O.synthetic_inputs(2, 140, 7)[0]
    g = m.native.reference_encoder(spec.cuda().contiguous())
    assert g.shape == (2, 256)
    assert rel_err(g.cpu().numpy(), d["g"]) <= REL
    g2 = m.ref_enc(spec.transpose(1, 2))
    assert torch.equal(g2, g)
    one = m.native.reference_encoder(spec[1:2].cuda().contiguous())     # batch items are independent
    assert torch.equal(one[0], g[1])
    for T in (64, 65, 257):                                              # odd sizes through the stride-2 stack
        sp = O.synthetic_inputs(1, T, 50 + T)[0]
        with torch.no_grad():
            ref = O.reference_encoder(synthetic_sd, sp.transpose(1, 2))
        assert rel_err(m.native.reference_encoder(sp.cuda().contiguous()).cpu().numpy(), ref.numpy()) <= REL, T


def test_spectrogram_kernel(native):
    """ovc_spectrogram vs the reference's spectrogram_torch output (golden) and vs the oracle on a
    ragged batch (reflect padding at each item's own end)."""
    d = np.load(os.path.join(GOLD, "convert_wave.npz"))
    L = int(d["L"])
    rng = np.random.default_rng(1000)
    wav = (0.5 * (2 * rng.random(L, dtype=np.float32) - 1)).astype(np.float32)
    spec, frames = native.native.spectrogram(torch.from_numpy(wav)[None].cuda(), torch.tensor([L]).cuda())
    assert int(frames[0]) == L // 256 and spec.shape == (1, 513, L // 256)
    assert rel_err(spec.cpu().numpy(), d["spec"]) < 2e-5
    lens = [L, 385, 256 * 9 + 255, 256 * 17]
    batch = torch.zeros(len(lens), L)
    for b, n in enumerate(lens):
        batch[b, :n] = torch.from_numpy(wav[:n]) * (1 + b)
    spec, frames = native.native.spectrogram(batch.cuda(), torch.tensor(lens).cuda())
    assert frames.tolist() == [n // 256 for n in lens]
    for b, n in enumerate(lens):
        ref = O.spectrogram(batch[b: b + 1, :n])
        got = spec[b, :, : n // 256].cpu()
        assert rel_err(got.numpy(), ref[0].numpy()) < 2e-5, b
        assert float(spec[b, :, n // 256:].abs().max()) == 0.0 if n // 256 < L // 256 else True


def test_full_size_batch_properties(tmp_path, synthetic_sd):
    """BASELINE-size workload (32 x 10 s clips) through the public API: finite, in [-1, 1], right lengths;
    the same torch seed reproduces the batch bit for bit; an item of the batch equals its solo conversion
    (tau = 0 so no noise is involved); ragged tails are not touched."""
    from openvoice_b200.api import ToneColorConverter
    cfg = tmp_path / "config.json"
    cfg.write_text(json.dumps(O.DEFAULT_HPARAMS))
    conv = ToneColorConverter(str(cfg), device="cuda:0", enable_watermark=False)
    conv.model.load_state_dict(synthetic_sd)
    rng = np.random.default_rng(7)
    lens = [220500] * 30 + [220500 - 4321, 66150]
    wavs = [(0.5 * (2 * rng.random(n, dtype=np.float32) - 1)).astype(np.float32) for n in lens]
    gen = torch.Generator().manual_seed(5)
    src = 0.1 * torch.randn(1, 256, 1, generator=gen)
    tgt = 0.1 * torch.randn(1, 256, 1, generator=gen)
    torch.manual_seed(123)
    a = conv.convert_batch(wavs, src, tgt, tau=0.3, max_batch=32)
    torch.manual_seed(123)
    b = conv.convert_batch(wavs, src, tgt, tau=0.3, max_batch=32)
    for x, y, n in zip(a, b, lens):
        assert x.shape == (256 * (n // 256),) and np.isfinite(x).all() and np.abs(x).max() <= 1.0
        assert np.array_equal(x, y)
    c = conv.convert_batch(wavs, src, tgt, tau=0.0, max_batch=32)
    for i in (0, 30, 31):
        assert np.array_equal(conv.convert(wavs[i], src, tgt, tau=0.0), c[i])
    torch.manual_seed(124)
    d = conv.convert_batch(wavs[:2], src, tgt, tau=0.3)
    assert not np.array_equal(d[0], a[0])            # a different seed draws different noise


def test_one_utterance_per_stream_equals_solo(tmp_path, synthetic_sd):
    """convert_concurrent (replica + CUDA stream per in-flight request) returns exactly the solo conversions."""
    from openvoice_b200.api import ToneColorConverter
    cfg = tmp_path / "config.json"
    cfg.write_text(json.dumps(O.DEFAULT_HPARAMS))
    conv = ToneColorConverter(str(cfg), device="cuda:0", enable_watermark=False)
    conv.model.load_state_dict(synthetic_sd)
    rng = np.random.default_rng(3)
    wavs = [(0.5 * (2 * rng.random(n, dtype=np.float32) - 1)).astype(np.float32)
            for n in (22050, 30000, 66150, 256 * 7 + 5, 44100, 22050 * 2, 51200, 9999, 70000, 12345, 33333)]
    gen = torch.Generator().manual_seed(4)
    src = 0.1 * torch.randn(1, 256, 1, generator=gen)
    tgt = 0.1 * torch.randn(1, 256, 1, generator=gen)
    res = conv.convert_concurrent(wavs, src, tgt, tau=0.0, streams=3)
    assert len(res) == len(wavs)
    for w, r in zip(wavs, res):
        assert np.array_equal(r, conv.convert(w, src, tgt, tau=0.0))


def test_time_tiled_long_clip_equals_whole_clip(tmp_path, synthetic_sd):
    """convert_long (row f4: windows + receptive-field halo, one ragged batch) reproduces convert on the whole
    clip: interiors do not see the window edges.  Both arithmetic modes; same explicit noise on both sides."""
    from openvoice_b200.api import ToneColorConverter
    cfg = tmp_path / "config.json"
    cfg.write_text(json.dumps(O.DEFAULT_HPARAMS))
    rng = np.random.default_rng(11)
    L = 22050 * 14 + 123
    wav = (0.5 * (2 * rng.random(L, dtype=np.float32) - 1)).astype(np.float32)
    T = L // 256
    gen = torch.Generator().manual_seed(8)
    src = 0.1 * torch.randn(1, 256, 1, generator=gen)
    tgt = 0.1 * torch.randn(1, 256, 1, generator=gen)
    noise = torch.randn(192, T, generator=gen)
    for precision in ("fp32", "f16x3"):
        conv = ToneColorConverter(str(cfg), device="cuda:0", enable_watermark=False, precision=precision)
        conv.model.load_state_dict(synthetic_sd)
        whole = conv.convert(wav, src, tgt, tau=0.3, noise=noise[None])
        tiled = conv.convert_long(wav, src, tgt, tau=0.3, noise=noise, window_frames=300)
        assert tiled.shape == whole.shape == (256 * T,)
        assert rel_err(tiled, whole) <= 2e-6, precision
        short = conv.convert_long(wav[: 256 * 90], src, tgt, tau=0.0, window_frames=2048)     # single window
        assert np.array_equal(short, conv.convert(wav[: 256 * 90], src, tgt, tau=0.0))


def test_streaming_equals_whole_clip(tmp_path, synthetic_sd):
    """Row f4, stateful streaming: audio pushed in irregular chunks through StreamingConverter (spectrogram frames, noise
    and audio tail carried between calls; window + 128-frame halo per call) gives the samples of convert on the whole
    clip, emits them incrementally, and keeps a bounded state."""
    from openvoice_b200.api import ToneColorConverter
    from openvoice_b200.streaming import StreamingConverter
    cfg = tmp_path / "config.json"
    cfg.write_text(json.dumps(O.DEFAULT_HPARAMS))
    rng = np.random.default_rng(21)
    L = 22050 * 9 + 77
    wav = (0.5 * (2 * rng.random(L, dtype=np.float32) - 1)).astype(np.float32)
    T = L // 256
    gen = torch.Generator().manual_seed(9)
    src = 0.1 * torch.randn(1, 256, 1, generator=gen)
    tgt = 0.1 * torch.randn(1, 256, 1, generator=gen)
    noise = torch.randn(192, T, generator=gen)
    conv = ToneColorConverter(str(cfg), device="cuda:0", enable_watermark=False)
    conv.model.load_state_dict(synthetic_sd)
    whole = conv.convert(wav, src, tgt, tau=0.3, noise=noise[None])
    for W, sizes in ((200, [100, 7000, 33, 66150, 12000, 256, 90001]), (64, [4096] * 60)):
        sc = StreamingConverter(conv, src, tgt, tau=0.3, window_frames=W, noise_fn=lambda a, b: noise[:, a:b])
        outs, pos, i, first_out_at, max_frames, max_samples = [], 0, 0, None, 0, 0
        while pos < L:
            n = min(sizes[i % len(sizes)], L - pos)
            got = sc.push(wav[pos: pos + n])
            pos += n
            i += 1
            if len(got) and first_out_at is None:
                first_out_at = pos
            outs.append(got)
            max_frames, max_samples = max(max_frames, sc.state_frames), max(max_samples, sc.state_samples)
        outs.append(sc.flush())
        stream = np.concatenate(outs)
        assert stream.shape == whole.shape == (256 * T,)
        assert rel_err(stream, whole) <= 2e-6, W
        # output starts once window + halo (+ the STFT support) has arrived, long before the end of the clip
        assert first_out_at is not None and first_out_at <= 256 * (W + 128 + 4) + max(sizes)
        # state: at most the two halos, one window and the frames of the largest chunk; audio tail of a few frames
        assert max_frames <= W + 2 * 128 + max(sizes) // 256 + 8, max_frames
        assert max_samples <= max(sizes) + 2048, max_samples
    # a stream shorter than one window + halo: nothing comes out before flush, and flush returns the whole clip
    Ls = 22050 + 5
    short = conv.convert(wav[:Ls], src, tgt, tau=0.3, noise=noise[None, :, : Ls // 256])
    sc = StreamingConverter(conv, src, tgt, tau=0.3, window_frames=200, noise_fn=lambda a, b: noise[:, a:b])
    early = [sc.push(wav[p: min(Ls, p + 5000)]) for p in range(0, Ls, 5000)]
    assert sum(len(e) for e in early) == 0
    tail = sc.flush()
    assert tail.shape == short.shape and rel_err(tail, short) <= 2e-6


def test_pipelined_single_gpu_api_equals_convert(tmp_path, synthetic_sd):
    """openvoice_b200.distributed.convert_sharded_async on one GPU (what bench.py's end-to-end leg calls): three calls
    back to back with one in flight -- upload slots alternate, downloads run on a side stream, graphs are captured and
    replayed -- return, per utterance, exactly what ToneColorConverter.convert returns (tau = 0: no random draw)."""
    from openvoice_b200 import distributed as D
    from openvoice_b200.api import ToneColorConverter
    cfg = tmp_path / "config.json"
    cfg.write_text(json.dumps(O.DEFAULT_HPARAMS))
    conv = ToneColorConverter(str(cfg), device="cuda:0", enable_watermark=False)
    conv.model.load_state_dict(synthetic_sd)
    rng = np.random.default_rng(31)
    waves = [(0.5 * (2 * rng.random(n, dtype=np.float32) - 1)).astype(np.float32) for n in (22050, 9000, 30011, 4096)]
    gen = torch.Generator().manual_seed(3)
    src = [0.1 * torch.randn(1, 256, 1, generator=gen) for _ in waves]
    tgt = [0.1 * torch.randn(1, 256, 1, generator=gen) for _ in waves]
    solo = [conv.convert(w, s, t, tau=0.0) for w, s, t in zip(waves, src, tgt)]
    jobs = []
    for _ in range(5):
        jobs.append(D.convert_sharded_async(conv, waves, src, tgt, tau=0.0, copy=True))
        if len(jobs) >= 2:
            res = jobs[-2].result()
            assert len(res) == len(waves)
            for a, b in zip(res, solo):
                assert a.shape == b.shape and np.array_equal(a, b)
    last = jobs[-1].result()
    for a, b in zip(last, solo):
        assert np.array_equal(a, b)
    assert conv.model.native.graph_replays > 0


def test_api_convert_matches_reference_golden(tmp_path, synthetic_sd):
    """ToneColorConverter.convert end to end (waveform -> spectrogram -> VC -> samples) against
    the real reference's convert() output."""
    from openvoice_b200.api import ToneColorConverter
    d = np.load(os.path.join(GOLD, "convert_wave.npz"))
    L = int(d["L"])
    rng = np.random.default_rng(1000)
    wav = (0.5 * (2 * rng.random(L, dtype=np.float32) - 1)).astype(np.float32)
    gen = torch.Generator().manual_seed(2000)
    src = 0.1 * torch.randn(1, 256, 1, generator=gen)
    tgt = 0.1 * torch.randn(1, 256, 1, generator=gen)
    cfg = tmp_path / "config.json"
    cfg.write_text(json.dumps(O.DEFAULT_HPARAMS))
    ckpt = tmp_path / "checkpoint.pth"
    torch.save({"model": synthetic_sd}, ckpt)
    conv = ToneColorConverter(str(cfg), device="cuda:0", enable_watermark=False)
    conv.load_ckpt(str(ckpt))
    wav_path = tmp_path / "a.npy"
    np.save(wav_path, wav)
    a0 = conv.convert(str(wav_path), src, tgt, tau=0.0)
    assert a0.dtype == np.float32 and a0.shape == d["audio_tau0"].shape
    assert rel_err(a0, d["audio_tau0"]) <= 2 * REL
    noise = torch.randn(1, 192, L // 256, generator=torch.Generator().manual_seed(4000))
    a1 = conv.convert(wav, src, tgt, tau=0.3, noise=noise)
    assert rel_err(a1, d["audio_tau03"]) <= 2 * REL
    out = tmp_path / "o.npy"
    assert conv.convert(str(wav_path), src, tgt, output_path=str(out), tau=0.0) is None
    assert np.array_equal(np.load(out), a0)
    # batch API: each item equals its solo conversion
    wavs = [wav, wav[: 256 * 11 + 3], wav[: 256 * 20]]
    res = conv.convert_batch(wavs, src, tgt, tau=0.0)
    assert np.array_equal(res[0], a0)
    for w, r in zip(wavs[1:], res[1:]):
        solo = conv.convert(w, src, tgt, tau=0.0)
        assert r.shape == (256 * (len(w) // 256),) and np.array_equal(r, solo)
    # speaker-embedding extraction against the reference's ReferenceEncoder
    se = conv.extract_se([wav])
    assert se.shape == (1, 256, 1)
    with torch.no_grad():
        g = O.reference_encoder(synthetic_sd, O.spectrogram(torch.from_numpy(wav)[None]).transpose(1, 2))
    assert rel_err(se.cpu().numpy()[0, :, 0], g.numpy()[0]) <= REL
