#!/usr/bin/env python
"""Per-kernel-variant report of one convert_batch call, from CUDA events around every conv launch
(ovc_profile_detail): launches, ms, share of the conv time, algorithmic TFLOP/s and GB/s.

  python tools/layer_report.py [--batch 32] [--secs 10] [--json out.json]
"""
import argparse
import collections
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--secs", type=float, default=10.0)
    ap.add_argument("--json", default=None)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "f16x3", "f16", "f16s"])
    ap.add_argument("--wide-variant", type=int, default=None)
    ap.add_argument("--pdl", type=int, default=None)
    ap.add_argument("--pair", type=int, default=None)
    ap.add_argument("--reps", type=int, default=1, help="profiled calls (per-variant times are averaged)")
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle import vc_oracle as O
    from openvoice_b200.api import ToneColorConverter

    with tempfile.TemporaryDirectory() as td:
        cfg = os.path.join(td, "config.json")
        json.dump(O.DEFAULT_HPARAMS, open(cfg, "w"))
        conv = ToneColorConverter(cfg, device="cuda:0", enable_watermark=False)
    conv.model.load_state_dict(O.synthetic_state_dict(1234))
    B, L = args.batch, int(round(args.secs * 22050))
    wav = (torch.rand(B, L, generator=torch.Generator().manual_seed(0)) - 0.5).cuda()
    wlen = torch.full((B,), L, dtype=torch.int64, device="cuda")
    g = 0.1 * torch.randn(B, 256, generator=torch.Generator().manual_seed(1)).cuda()
    nat = conv.model.native
    nat.set_precision(args.precision)
    if args.wide_variant is not None:
        nat.set_option("wide_variant", args.wide_variant)
    if args.pdl is not None:
        nat.set_option("pdl", args.pdl)
    if args.pair is not None:
        nat.set_option("pair", args.pair)
    nat.set_option("graph", 0)
    for _ in range(2):
        nat.convert_waveform(wav, wlen, g, g, tau=0.3, seed=1)
    torch.cuda.synchronize()
    nat.profile_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    nat.convert_waveform(wav, wlen, g, g, tau=0.3, seed=2)
    e1.record()
    torch.cuda.synchronize()
    rows = nat.profile_detail()
    nat.profile_read()
    nat.profile_enable(False)
    agg = collections.OrderedDict()
    for name, ms, fl, by, fam in rows:
        a = agg.setdefault(name, [0, 0.0, 0.0, 0.0])
        a[0] += 1; a[1] += ms; a[2] += fl; a[3] += by
    tot = sum(a[1] for a in agg.values())
    step_ms = e0.elapsed_time(e1)
    print(f"batch {B} x {args.secs:g} s: call {step_ms:.2f} ms (with event overhead), conv kernels {tot:.2f} ms, "
          f"{sum(a[2] for a in agg.values()) / tot / 1e9:.1f} TFLOP/s over convs")
    print(f"{'variant':12s} {'n':>4s} {'ms':>9s} {'share':>6s} {'TFLOP/s':>8s} {'GB/s(T2)':>9s}")
    out = []
    for name, (n, ms, fl, by) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print(f"{name:12s} {n:4d} {ms:9.3f} {100 * ms / tot:5.1f}% {fl / ms / 1e9:8.1f} {by / ms / 1e6:9.0f}")
        out.append(dict(variant=name, launches=n, ms=ms, share=ms / tot, tflops=fl / ms / 1e9, gbs=by / ms / 1e6))
    if args.json:
        json.dump(dict(batch=B, secs=args.secs, call_ms=step_ms, conv_ms=tot, variants=out), open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
