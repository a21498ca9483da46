#!/usr/bin/env python
"""Same-box A/B of the tuning switches (ovc_set_option): whole-call device time of convert_waveform, CUDA events,
settings interleaved round-robin so that clock / thermal drift hits all of them alike.

  python tools/ab_bench.py --batch 32 --secs 10 --rounds 4 --settings "pdl=0;pdl=1;pdl=2"
  python tools/ab_bench.py --settings "precision=f16x3;precision=f16;precision=f16s"   (modes alternate in one process)

A setting without precision= runs in --precision.
"""
import argparse
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
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--calls", type=int, default=3, help="timed calls per setting per round")
    ap.add_argument("--precision", default="f16x3")
    ap.add_argument("--settings", default="pdl=0;pdl=1;pdl=2")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle import vc_oracle as O
    from openvoice_b200.api import ToneColorConverter

    with tempfile.TemporaryDirectory() as td:
        cfg = os.path.join(td, "config.json")
        json.dump(O.DEFAULT_HPARAMS, open(cfg, "w"))
        conv = ToneColorConverter(cfg, device="cuda:0", enable_watermark=False, precision=args.precision)
    conv.model.load_state_dict(O.synthetic_state_dict(1234))
    nat = conv.model.native
    B, L = args.batch, int(round(args.secs * 22050))
    wav = (torch.rand(B, L, generator=torch.Generator().manual_seed(0)) - 0.5).cuda()
    wlen = torch.full((B,), L, dtype=torch.int64, device="cuda")
    g = 0.1 * torch.randn(B, 256, generator=torch.Generator().manual_seed(1)).cuda()
    out = torch.empty(B, (L // 256) * 256, device="cuda")
    fr = torch.empty(B, dtype=torch.int64, device="cuda")
    def value(k, v):
        return v if k == "precision" else int(v)

    settings = [dict((kv.split("=")[0], value(*kv.split("="))) for kv in s.split(",")) for s in args.settings.split(";")]
    times = [[] for _ in settings]

    def apply(st):
        nat.set_precision(st.get("precision", args.precision))
        for k in ("graph", "pdl", "wide_variant", "branches", "pair"):
            if k in st:
                nat.set_option(k, st[k])
        if "graph" not in st:
            nat.set_option("graph", 0)

    for st in settings:            # warm-up, also captures graphs where enabled
        apply(st)
        for i in range(3):
            nat.convert_waveform(wav, wlen, g, g, tau=0.3, seed=i, out=out, frames_out=fr)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for si, st in enumerate(settings):
            apply(st)
            nat.convert_waveform(wav, wlen, g, g, tau=0.3, seed=5, out=out, frames_out=fr)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.calls):
                nat.convert_waveform(wav, wlen, g, g, tau=0.3, seed=10 + i, out=out, frames_out=fr)
            e1.record()
            torch.cuda.synchronize()
            times[si].append(e0.elapsed_time(e1) / args.calls)
    res = []
    for st, ts in zip(settings, times):
        res.append({"setting": st, "ms_median": float(np.median(ts)), "ms_min": float(np.min(ts)), "ms_max": float(np.max(ts)),
                    "ms_all": ts})
        print(f"B={B} x {args.secs:g}s  {st}:  median {np.median(ts):8.3f} ms   min {np.min(ts):8.3f} ms   "
              f"max {np.max(ts):8.3f} ms", flush=True)
    if args.json:
        json.dump({"batch": B, "secs": args.secs, "precision": args.precision, "results": res}, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
