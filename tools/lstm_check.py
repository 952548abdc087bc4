"""Encoder check + timing (run on a GPU).

    python tools/lstm_check.py --config cfg2 --B 32 --T 124 --out enc_a.npy
    python tools/lstm_check.py ... --out enc_b.npy --compare enc_a.npy

Feeds seeded random features (not audio: the encoder is what is under test), checks the encoder output and
final state against the CPU oracle on the first `--oracle-rows` utterances (full size would take minutes) and,
with --compare, against a saved run (for example of another build of the library).  Prints encode ms (CUDA events, 10 runs).
Test infrastructure (imports oracle/).
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from libreasr_b200 import synth  # noqa: E402
from libreasr_b200.engine import Engine, EngineConfig  # noqa: E402
from oracle import rnnt_oracle as O  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--B", type=int, default=32)
    ap.add_argument("--T", type=int, default=124)
    ap.add_argument("--out", default="")
    ap.add_argument("--compare", default="")
    ap.add_argument("--oracle-rows", type=int, default=2)
    ap.add_argument("--ragged", action="store_true")
    ap.add_argument("--state", action="store_true", help="also run as two chunks with carried state")
    a = ap.parse_args()
    cfg = synth.CONFIGS[a.config]
    sd = synth.make_state_dict(cfg, 1234)
    ec = EngineConfig(n_mels=cfg.n_mels, n_stack=cfg.n_stack, downsample=cfg.downsample, enc_layers=cfg.enc_layers,
                      pred_layers=cfg.pred_layers, hidden_sz=cfg.hidden_sz, embed_sz=cfg.embed_sz,
                      joint_sz=cfg.joint_sz, vocab_sz=cfg.vocab_sz)
    eng = Engine(ec).load_state_dict(sd)
    g = torch.Generator().manual_seed(77)
    X = cfg.n_mels * cfg.n_stack
    feats = torch.randn(a.B, a.T, X, generator=g) * 2.0
    lens = None
    if a.ragged:
        lens = torch.tensor([max(1, a.T - 3 * b) for b in range(a.B)], dtype=torch.int32)
    fd = feats.cuda()
    ld = lens.cuda() if lens is not None else None
    res = {"B": a.B, "T": a.T, "config": a.config}
    enc, st = eng.encode(fd, ld, want_state=True)
    torch.cuda.synchronize()
    enc_c = enc.cpu()
    res["finite"] = bool(torch.isfinite(enc_c).all())
    # oracle on a few rows
    orc = O.OracleTransducer(cfg, sd)
    n = min(a.oracle_rows, a.B)
    worst = 0.0
    worst_s = 0.0
    with torch.no_grad():
        for b in range(n):
            Tb = int(lens[b]) if lens is not None else a.T
            e_ref, s_ref = orc.encoder(feats[b:b + 1, :Tb], None, "aten")
            worst = max(worst, float((enc_c[b, :Tb] - e_ref[0]).abs().max()))
            for l, (hh, cc) in enumerate(s_ref):
                worst_s = max(worst_s, float((st[0][l, b].cpu() - hh.reshape(-1)).abs().max()), float((st[1][l, b].cpu() - cc.reshape(-1)).abs().max()))
    res["max_abs_vs_oracle"] = worst
    res["max_abs_state_vs_oracle"] = worst_s
    if a.state and a.T >= 4:
        t1 = a.T // 2
        e1, s1 = eng.encode(fd[:, :t1].contiguous(), None, want_state=True)
        e2, s2 = eng.encode(fd[:, t1:].contiguous(), None, state=s1, want_state=True)
        full, sf = eng.encode(fd, None, want_state=True)
        torch.cuda.synchronize()
        res["chunked_vs_full_max_abs"] = float((torch.cat([e1, e2], 1) - full).abs().max())
        res["chunked_state_max_abs"] = float(max((s2[0] - sf[0]).abs().max(), (s2[1] - sf[1]).abs().max()))
    if a.out:
        np.save(a.out, enc_c.numpy())
    if a.compare and os.path.exists(a.compare):
        other = torch.from_numpy(np.load(a.compare))
        res["max_abs_vs_other_version"] = float((enc_c - other).abs().max())
    # timing
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        eng.encode(fd, ld)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(10):
        eng.encode(fd, ld)
    ev1.record()
    torch.cuda.synchronize()
    res["encode_ms"] = ev0.elapsed_time(ev1) / 10
    print(json.dumps(res), flush=True)
    eng.close()


if __name__ == "__main__":
    main()
