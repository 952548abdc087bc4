"""Accuracy / speed of the library GEMM arithmetic modes against an fp64 product (GPU box)."""
import json, os, sys, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from libreasr_b200.engine import Engine, EngineConfig

def main():
    eng = Engine(EngineConfig(n_mels=16, enc_layers=1, pred_layers=1, hidden_sz=64, embed_sz=32, joint_sz=64, vocab_sz=64))
    res = []
    g = torch.Generator(device="cuda").manual_seed(0)
    for (M, N, K) in [(128, 256, 64), (300, 260, 160), (1000, 512, 800), (3968, 4096, 800), (3968, 4096, 1024), (3968, 1024, 1024)]:
        A = torch.randn(M, K, device="cuda", generator=g)
        W = (torch.rand(N, K, device="cuda", generator=g) * 2 - 1) * 0.1
        b = torch.randn(N, device="cuda", generator=g)
        ref = (A.double() @ W.double().t() + b.double())
        scale = float(ref.abs().mean())
        row = {"M": M, "N": N, "K": K}
        for mode in (0, 1):
            try:
                C = eng.selftest_gemm(A, W, b, gemm_mode=mode)
                torch.cuda.synchronize()
                err = (C.double() - ref).abs()
                row[f"mode{mode}_maxerr"] = float(err.max()); row[f"mode{mode}_rel_rms"] = float(err.pow(2).mean().sqrt() / scale)
                t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(5):
                    eng.selftest_gemm(A, W, b, gemm_mode=mode)
                t1.record(); torch.cuda.synchronize()
                row[f"mode{mode}_ms"] = t0.elapsed_time(t1) / 5
            except Exception as e:
                row[f"mode{mode}_exc"] = repr(e)
        tf = (A.to(torch.float32) @ W.t() + b)
        row["torch_f32_maxerr"] = float((tf.double() - ref).abs().max())
        print(row, flush=True)
        res.append(row)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(res, open(os.path.join(ROOT, "gpurun_out", "gemm_check.json"), "w"), indent=1)

if __name__ == "__main__":
    main()
