"""Soak tests of the persistent kernels (tuning / debugging aid): many back-to-back calls with a watchdog that reports where a
stall happened, and a determinism check across repeats of the same input.  STRESS_LIB=<librnnt_b200 build> picks the library.
  STRESS_MODE=offline  (default) bench workload, 32 x 10 s on 8 rotated batches: cluster kernels (STRESS_STAGED=1: stage by stage)
  STRESS_MODE=lm       the same batches with the 4x768 LM fused (round-1 decode kernel with LM)
  STRESS_MODE=b64      64 x 10 s stateless (32-row sub-batches of the cluster kernels)
  STRESS_MODE=cfg4     128 x 15 s on the 6x1536 shape (round-1 kernels, CTAs sitting phases out)
  STRESS_MODE=pipe     the offline workload through rnnt_b200_pipeline_submit / _collect (STRESS_HOST=1: pinned host inputs)
  STRESS_MODE=stream   STRESS_STREAMS (64: round-1 kernels, 32: cluster kernels) concurrent streams through rnnt_b200_stream_push"""
import os, sys, threading, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from libreasr_b200 import _capi
if os.environ.get("STRESS_LIB"):
    _capi.LIB_PATH = os.environ["STRESS_LIB"]
from libreasr_b200 import synth
from libreasr_b200.engine import Engine, EngineConfig

mode = os.environ.get("STRESS_MODE", "offline")
calls = int(os.environ.get("STRESS_CALLS", "600"))
staged = os.environ.get("STRESS_STAGED", "0") == "1"
progress = [time.time(), "start"]


def dog():
    while True:
        time.sleep(0.5)
        if time.time() - progress[0] > float(os.environ.get("STRESS_WAIT", "8")):
            print("STALL at", progress[1], flush=True)
            os._exit(3)


def econf(cfg, lc=None):
    kw = dict(n_mels=cfg.n_mels, n_stack=cfg.n_stack, downsample=cfg.downsample, enc_layers=cfg.enc_layers, pred_layers=cfg.pred_layers,
              hidden_sz=cfg.hidden_sz, embed_sz=cfg.embed_sz, joint_sz=cfg.joint_sz, vocab_sz=cfg.vocab_sz)
    if lc is not None:
        kw.update(lm_layers=lc.num_layers, lm_hidden_sz=lc.hidden_sz, lm_embed_sz=lc.embed_sz)
    return EngineConfig(**kw)


threading.Thread(target=dog, daemon=True).start()
t_all = time.time()
if mode in ("offline", "lm", "b64"):
    cfg = synth.CONFIGS["cfg2"]
    lc = synth.LM_CONFIGS["en"] if mode == "lm" else None
    eng = Engine(econf(cfg, lc)).load_state_dict(synth.make_state_dict(cfg, 1234), lm_state_dict=synth.make_lm_state_dict(lc, 4321) if lc else None)
    B, n, NR = (64 if mode == "b64" else 32), 160000, 8
    eng.reserve(B, n)
    base = synth.make_audio(B, n, seed=synth.BENCH_AUDIO_SEED)
    dev = [torch.from_numpy(np.roll(base, 997 * r, axis=1).copy()).cuda() for r in range(NR)]
    want = {}
    t0 = time.time()
    for i in range(calls):
        r = i % NR
        if staged:
            progress[:] = [time.time(), f"call {i} batch {r} features"]
            f = eng.features(dev[r]); torch.cuda.synchronize()
            progress[:] = [time.time(), f"call {i} batch {r} encode"]
            e = eng.encode(f); torch.cuda.synchronize()
            progress[:] = [time.time(), f"call {i} batch {r} decode"]
            res = eng.decode_greedy(e[0] if isinstance(e, tuple) else e); torch.cuda.synchronize()
        else:
            progress[:] = [time.time(), f"call {i} batch {r}"]
            res = eng.transcribe(dev[r]); torch.cuda.synchronize()
        nt = res["ntok"].tolist()
        assert r not in want or nt == want[r], f"call {i} batch {r}: token counts changed"
        want[r] = nt
    print(f"OK mode={mode} {calls} calls, {(time.time()-t0)*1e3/calls:.3f} ms/call, fp32 decode launches {eng.fp32_decode_launches()}", flush=True)
elif mode == "pipe":
    cfg = synth.CONFIGS["cfg2"]
    eng = Engine(econf(cfg)).load_state_dict(synth.make_state_dict(cfg, 1234))
    B, n, NR = 32, 160000, 8
    eng.reserve(B, n)
    base = synth.make_audio(B, n, seed=synth.BENCH_AUDIO_SEED)
    host = [torch.from_numpy(np.roll(base, 997 * r, axis=1).copy()).pin_memory() for r in range(NR)]
    inp = host if os.environ.get("STRESS_HOST", "0") == "1" else [h.cuda() for h in host]
    want = [eng.transcribe_host(h)["ntok"].tolist() for h in host]
    U = 3 * eng.num_steps(n)
    outs = [Engine.alloc_host_outputs(B, U), Engine.alloc_host_outputs(B, U)]
    torch.cuda.synchronize()
    t0 = time.time()
    prev = None
    for i in range(calls):
        progress[:] = [time.time(), f"submit {i}"]
        eng.pipeline_submit(inp[i % NR], i & 1, out=outs[i & 1])
        if prev is not None:
            progress[:] = [time.time(), f"collect {prev[1]} (slot states {eng.pipeline_query(0)} {eng.pipeline_query(1)})"]
            eng.pipeline_collect(prev[0])
            assert outs[prev[0]]["ntok"].tolist() == want[prev[1] % NR], f"batch {prev[1]}: token counts differ from the plain call"
        prev = (i & 1, i)
    eng.pipeline_collect(prev[0])
    dt = time.time() - t0
    t0 = time.time()
    for i in range(min(calls, 200)):
        progress[:] = [time.time(), f"plain call {i}"]
        eng.transcribe_host(host[i % NR], out=outs[0]) if inp is host else eng.transcribe(inp[i % NR])
    torch.cuda.synchronize()
    print(f"OK mode=pipe {calls} batches, {dt*1e3/calls:.3f} ms/batch pipelined vs {(time.time()-t0)*1e3/min(calls,200):.3f} plain, host inputs={inp is host}", flush=True)
elif mode == "cfg4":
    cfg = synth.CONFIGS["cfg4"]
    eng = Engine(econf(cfg)).load_state_dict(synth.make_state_dict(cfg, 1234))
    n = 15 * 16000
    pool = synth.make_audio(16, n, seed=2)
    audio = [torch.from_numpy(np.concatenate([np.roll(pool, 1237 * r + 311 * k, axis=1) for r in range(8)], 0)).cuda() for k in range(2)]
    eng.reserve(128, n)
    want = {}
    t0 = time.time()
    for i in range(calls):
        progress[:] = [time.time(), f"call {i}"]
        res = eng.transcribe(audio[i & 1]); torch.cuda.synchronize()
        nt = res["ntok"].tolist()
        assert (i & 1) not in want or nt == want[i & 1], f"call {i}: token counts changed"
        want[i & 1] = nt
    print(f"OK mode=cfg4 {calls} calls, {(time.time()-t0)*1e3/calls:.3f} ms/call", flush=True)
elif mode == "stream":
    from libreasr_b200.api import StreamBatch
    S = int(os.environ.get("STRESS_STREAMS", "64"))
    cfg = synth.CONFIGS["cfg2"]
    eng = Engine(econf(cfg)).load_state_dict(synth.make_state_dict(cfg, 1234))
    CH = 1280
    pool = synth.make_audio(S, 8 * 16000, seed=1)
    nck = pool.shape[1] // CH
    host = torch.from_numpy(pool[:, : nck * CH].reshape(S, nck, CH).transpose(1, 0, 2).copy()).pin_memory()
    sb = StreamBatch(eng, S, max_iters=10)
    t0 = time.time()
    for j in range(calls):
        progress[:] = [time.time(), f"tick {j}"]
        sb.push(host[j % nck])
    torch.cuda.synchronize()
    print(f"OK mode=stream streams={S} {calls} ticks, {(time.time()-t0)*1e3/calls:.3f} ms/tick, tokens {sum(len(t) for t in sb.tokens)}, fp32 decode launches {eng.fp32_decode_launches()}", flush=True)
    sb.close()
print(f"total {time.time()-t_all:.1f} s", flush=True)
