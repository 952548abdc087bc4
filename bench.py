#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 RNN-T inference path (driver contract).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N ...            # the reference's own CPU path (same metric / config)

Headline workload (BASELINE.json configs[1]): batch = 32 synthetic 16 kHz utterances of 10 s,
80-mel x 10-stack features, 4x1024 LSTM encoder, 2x1024 GRU predictor, joint 1024,
vocab 2048, greedy decode (max_iters = 3).  One "step" = the whole hot path over one batch:
audio -> log-mel/stack -> LayerNorm -> LSTM stack -> joint/predictor greedy loop -> tokens.
Metric: streaming RTFx = audio-seconds processed / wall-second (whole job, all GPUs).

Prints ONE JSON line (rank 0).  Under torchrun every rank processes its own 32-utterance batch for the
headline (`"scaling": "weak"`, no data-path collective).  Next to the headline the line carries, under `extra`,
the other BASELINE configs measured in the same run (VERDICT r1 item 3): `stream64` (configs[2] through the C
streaming session), `lm_4x768` (LM shallow fusion), `cfg4_b128` (configs[3] shape, greedy), and `strong`
(configs[4]: rank 0 holds 256..2048 utterances, NCCL scatter -> per-rank transcribe -> NCCL gather).
"""
import argparse
import dataclasses
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "cfg2"
BATCH = 32
SECONDS = 10.0
MAX_ITERS = 3
N_ROTATE = 8  # distinct input batches cycled through the timed region (8 x 20.5 MB > 126 MB L2)
CHUNK = 1280


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock / throttle reasons through NVML, sampled every few ms from a thread that starts BEFORE warm-up; only
    samples that fall inside a timed region (`begin()` .. `end()`) are reported, so even a 0.2 s region yields dozens."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, device, period_s=0.004):
        self.period, self.rows, self.windows, self._t0 = period_s, [], [], None
        self.stop_ev = threading.Event()
        self.h = None
        try:
            import pynvml

            self.nv = pynvml
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(device).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if not uuid.startswith("GPU-") else uuid.encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                idx = int(vis.split(",")[device.index]) if vis and vis.split(",")[0].isdigit() else device.index
                self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
            self.h = None

    def start(self):
        if self.h is None:
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_ev.is_set():
            try:
                self.rows.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), int(get_reasons(self.h))))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def begin(self):
        self._t0 = time.perf_counter()

    def end(self):
        self.windows.append((self._t0, time.perf_counter()))

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")], "samples": 0}
        self.stop_ev.set()
        self.thread.join(timeout=1)
        inside = [(mhz, r) for (t, mhz, r) in self.rows if any(a <= t <= b for a, b in self.windows)]
        reasons = sorted({name for _, r in inside for bit, name in self.REASONS if r & bit})
        return {"sm_mhz": float(np.median([m for m, _ in inside])) if inside else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside), "samples_total": len(self.rows),
                "source": "NVML, sampled inside the timed regions (device-resident and e2e loops)"}


def model_flops_bytes(cfg, B, T, evals, emitted):
    """Algorithmic work of one step (DESIGN.md section 'Algorithmic bytes and flops')."""
    H, X, J, V, L = cfg.hidden_sz, cfg.feature_sz, cfg.joint_sz, cfg.vocab_sz, cfg.enc_layers
    enc = B * T * (2 * (X + H) * 4 * H + (L - 1) * 2 * (2 * H) * 4 * H)
    joint_enc = B * T * 2 * H * J
    dec = evals * 2 * J * V + emitted * (2 * H * J + 2 * H * 3 * H * (2 * cfg.pred_layers - 1))
    return {"encoder_flops": enc, "joint_enc_flops": joint_enc, "decode_flops": dec}


def engine_config(cfg, gemm_mode, lm=None):
    from libreasr_b200.engine import EngineConfig

    ec = EngineConfig(n_mels=cfg.n_mels, n_stack=cfg.n_stack, downsample=cfg.downsample, enc_layers=cfg.enc_layers,
                      pred_layers=cfg.pred_layers, hidden_sz=cfg.hidden_sz, embed_sz=cfg.embed_sz, joint_sz=cfg.joint_sz,
                      vocab_sz=cfg.vocab_sz, gemm_mode=gemm_mode)
    if lm is not None:
        ec = dataclasses.replace(ec, lm_layers=lm.num_layers, lm_hidden_sz=lm.hidden_sz, lm_embed_sz=lm.embed_sz)
    return ec


def dump_outputs(out_dir, out):
    """Writes what the headline path returned for its last timed batch as <out_dir>/<name>.npy (float64; token slots past
    a row's ntok are -1, so two builds compare equal when they emit the same transcripts)."""
    os.makedirs(out_dir, exist_ok=True)
    tokens = out["tokens"].cpu().numpy().astype(np.float64)
    ntok = out["ntok"].cpu().numpy()
    tokens[np.arange(tokens.shape[1])[None, :] >= ntok[:, None]] = -1.0
    arrays = {"tokens": tokens, "ntok": ntok.astype(np.float64), "neg_logp": out["neg_logp"].cpu().numpy().astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def timed_ms(fn, steps, warmup, dev):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / steps


# ---------------------------------------------------------------------------------------------------------------
# extra legs (the other BASELINE configs, same run, same clock)
# ---------------------------------------------------------------------------------------------------------------
def leg_stream64(eng, dev, seconds=60.0, streams=64):
    """BASELINE configs[2]: 64 concurrent 80 ms-chunk streams through rnnt_b200_stream_push (pinned host chunks in, host
    tokens out every tick), reference windowing (3-chunk window, Buffer of 2), max_iters 10."""
    from libreasr_b200 import synth
    from libreasr_b200.api import StreamBatch

    n_chunks = int(seconds * 16000) // CHUNK
    pool = synth.make_audio(streams, 8 * 16000, seed=1)      # seed 1: SURVEY 8d config 3; tiled with per-stream shifts to `seconds`
    reps = -(-n_chunks * CHUNK // pool.shape[1])
    audio = np.concatenate([np.roll(pool, 4099 * r, axis=1) for r in range(reps)], axis=1)[:, : n_chunks * CHUNK]
    host = torch.from_numpy(audio.reshape(streams, n_chunks, CHUNK).transpose(1, 0, 2).copy()).pin_memory()
    sb = StreamBatch(eng, streams, max_iters=10)
    warm, lat = 10, []
    t0 = None
    for j in range(n_chunks):
        if j == warm:
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
        t1 = time.perf_counter()
        new = sb.push(host[j])
        if new is not None and j >= warm:
            lat.append(time.perf_counter() - t1)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    audio_s = streams * (n_chunks - warm) * CHUNK / 16000.0
    ntok = int(sum(len(t) for t in sb.tokens))
    sb.close()
    return {"workload": "BASELINE.json configs[2]: 64 concurrent streams, 80 ms chunks, 4x1024 LSTM, greedy max_iters 10, reference windowing",
            "value": round(audio_s / dt, 1), "unit": "x real-time", "streams": streams,
            "audio_s_per_stream": round((n_chunks - warm) * 0.08, 2), "wall_s": round(dt, 3),
            "tick_ms_p50": round(1e3 * float(np.median(lat)), 3), "tick_ms_p99": round(1e3 * float(np.quantile(lat, 0.99)), 3),
            "tick_ms_mean": round(1e3 * float(np.mean(lat)), 3), "model_ticks": len(lat), "tokens": ntok,
            "api": "rnnt_b200_stream_push (host chunks in, host tokens out, one call per 80 ms tick for all streams)",
            "h2d_bytes_per_tick": streams * CHUNK * 4}


def leg_lm(dev, gemm_mode, devb, steps):
    """configs[1] workload with the shipped 4x768 LM fused in the decode loop (testing.yaml:306-313, lm.py:43-83)."""
    from libreasr_b200 import synth
    from libreasr_b200.engine import Engine

    cfg, lc = synth.CONFIGS[WORKLOAD], synth.LM_CONFIGS["en"]
    eng = Engine(engine_config(cfg, gemm_mode, lc), device=dev).load_state_dict(synth.make_state_dict(cfg, 1234),
                                                                                 lm_state_dict=synth.make_lm_state_dict(lc, 4321))
    k = [0]

    def step():
        k[0] += 1
        return eng.transcribe(devb[k[0] % len(devb)], max_iters=MAX_ITERS)

    ms = timed_ms(step, steps, 3, dev)
    r = step()
    ntok = int(r["ntok"].sum())
    eng.close()
    return {"workload": "configs[1] batch with the 4x768 LSTM LM shallow-fused (LMFuser)", "value": round(BATCH * SECONDS / (ms / 1e3), 1),
            "unit": "x real-time", "ms_per_step": round(ms, 4), "tokens_per_step": ntok}


def leg_cfg4(dev, gemm_mode, steps=3):
    """BASELINE configs[3] shape: 128 x 15 s, 6x1536 LSTM encoder, greedy (beam search: see `beam` when present)."""
    from libreasr_b200 import synth
    from libreasr_b200.engine import Engine

    cfg = synth.CONFIGS["cfg4"]
    eng = Engine(engine_config(cfg, gemm_mode), device=dev).load_state_dict(synth.make_state_dict(cfg, 1234))
    n = 15 * 16000
    pool = synth.make_audio(16, n, seed=2)          # seed 2: SURVEY 8d config 4; 128 = 8 shifted copies of 16 distinct utterances
    audio = torch.from_numpy(np.concatenate([np.roll(pool, 1237 * r, axis=1) for r in range(8)], 0)).to(dev)
    eng.reserve(128, n)
    ms = timed_ms(lambda: eng.transcribe(audio, max_iters=MAX_ITERS), steps, 2, dev)
    r = eng.transcribe(audio, max_iters=MAX_ITERS)
    out = {"workload": "BASELINE.json configs[3] shape: batch=128 x 15 s, 6x1536 LSTM, greedy", "value": round(128 * 15.0 / (ms / 1e3), 1),
           "unit": "x real-time", "ms_per_step": round(ms, 3), "tokens_per_step": int(r["ntok"].sum())}
    # configs[3] as written: beam search, width 4 (not in the reference; algorithm of oracle/beam.py, rnnt_b200_decode_beam)
    try:
        msb = timed_ms(lambda: eng.transcribe_beam(audio, width=4, max_iters=MAX_ITERS), 2, 1, dev)
        rb = eng.transcribe_beam(audio, width=4, max_iters=MAX_ITERS)
        out["beam4"] = {"workload": "BASELINE.json configs[3]: offline beam search width=4, batch=128 x 15 s, 6x1536 LSTM", "value": round(128 * 15.0 / (msb / 1e3), 1),
                        "unit": "x real-time", "ms_per_step": round(msb, 3), "tokens_per_step": int(rb["ntok"].sum()),
                        "note": "first device implementation (per-expansion launch sequence, all contractions on tcgen05), parity vs oracle/beam.py in tests/test_gpu_beam.py"}
    except Exception as e:  # noqa: BLE001
        out["beam4"] = {"error": repr(e)[:300]}
    eng.close()
    return out


def leg_strong(eng, dev, dist, rank, world, base_dev, sizes=(256, 512, 1024, 2048)):
    """BASELINE configs[4]: rank 0 holds N utterances in HBM; scatter over NVLink (NCCL send/recv, block-pipelined with the
    first blocks' compute) -> per-rank transcribe -> gather of the padded token arrays to rank 0.  Strong scaling: the
    driver's N=1,2,4,8 runs give RTFx(G) for the same N; efficiency = RTFx(G) / (G * RTFx(1))."""
    from libreasr_b200 import parallel

    n = base_dev.shape[1]
    out = {}
    for N in sizes:
        audio = None
        if rank == 0:   # N utterances = shifted copies of the rank's distinct batches (content does not change the work per frame much)
            reps = -(-N // base_dev.shape[0])
            audio = torch.cat([torch.roll(base_dev, 811 * r, dims=1) for r in range(reps)], 0)[:N].contiguous()
        times = []
        for it in range(3):
            if dist:
                dist.barrier()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            if dist:
                toks = parallel.transcribe_sharded(eng, audio, None, N, n, max_iters=MAX_ITERS, block=64)
            else:
                r = eng.transcribe(audio, max_iters=MAX_ITERS)
                toks = [r["tokens"].cpu(), r["ntok"].cpu()]
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            if dist:
                tt = torch.tensor([dt], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt[0])
            times.append(dt)
        del audio, toks
        best = min(times[1:])   # first pass warms workspaces / NCCL channels
        out[str(N)] = {"value": round(N * n / 16000.0 / best, 1), "unit": "x real-time", "wall_ms": round(best * 1e3, 2),
                       "utterances_per_s": round(N / best, 1)}
    out["note"] = ("rank 0 holds the audio in HBM; NCCL scatter + per-rank transcribe + NCCL gather of tokens inside the timed region, "
                   "max over ranks; 10 s utterances, greedy" if dist else "single GPU reference point for the strong-scaling curve (no collective)")
    return out


def _trace(msg):
    """BENCH_TRACE=1: phase markers on stderr (where did a run stall?)."""
    if os.environ.get("BENCH_TRACE"):
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def run_product(args):
    from libreasr_b200 import synth
    from libreasr_b200.engine import Engine, tokens_to_lists

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()   # before warm-up: the thread is sampling long before the timed region opens

    cfg = synth.CONFIGS[WORKLOAD]
    n = int(SECONDS * cfg.sample_rate)
    eng = Engine(engine_config(cfg, args.gemm_mode), device=dev).load_state_dict(synth.make_state_dict(cfg, 1234))
    eng.reserve(BATCH, n)
    T = eng.num_steps(n)
    U = MAX_ITERS * T

    # synthetic input: N_ROTATE distinct batches per rank, in pinned host memory and in HBM
    # every rank gets the SAME synthetic batches (same seed): the number of lock-steps of the greedy loop depends on the content,
    # and the max over ranks is meant to measure the system, not which rank drew the longest transcript
    base = synth.make_audio(BATCH, n, seed=synth.BENCH_AUDIO_SEED)  # see synth.BENCH_AUDIO_SEED
    host = [torch.from_numpy(np.roll(base, 997 * r, axis=1).copy()).pin_memory() for r in range(N_ROTATE)]
    devb = [h.to(dev) for h in host]
    out_host = Engine.alloc_host_outputs(BATCH, U)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput (value) ----
    _trace("engine ready; warm-up")
    for i in range(args.warmup):
        _trace(f"warm-up step {i}")
        res = eng.transcribe(devb[i % N_ROTATE], max_iters=MAX_ITERS)
    barrier()
    l0 = eng.kernel_launches()
    eng.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.begin()
    e0.record()
    for i in range(args.steps):
        res = eng.transcribe(devb[i % N_ROTATE], max_iters=MAX_ITERS)
        if os.environ.get("BENCH_TRACE"):
            torch.cuda.synchronize(dev)
            _trace(f"timed step {i} (batch {i % N_ROTATE}) done")
    e1.record()
    barrier()
    _trace("device-resident loop done")
    sampler.end()
    ms_total = e0.elapsed_time(e1)
    stage = eng.stage_times_ms()
    eng.set_profiling(False)
    launches = (eng.kernel_launches() - l0) // max(args.steps, 1)
    toks = tokens_to_lists(res["tokens"], res["ntok"])
    iters = res["iters"].cpu().numpy()
    evals, emitted = int(iters.sum()), int(sum(len(t) for t in toks))

    if args.profile:
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, res)
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_total / args.steps, "launches_per_step": int(launches),
                              "stage_ms": stage}), flush=True)
        return None

    # ---- the same K steps with two batches in flight (rnnt_b200_pipeline_submit / _collect: copy + front end of batch i+1 under
    # the recurrent kernels of batch i).  The sequential numbers above are always reported; the pipelined ones replace `value` /
    # `e2e` only when they are faster, and a watchdog keeps a stall in this section from taking the bench line down.
    seq_ms_total = ms_total
    pipe_depth = 1
    out_slots = [Engine.alloc_host_outputs(BATCH, U), Engine.alloc_host_outputs(BATCH, U)]
    pipe_guard = {"deadline": None}

    def run_pipelined(inputs, steps, after_collect=None):
        prev = None
        for i in range(steps):
            pipe_guard["deadline"] = time.time() + 20.0
            eng.pipeline_submit(inputs[i % N_ROTATE], i & 1, max_iters=MAX_ITERS, out=out_slots[i & 1])
            if prev is not None:
                eng.pipeline_collect(prev)
                if after_collect:
                    after_collect(out_slots[prev])
            prev = i & 1
        if prev is not None:
            eng.pipeline_collect(prev)
            if after_collect:
                after_collect(out_slots[prev])
        pipe_guard["deadline"] = None

    def pipe_watchdog():
        while True:
            time.sleep(1.0)
            d = pipe_guard["deadline"]
            if d is not None and time.time() > d:
                sys.stderr.write("[bench] the pipelined section made no progress for 20 s: starting over without it (--no-pipeline)\n")
                sys.stderr.flush()
                if dist:
                    os._exit(17)   # the other ranks sit in a collective: fail loudly
                os.execv(sys.executable, [sys.executable] + sys.argv + ["--no-pipeline"])

    use_pipe = not args.no_pipeline
    if use_pipe:
        threading.Thread(target=pipe_watchdog, daemon=True).start()
        _trace("pipelined device-resident loop")
        run_pipelined(devb, max(args.warmup, 2))
        barrier()
        sampler.begin()
        e0.record()
        run_pipelined(devb, args.steps)
        e1.record()
        barrier()
        sampler.end()
        pipe_ms_total = e0.elapsed_time(e1)
        last = out_slots[(args.steps - 1) & 1]   # the last batch of both timed loops is the same one
        if tokens_to_lists(last["tokens"], last["ntok"]) != toks:
            raise RuntimeError("pipelined run produced different tokens than the sequential run on the same batch")
        if pipe_ms_total < ms_total:
            ms_total, pipe_depth = pipe_ms_total, 2
        _trace(f"pipelined loop done: {pipe_ms_total / args.steps:.3f} vs {seq_ms_total / args.steps:.3f} ms per step")
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last if pipe_depth == 2 else res)

    # ---- end-to-end through the public host-buffer call (e2e) ----
    def gather_tokens(o=None):
        if not dist:
            return
        t = (o or out_host)["tokens"].to(dev, non_blocking=True)
        gl = [torch.empty_like(t) for _ in range(world)] if rank == 0 else None
        dist.gather(t, gl, dst=0)
        if rank == 0:
            torch.stack(gl).cpu()

    for i in range(min(args.warmup, 3)):
        eng.transcribe_host(host[i % N_ROTATE], max_iters=MAX_ITERS, out=out_host)
        gather_tokens()
    barrier()
    sampler.begin()
    t0 = time.perf_counter()
    for i in range(args.steps):
        eng.transcribe_host(host[i % N_ROTATE], max_iters=MAX_ITERS, out=out_host)
        gather_tokens()
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    sampler.end()
    _trace("e2e loop done")
    e2e_seq_s, e2e_api = e2e_s, "rnnt_b200_transcribe_host (pinned host audio in, host tokens out)"
    if use_pipe:
        run_pipelined(host, 3, after_collect=lambda o: gather_tokens(o))
        barrier()
        sampler.begin()
        t0 = time.perf_counter()
        run_pipelined(host, args.steps, after_collect=lambda o: gather_tokens(o))
        torch.cuda.synchronize(dev)
        e2e_pipe_s = time.perf_counter() - t0
        sampler.end()
        if e2e_pipe_s < e2e_s:
            e2e_s = e2e_pipe_s
            e2e_api = ("rnnt_b200_pipeline_submit / _collect, two batches in flight (pinned host audio in, host tokens out; the copy and "
                       "the front end of batch i+1 run under the recurrent kernels of batch i)")
        _trace(f"pipelined e2e loop done: {e2e_pipe_s * 1e3 / args.steps:.3f} vs {e2e_seq_s * 1e3 / args.steps:.3f} ms per step")
    clocks = sampler.stop() if rank == 0 else None

    # max over ranks (+ every rank's own time: explains where a weak-scaling loss comes from)
    per_rank = None
    if dist:
        mine = torch.tensor([ms_total, e2e_s * 1e3], device=dev, dtype=torch.float64)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [[round(float(t[0]) / args.steps, 4), round(float(t[1]) / args.steps, 4)] for t in allr]
        ms_total, e2e_s = max(float(t[0]) for t in allr), max(float(t[1]) for t in allr) / 1e3

    audio_s = BATCH * SECONDS * world
    value = audio_s * args.steps / (ms_total / 1e3)
    e2e_value = audio_s * args.steps / e2e_s

    # ---- the other BASELINE configs, same run ----
    extra = {}
    if not args.no_extra:
        def leg(name, fn):
            try:
                t0 = time.perf_counter()
                extra[name] = fn()
                extra[name]["leg_wall_s"] = round(time.perf_counter() - t0, 1)
            except Exception as e:  # noqa: BLE001 -- an extra leg must never take the headline down
                extra[name] = {"error": repr(e)[:300]}
        leg("strong", lambda: leg_strong(eng, dev, dist, rank, world, devb[0]))
        if world == 1:
            leg("stream64", lambda: leg_stream64(eng, dev))
            leg("lm_4x768", lambda: leg_lm(dev, args.gemm_mode, devb, max(args.steps // 2, 5)))
            leg("cfg4_b128", lambda: leg_cfg4(dev, args.gemm_mode))

    line = None
    if rank == 0:
        peaks = load_peaks()
        work = model_flops_bytes(cfg, BATCH, T, evals, emitted)
        # per-kernel rooflines from the live CUDA-event stage times of the timed region.  Algorithmic work
        # (DESIGN.md section 4): tensor-bound kernels in flops vs the sustained bf16 peak (the kernels sit inside
        # a long step), the front end in bytes vs the measured HBM copy bandwidth.
        tc = args.gemm_mode == 1
        peak_t = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
        H, X, L = cfg.hidden_sz, cfg.feature_sz, cfg.enc_layers
        hoist_flops = BATCH * T * (2 * X * 4 * H + (L - 1) * 2 * H * 4 * H)
        rec_flops = work["encoder_flops"] - hoist_flops
        rec_ms = max(stage["encoder"] - stage["encoder_input_gemms"], 1e-6)
        fe_bytes = BATCH * (4 * n + 4 * T * X)
        lstm_v = os.environ.get("RNNT_LSTM_V", "2")

        def tens(name, flops, ms, launches):
            a = flops / (ms * 1e-3) / 1e12
            return {"kernel": name, "bound": "tensor", "achieved": round(a, 3), "peak": peak_t, "unit": "TFLOP/s",
                    "frac": round(a / peak_t, 5), "ms_per_step": round(ms, 4), "launches_per_step": launches,
                    "algorithmic_flops_per_step": int(flops)}
        lstm_name = ("lstm_layer_tc2_kernel" if lstm_v == "2" else "lstm_layer_tc_kernel") if tc else "lstm_step_kernel"
        dec_name = ("decode_tc2_kernel" if os.environ.get("RNNT_DEC_V", "2") == "2" else "decode_tc_kernel") if tc else "decode_greedy_kernel"
        per_kernel = [
            tens(dec_name, work["decode_flops"], stage["decode"], 1),
            tens(lstm_name, rec_flops, rec_ms, L if tc else L * T),
            tens("gemm_tc_f16x3_kernel" if tc else "gemm_nt_f32_kernel", hoist_flops, max(stage["encoder_input_gemms"], 1e-6), L),
            {"kernel": "mel_stack_kernel", "bound": "hbm", "achieved": round(fe_bytes / (stage["features"] * 1e-3) / 1e9, 1),
             "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(fe_bytes / (stage["features"] * 1e-3) / 1e9 / peaks["hbm_gbs"], 5),
             "ms_per_step": round(stage["features"], 4), "launches_per_step": 1, "algorithmic_bytes_per_step": fe_bytes},
        ]
        dom = max(per_kernel[:3], key=lambda k: k["ms_per_step"])
        # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/)
        ncu_traffic = {}
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            ncu_traffic = json.load(open(tpath))
        roofline = {"kernel": dom["kernel"], "bound": dom["bound"], "achieved": dom["achieved"], "peak": dom["peak"], "unit": dom["unit"],
                    "frac": dom["frac"], "traffic": ncu_traffic.get(dom["kernel"], {}).get("bytes"),
                    "traffic_source": ncu_traffic.get(dom["kernel"], {}).get("source"), "peak_source": peaks["source"] + ", sustained bf16 GEMM",
                    "ms_per_launch": round(dom["ms_per_step"] / dom["launches_per_step"], 4),
                    "flops_per_launch": int(dom["algorithmic_flops_per_step"] / dom["launches_per_step"]),
                    "note": ("dependent-chain (latency) bound at batch 32 (DESIGN.md section 4): fraction = algorithmic flops / sustained bf16 tensor peak; "
                             "the 3xFP16 split issues 3 fp16 MACs per algorithmic MAC" if tc else "fp32 CUDA-core mode; fraction vs the bf16 tensor peak"),
                    "per_kernel": per_kernel}
        _trace("cpu baseline")
        cpu = cpu_baseline(cfg, n, budget_s=args.cpu_budget)
        _trace("cpu baseline done")
        line = {
            "metric": "streaming RTFx (audio-s/wall-s)", "value": round(value, 1), "unit": "x real-time",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (3xFP16 split on tcgen05, fp32 accumulate)" if args.gemm_mode == 1 else "f32", "data": "synthetic",
            "utterances_per_s": round(BATCH * world * args.steps / (ms_total / 1e3), 1),
            "config": {"workload": "BASELINE.json configs[1]: batch=32 x 10 s synthetic 16 kHz, 80-mel, 4x1024 LSTM encoder, 2x1024 GRU predictor, greedy",
                       "global_batch": BATCH * world, "audio_s_per_utt": SECONDS, "enc_steps": T, "max_iters": MAX_ITERS,
                       "gemm_mode": {0: "fp32_simt", 1: "tc_fp16x3", 2: "tc_bf16"}[args.gemm_mode],
                       "parallelism": f"dp{world} (utterance shards, no data-path collective)",
                       "rank_batches": "identical synthetic batches on every rank (same seed)",
                       "l2": f"rotating {N_ROTATE} distinct input batches ({N_ROTATE * BATCH * n * 4 / 1e6:.0f} MB) > 126 MB L2",
                       "batches_in_flight": pipe_depth,
                       "sequential_ms_per_step": round(seq_ms_total / args.steps, 4),
                       "joint_evals_per_step": evals, "tokens_per_step": emitted,
                       "emission_rate_tok_per_frame": round(emitted / (BATCH * T), 3)},
            "e2e": {"value": round(e2e_value, 1), "unit": "x real-time", "h2d_bytes_per_step": BATCH * n * 4,
                    "d2h_bytes_per_step": BATCH * U * 4 + BATCH * 4 + BATCH * 8, "ms_per_step": round(e2e_s * 1e3 / args.steps, 4),
                    "api": e2e_api, "sequential_ms_per_step": round(e2e_seq_s * 1e3 / args.steps, 4)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "per_rank_ms_per_step": per_rank,
            "stage_ms": {k: round(v, 4) for k, v in stage.items()},
            "roofline": roofline,
            "cpu_baseline": cpu,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return line


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference when it is importable (/root/reference or baseline/_ref), else the oracle port
# ---------------------------------------------------------------------------------------------------------------
def make_cpu_runner(cfg):
    """Returns (transcribe_batch(audio [B, n]) -> token lists, kind, description)."""
    from oracle import ref_runner

    if ref_runner.available():
        rr = ref_runner.ReferenceRunner(cfg)
        return (lambda audio: rr.transcribe_batch(audio, MAX_ITERS)), "reference", f"unmodified libreasr.lib.models from {rr.root} (Transducer.decode_greedy, bs=1)"
    from libreasr_b200 import synth
    from oracle import rnnt_oracle as O

    orc = O.OracleTransducer(cfg, synth.make_state_dict(cfg, 1234))
    return (lambda audio: O.transcribe_batch(orc, audio, max_iters=MAX_ITERS)), "port", "oracle restatement (reference package not importable here)"


def pick_cpu_threads(run, probe_audio):
    """torch's intra-op pool is slow when oversubscribed on batch-1 GEMVs (128 threads on a
    128-core host are ~500x slower than 8), so the CPU arm uses the fastest of a few pool sizes
    (the reference itself pins 2 threads, inference.py:21)."""
    best, best_t = None, None
    ncpu = os.cpu_count() or 1
    for th in sorted({2, 4, 8, 16, 32} & set(range(1, ncpu + 1)) | {min(ncpu, 8)}):
        torch.set_num_threads(th)
        run(probe_audio)  # warm the pool
        t0 = time.perf_counter()
        run(probe_audio)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
        if dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best


def cpu_baseline(cfg, n, budget_s=12.0, max_utts=512, pool=16, seed=100):
    """The reference's CPU path, utterance by utterance as the reference serves them, on this host's cores, on a bounded
    sample of the workload (a rate metric: 10 s utterances of the same distribution, so the sample size does not bias it)."""
    from libreasr_b200 import synth

    run, kind, what = make_cpu_runner(cfg)
    audio = synth.make_audio(pool, n, seed=seed)   # the sample cycles over a pool of distinct utterances
    threads = pick_cpu_threads(run, audio[:1, : n // 5])
    done, t0 = 0, time.perf_counter()
    while done < max_utts and (done < 1 or time.perf_counter() - t0 < budget_s):
        run(audio[done % pool:done % pool + 1])
        done += 1
    dt = time.perf_counter() - t0
    # as shipped: the reference pins 2 intra-op threads (inference.py:21); a short sample of the same workload
    torch.set_num_threads(2)
    run(audio[:1, : n // 5])
    k2, t2 = 0, time.perf_counter()
    while k2 < 3 and (k2 < 1 or time.perf_counter() - t2 < 4.0):
        run(audio[k2 % pool:k2 % pool + 1])
        k2 += 1
    d2 = time.perf_counter() - t2
    torch.set_num_threads(threads)
    return {"value": round(done * n / cfg.sample_rate / dt, 2), "unit": "x real-time", "cores": threads,
            "as_shipped_2_threads": round(k2 * n / cfg.sample_rate / d2, 2),
            "host_cpus": os.cpu_count(), "kind": kind, "implementation": what,
            "threads_note": "intra-op pool size picked by probing {2,4,8,16,32}: the bs=1 GEMVs of this path get slower beyond it",
            "same_config": "same model / utterance length / greedy settings; a bounded sample (rate metric), bs=1 because the reference has no batched decode (testing.yaml:380)",
            "sample": f"{done} utterances x {n / cfg.sample_rate:.0f} s of the same workload, sequential, {dt:.1f} s wall"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the unmodified package when importable,
    else the oracle port), all useful host threads, same metric/config; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from libreasr_b200 import synth

    cfg = synth.CONFIGS[WORKLOAD]
    n = int(SECONDS * cfg.sample_rate)
    run, kind, what = make_cpu_runner(cfg)
    per_step = 2  # bounded sample: 2 of the 32 utterances per step
    audio = synth.make_audio(per_step * (args.steps + args.warmup), n, seed=100)
    threads = pick_cpu_threads(run, audio[:1, : n // 5])
    k = 0
    for _ in range(args.warmup):
        run(audio[k:k + per_step])
        k += per_step
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run(audio[k:k + per_step])
        k += per_step
    dt = time.perf_counter() - t0
    value = per_step * args.steps * SECONDS / dt
    sample = f"{per_step} of {BATCH} utterances per step, sequential bs=1 (the reference has no batched decode), torch fp32 CPU, {threads} intra-op threads"
    print(json.dumps({
        "impl": "reference", "metric": "streaming RTFx (audio-s/wall-s)", "value": round(value, 2), "unit": "x real-time",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt * 1e3 / args.steps, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[1] (bounded sample): 10 s synthetic 16 kHz utterances, 80-mel, 4x1024 LSTM, greedy",
                   "sample": sample, "implementation": what},
        "cpu_baseline": {"value": round(value, 2), "unit": "x real-time", "cores": threads, "kind": kind, "sample": sample, "implementation": what},
        "e2e": {"value": round(value, 2), "unit": "x real-time", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--gemm-mode", type=int, default=1, help="1 = tcgen05 3xFP16 (default), 0 = fp32 CUDA cores")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-pipeline", action="store_true", help="time only one batch at a time (rnnt_b200_transcribe / _transcribe_host)")
    ap.add_argument("--no-extra", action="store_true", help="headline only (skip the stream64 / LM / cfg4 / strong-scaling legs)")
    ap.add_argument("--profile", action="store_true",
                    help="for runs under ncu: device-resident steps only, no e2e / CPU legs, warm-up not forced to 3 "
                         "(numbers printed in this mode are not bench values)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the headline path's outputs for its last batch as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if not args.profile:
        args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
