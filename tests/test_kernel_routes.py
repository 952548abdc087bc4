"""Which recurrent kernel each call runs (capi.cu: route_encoder / route_decoder).

* CPU: the library reads only the environment switches it documents, and the retired CTA-pair GEMM stays gone.
* GPU: the kernels launched per call, recorded with torch.profiler, pin the route table at the cfg2 shape (4 x 1024
  encoder, 2 x 1024 predictor): stateless batches of up to 32 rows run the cluster kernels, wider ones 32-row
  sub-batches of them; a 40-stream streaming tick runs the round-1 kernels; the fused LM runs decode_tc_kernel<true>;
  gemm_mode 0 runs the fp32 kernels.
"""
import glob
import os
import re

import pytest
import torch

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "libreasr_b200", "csrc")


def test_environment_switches_and_retired_kernels():
    names, pair = set(), []
    for path in glob.glob(os.path.join(CSRC, "*")):
        with open(path) as f:
            src = f.read()
        names |= set(re.findall(r'getenv\("([A-Z0-9_]+)"\)', src))
        if "gemm_tc2" in src:
            pair.append(os.path.basename(path))
    assert names == {"RNNT_NO_COOP", "RNNT_LSTM_DBG", "RNNT_DEC_DBG"}
    assert not os.path.exists(os.path.join(CSRC, "gemm_tc2.cu"))
    assert pair == []


# ---------------- route table on the GPU ----------------
LSTM_TC2, LSTM_TC, LSTM_STEP = "lstm_layer_tc2_kernel", "lstm_layer_tc_kernel", "lstm_step_kernel"
DEC_TC2, DEC_TC, DEC_FP32 = "decode_tc2_kernel", "decode_tc_kernel", "decode_greedy_kernel"
ROUTED = (LSTM_TC2, LSTM_TC, LSTM_STEP, DEC_TC2, DEC_TC, DEC_FP32)


def _launched(fn):
    """Names (kernel identifier with template arguments) and counts of the routed kernels `fn` launches."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    counts = {}
    for ev in prof.events():
        if ev.device_type != DeviceType.CUDA:
            continue
        for k in ROUTED:
            m = re.search(k + r"(<[^>]*>)?\(", ev.name)
            if m:
                key = k + (m.group(1) or "")
                counts[key] = counts.get(key, 0) + 1
    return counts


def _cfg2(gemm_mode):
    from test_gpu_parity import Lang
    from libreasr_b200.lib.models import Transducer
    from oracle import weights

    cfg = weights.CONFIGS["cfg2"]
    m = Transducer(cfg.feature_sz, cfg.embed_sz, cfg.vocab_sz, cfg.hidden_sz, cfg.out_sz, cfg.joint_sz, Lang(),
                   encoder_kwargs={"num_layers": cfg.enc_layers}, predictor_kwargs={"num_layers": cfg.pred_layers},
                   gemm_mode=gemm_mode)
    m.load_state_dict({k: torch.as_tensor(v) for k, v in weights.make_state_dict(cfg, 1234).items()}, strict=True)
    return cfg, m.to("cuda:0").engine()


def _inputs(cfg, B, T, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, T, cfg.feature_sz, generator=g).cuda()


@pytest.mark.gpu
def test_route_table_cfg2():
    from test_gpu_parity import lm_model_for

    cfg, eng = _cfg2(1)
    L = cfg.enc_layers

    def offline(e, B):
        enc, _ = e.encode(_inputs(cfg, B, 24, B))
        return lambda: e.decode_greedy(enc, max_iters=3)

    for B, n in ((32, 1), (64, 2)):   # stateless: the cluster kernels, one launch per 32 rows
        feats = _inputs(cfg, B, 24, B)
        assert _launched(lambda: eng.encode(feats)) == {LSTM_TC2: n * L}, B
        assert _launched(offline(eng, B)) == {DEC_TC2: n}, B

    # a streaming tick of 40 streams (carried state, T = 2): one wide launch of the round-1 kernels
    S = 40
    feats = _inputs(cfg, S, 2, 7)
    _, st = eng.encode(feats, want_state=True)
    enc_counts = _launched(lambda: eng.encode(feats, state=st, want_state=True))
    assert set(enc_counts) == {LSTM_TC + "<true>"} and enc_counts[LSTM_TC + "<true>"] == L
    enc, _ = eng.encode(feats, state=st)
    r0 = eng.decode_greedy(enc, max_iters=10, want_state=True)
    assert _launched(lambda: eng.decode_greedy(enc, max_iters=10, state=r0["state"], want_state=True)) == {DEC_TC + "<false>": 1}

    # the fused LM (4 x 768) inside the round-1 decode kernel
    _, _, mlm, _, _ = lm_model_for("cfg2", "en")
    elm = mlm.engine()
    enc, _ = elm.encode(_inputs(cfg, 8, 24, 11))
    assert _launched(lambda: elm.decode_greedy(enc, max_iters=3)) == {DEC_TC + "<true>": 1}

    # gemm_mode 0: the fp32 kernels (one LSTM step launch per layer and frame)
    _, e0 = _cfg2(0)
    feats = _inputs(cfg, 8, 6, 13)
    assert _launched(lambda: e0.encode(feats)) == {LSTM_STEP: 6 * L}
    assert _launched(offline(e0, 8)) == {DEC_FP32: 1}
