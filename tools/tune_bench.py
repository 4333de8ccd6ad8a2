#!/usr/bin/env python
"""Decoder fine-tuning on one GPU: ms per training step of B = 128 clips x T = 250 chunks (8 s at 16 kHz) at both rates, by stage,
against the reference's training loop (tuning/utils.py:231-243: per chunk stft -> encoder -> LSTMCell -> head, autograd) with the
reference TorchScript model from baseline/_ref moved to the same GPU; and the threshold search on 1000 files x 250 chunks
against its pure-Python loop (timed on a subset whose size is printed).  Prints one JSON line (with the card and its power limit).

    python tools/tune_bench.py [--steps 20] [--out FILE]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch
import torch.nn as nn

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
from silero_vad_b200 import (SileroVADB200, VADDecoderRNNJIT, calculate_best_thresholds, decoder_state_dict,  # noqa: E402
                             encoder_features, train)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.splitlines()[0]
        name, pl = [s.strip() for s in out.split(",")]
        return name, pl
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def timed(fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


class _Cfg:
    def __init__(self, tune_8k):
        self.tune_8k = tune_8k


def reference_step(jit, sr, x, targets, masks, steps):
    """The reference's loop on the GPU: pad(x, (ctx, 0)), per chunk stft -> encoder -> nn.LSTMCell -> head, BCE * masks, Adam."""
    ctx, n = (64, 512) if sr == 16000 else (32, 256)
    br = jit._model if sr == 16000 else jit._model_8k
    rnn = nn.LSTMCell(128, 128).cuda()
    head = nn.Sequential(nn.Dropout(0.1), nn.ReLU(), nn.Conv1d(128, 1, kernel_size=1), nn.Sigmoid()).cuda()
    sd = decoder_state_dict(sr)
    rnn.load_state_dict({k[4:]: v for k, v in sd.items() if k.startswith("rnn.")})
    head.load_state_dict({k[8:]: v for k, v in sd.items() if k.startswith("decoder.")})
    params = list(rnn.parameters()) + list(head.parameters())
    opt = torch.optim.Adam(params, lr=5e-4)
    crit = nn.BCELoss(reduction="none")

    def step():
        with torch.enable_grad():
            xp = torch.nn.functional.pad(x, (ctx, 0))
            outs, state = [], None
            for i in range(ctx, xp.shape[1], n):
                out = br.encoder(br.stft(xp[:, i - ctx:i + n])).squeeze(-1)
                state = rnn(out) if state is None else rnn(out, state)
                outs.append(head(state[0].unsqueeze(-1)))
            probs = torch.cat(outs, dim=2).squeeze(1)
            loss = (crit(probs, targets) * masks).mean()
            opt.zero_grad()
            loss.backward()
            opt.step()
            loss.item()
    return timed(step, steps, warmup=1)


def python_thresholds(all_predicts, all_gts):
    """The reference's calculate_best_thresholds loop (accuracy = fraction of equal labels)."""
    best = 0
    for enter in np.linspace(0, 1, 20):
        for ex in np.linspace(0, 1, 20):
            if ex >= enter:
                continue
            accs = []
            for pr, gt in zip(all_predicts, all_gts):
                s, pb = False, []
                for v in pr:
                    if v >= enter:
                        s = True
                    elif v <= ex:
                        s = False
                    pb.append(1 if s else 0)
                accs.append(round(sum(a == b for a, b in zip(gt, pb)) / len(pb), 4))
            best = max(best, round(np.mean(accs), 3))
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--ref-steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "tune_bench needs a GPU"
    name, pl = card()
    res = {"bench": "decoder fine-tuning", "gpu": name, "power_limit": pl, "B": 128, "T": 250, "steps": a.steps}
    model = SileroVADB200(device=0)
    B, T = 128, 250
    L = _load_reference()
    for sr in (16000, 8000):
        n = 512 if sr == 16000 else 256
        g = torch.Generator().manual_seed(sr)
        x = (torch.randn(B, T * n, generator=g) * 0.1).cuda()
        targets = torch.randint(0, 2, (B, T), generator=g).float().cuda()
        masks = torch.ones(B, T).cuda()
        dec = VADDecoderRNNJIT().cuda()
        dec.load_state_dict(decoder_state_dict(sr))
        dec.train()
        crit = nn.BCELoss(reduction="none")
        r = {}
        r["features_ms"] = timed(lambda: encoder_features(model, x, sr), a.steps)
        feat = encoder_features(model, x, sr)
        r["decoder_forward_ms"] = timed(lambda: dec(feat), a.steps)

        def fwd_bwd():
            loss = (crit(dec(feat), targets) * masks).mean()
            loss.backward()
        r["decoder_forward_backward_ms"] = timed(fwd_bwd, a.steps)
        r["decoder_backward_with_weight_grads_ms"] = r["decoder_forward_backward_ms"] - r["decoder_forward_ms"]
        # per-kernel device time of one forward + backward
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                fwd_bwd()
            torch.cuda.synchronize()
        kt = {}
        for ev in prof.key_averages():
            for k in ("dec_inproj", "dec_fwd", "dec_bwd", "dec_wgrad", "dec_reduce"):
                if k + "<" in ev.key or ev.key.startswith("svad::" + k + "(") or (k in ev.key and "svad" in ev.key):
                    kt[k] = kt.get(k, 0.0) + ev.device_time_total / 1e3 / 5
        r["kernel_ms"] = {k: round(v, 4) for k, v in kt.items()}
        opt = torch.optim.Adam(dec.parameters(), lr=5e-4)
        loader = [(x, targets, masks)]
        r["train_step_adam_ms"] = timed(lambda: train(_Cfg(sr == 8000), loader, model, dec, crit, opt, "cuda"), a.steps)
        if L is not None:
            r["reference_train_step_adam_ms"] = reference_step(L, sr, x, targets, masks, a.ref_steps)
            r["speedup_train_step"] = r["reference_train_step_adam_ms"] / r["train_step_adam_ms"]
        else:
            r["reference_train_step_adam_ms"] = "not measured (baseline/_ref not staged)"
        res[str(sr)] = {k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()}
    # threshold search
    rng = np.random.default_rng(0)
    preds = [np.clip(np.cumsum(rng.normal(0, 0.2, 250)) % 2.0, 0, 1).astype(np.float32).tolist() for _ in range(1000)]
    gts = [rng.integers(0, 2, 250).astype(float).tolist() for _ in range(1000)]
    calculate_best_thresholds(preds[:10], gts[:10])
    t0 = time.perf_counter()
    calculate_best_thresholds(preds, gts)
    ours = (time.perf_counter() - t0) * 1e3
    sub = 20
    t0 = time.perf_counter()
    python_thresholds(preds[:sub], gts[:sub])
    ref_sub = (time.perf_counter() - t0) * 1e3
    res["thresholds"] = {"files": 1000, "chunks": 250, "ms": round(ours, 2), "python_loop_subset_files": sub,
                         "python_loop_subset_ms": round(ref_sub, 1), "python_loop_1000_files_ms_extrapolated": round(ref_sub * 1000 / sub, 0)}
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


def _load_reference():
    p = REPO / "baseline" / "_ref" / "silero_vad" / "data" / "silero_vad.jit"
    if not p.exists():
        return None
    m = torch.jit.load(str(p), map_location="cuda")
    m.eval()
    return m


if __name__ == "__main__":
    main()
