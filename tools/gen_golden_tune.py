#!/usr/bin/env python
"""Decoder fine-tuning fixtures (tests/golden/tune.npz, tune.json), generated from the REFERENCE TorchScript model (needs the
reference package, silero_vad, importable from /root/reference/src; CPU only).

Per rate (16 kHz from test16k, 8 kHz from aepyx8k; audio = pcm / 32768):
  f{sr}_feat  [2, 64, 128]       reference features of two clips of 64 chunks cut from the fixture at the sample offsets
                                 tune.json["f{sr}_offsets"]: pad(x, (ctx, 0)), windows of ctx + n, _model[_8k].stft -> .encoder
                                 (tuning/utils.py:224-235)
  g{sr}_targets / g{sr}_masks    seeded targets (0 / 1) and masks ({0, 0.5, 1})
  g{sr}_loss, g{sr}_<param>      (BCE(probs, targets) * masks).mean() and its gradients through nn.LSTMCell + head loaded from the
                                 reference decoder's state dict, eval mode (no dropout).  The biases and the head are stored whole;
                                 the two [512, 128] weight gradients as row sums, column sums and Frobenius norm (float64), which
                                 keeps the fixture small (the GPU tests also compare whole matrices with a float64 nn.LSTMCell twin)
  t{sr}_probs                    audio_forward of the reference model with a "tuned" decoder swapped in (as tune.py:60-63 does) on
                                 the whole fixture; tune.json holds its get_speech_timestamps.  The tuned decoder is not stored: it is
                                 tuned_decoder(stock, sr), seeded perturbations of the stock tensors with numpy's RandomState
                                 (a stream numpy keeps fixed across versions); tune.json["t{sr}_abs_sum"] checks the recomputation.
"""
import json
import sys
from pathlib import Path

import numpy as np
import torch
import torch.nn as nn

REPO = Path(__file__).resolve().parents[1]
REF = Path("/root/reference")
OUT = REPO / "tests" / "golden"

PARAMS = ["rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh", "decoder.2.weight", "decoder.2.bias"]


def key(p):
    return p.replace(".", "_")


def tuned_decoder(stock, sr):
    """name -> float32 array: stock + 0.05 * mean|stock| * N(0, 1) per tensor, the noise from RandomState(1000 + sr + i)."""
    out = {}
    for i, p in enumerate(PARAMS):
        base = np.asarray(stock[p], np.float32)
        scale = np.float32(0.05 * float(np.abs(base.astype(np.float64)).mean()))
        noise = np.random.RandomState(1000 + sr + i).standard_normal(base.shape).astype(np.float32)
        out[p] = (base + scale * noise).astype(np.float32)
    return out


def abs_sum(tensors):
    return float(sum(np.abs(np.asarray(tensors[p], np.float64)).sum() for p in PARAMS))


def fingerprint(g):
    g = np.asarray(g, np.float64)
    return g.sum(axis=1), g.sum(axis=0), np.array(np.linalg.norm(g))


class Decoder(nn.Module):   # the reference's VADDecoderRNNJIT parameters (tuning/utils.py:149-172), run over a whole sequence
    def __init__(self):
        super().__init__()
        self.rnn = nn.LSTMCell(128, 128)
        self.decoder = nn.Sequential(nn.Dropout(0.1), nn.ReLU(), nn.Conv1d(128, 1, kernel_size=1), nn.Sigmoid())

    def forward(self, feat):
        h = c = torch.zeros(feat.shape[0], 128, dtype=feat.dtype)
        out = []
        for t in range(feat.shape[1]):
            h, c = self.rnn(feat[:, t], (h, c))
            out.append(self.decoder(h.unsqueeze(-1)).squeeze(-1))
        return torch.cat(out, 1)


def features(branch, x, ctx, n):
    x = torch.nn.functional.pad(torch.from_numpy(x), (ctx, 0))
    outs = []
    with torch.no_grad():
        for i in range(ctx, x.shape[1], n):
            outs.append(branch.encoder(branch.stft(x[:, i - ctx:i + n])).squeeze(-1))
    return torch.stack(outs, 1).numpy()


def main():
    sys.path.insert(0, str(REF / "src"))
    torch.set_num_threads(4)
    from silero_vad import get_speech_timestamps, load_silero_vad
    model = load_silero_vad(onnx=False)
    out, meta = {}, {}
    for sr, name, offs in ((16000, "test16k", (48000, 480000)), (8000, "aepyx8k", (16000, 800000))):
        n, ctx = (512, 64) if sr == 16000 else (256, 32)
        branch = model._model if sr == 16000 else model._model_8k
        pcm = np.load(OUT / f"{name}.npz")["pcm"]
        audio = pcm.astype(np.float32) / 32768.0
        clips = np.stack([audio[o:o + 64 * n] for o in offs]).copy()
        feat = features(branch, clips, ctx, n)
        out[f"f{sr}_feat"] = feat
        meta[f"f{sr}_offsets"] = list(offs)
        # loss and gradients of the stock decoder (eval mode)
        rng = np.random.default_rng(sr)
        targets = rng.integers(0, 2, (2, 64)).astype(np.float32)
        masks = rng.choice(np.array([0.0, 0.5, 1.0], np.float32), (2, 64))
        dec = Decoder()
        dec.load_state_dict(branch.decoder.state_dict())
        dec.eval()
        probs = dec(torch.from_numpy(feat))
        loss = (nn.BCELoss(reduction="none")(probs, torch.from_numpy(targets)) * torch.from_numpy(masks)).mean()
        loss.backward()
        out[f"g{sr}_targets"], out[f"g{sr}_masks"] = targets, masks
        out[f"g{sr}_loss"] = np.float64(loss.item())
        out[f"g{sr}_probs"] = probs.detach().numpy()
        for p, prm in dec.named_parameters():
            g = prm.grad.numpy().copy()
            if g.shape == (512, 128):
                out[f"g{sr}_{key(p)}_rowsum"], out[f"g{sr}_{key(p)}_colsum"], out[f"g{sr}_{key(p)}_norm"] = fingerprint(g)
            else:
                out[f"g{sr}_{key(p)}"] = g
        # a tuned decoder: seeded perturbations swapped into the reference model
        sd = {k: v.clone() for k, v in branch.decoder.state_dict().items()}
        tuned = {p: torch.from_numpy(v) for p, v in tuned_decoder({p: sd[p].numpy() for p in PARAMS}, sr).items()}
        branch.decoder.load_state_dict(tuned)
        with torch.no_grad():
            tp = model.audio_forward(torch.from_numpy(audio), sr=sr)[0].numpy()
        model.reset_states()
        segs = get_speech_timestamps(torch.from_numpy(audio), model, sampling_rate=sr)
        branch.decoder.load_state_dict(sd)
        model.reset_states()
        meta[f"t{sr}_abs_sum"] = abs_sum({p: tuned[p].numpy() for p in PARAMS})
        out[f"t{sr}_probs"] = tp
        meta[f"t{sr}_segments"] = [[int(d["start"]), int(d["end"])] for d in segs]
        meta[f"t{sr}_fixture"] = name
        print(sr, "feat", feat.shape, "loss", loss.item(), "tuned segments", len(segs))
    np.savez_compressed(OUT / "tune.npz", **out)
    (OUT / "tune.json").write_text(json.dumps(meta, indent=1) + "\n")


if __name__ == "__main__":
    main()
