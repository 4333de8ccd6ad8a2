"""Fine-tuning the VAD decoder on labelled audio, on the GPU.

Mirrors the reference's tuning/utils.py (train, validate, predict, calculate_best_thresholds, VADDecoderRNNJIT) with the engine in
place of the TorchScript module:

    model = SileroVADB200()                                    # frozen STFT + encoder (fp32 kernel in features mode)
    decoder = VADDecoderRNNJIT().cuda()
    decoder.load_state_dict(decoder_state_dict(16000))         # the stock decoder of the 16 kHz branch
    optimizer = torch.optim.Adam(decoder.parameters(), lr=5e-4)
    criterion = torch.nn.BCELoss(reduction="none")
    train(config, train_loader, model, decoder, criterion, optimizer, "cuda")     # config needs only .tune_8k
    val_loss, val_roc = validate(config, val_loader, model, decoder, criterion, "cuda")
    save_tuned("tuned.weights", decoder, 16000)                # stock container with this branch's decoder replaced
    tuned = SileroVADB200(weights="tuned.weights")             # every inference entry point runs the tuned decoder
    enter, exit_, acc = calculate_best_thresholds(*predict(tuned, val_loader, "cuda", 16000))

Batches are the reference's (x [B, L], targets [B, T], masks [B, T]) with L = T * n (n = 512 at 16 kHz, 256 at 8 kHz), as its
dataset pads them.  The loss stays in torch, so any criterion or optimizer works; the decoder's forward and backward passes are
CUDA kernels (csrc/svad_train.cuh) reached through a torch.autograd.Function.
"""
import struct
from collections import OrderedDict
from pathlib import Path

import numpy as np
import torch
import torch.nn as nn

from . import _cabi
from .model import WEIGHTS

DECODER_SHAPES = OrderedDict([("rnn.weight_ih", (512, 128)), ("rnn.weight_hh", (512, 128)), ("rnn.bias_ih", (512,)),
                              ("rnn.bias_hh", (512,)), ("decoder.2.weight", (1, 128, 1)), ("decoder.2.bias", (1,))])
_ENGINES = {}


def _branch(sr):
    if sr not in (8000, 16000):
        raise ValueError(f"Supported sampling rates: [8000, 16000] (got {sr})")
    return "_model" if sr == 16000 else "_model_8k"


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream(device):
    return torch.cuda.current_stream(device).cuda_stream


def _engine(device):
    """Engine used by the decoder kernels of a device (they take every parameter from the caller; the engine supplies the
    device and its SM count)."""
    idx = torch.device(device).index
    idx = torch.cuda.current_device() if idx is None else idx
    if idx not in _ENGINES:
        _ENGINES[idx] = _cabi.Engine(WEIGHTS, idx)
    return _ENGINES[idx]


# ---------------------------------------------------------------------------------------------------------------- containers
def read_container(path):
    """SVADW001 container -> OrderedDict name -> float32 CPU tensor, in file order."""
    out = OrderedDict()
    with open(path, "rb") as f:
        if f.read(8) != b"SVADW001":
            raise ValueError(f"{path}: not an SVADW001 weight container")
        (n,) = struct.unpack("<I", f.read(4))
        for _ in range(n):
            (ln,) = struct.unpack("<I", f.read(4))
            name = f.read(ln).decode()
            (nd,) = struct.unpack("<I", f.read(4))
            dims = struct.unpack("<%dI" % nd, f.read(4 * nd))
            cnt = int(np.prod(dims)) if nd else 1
            data = np.frombuffer(f.read(4 * cnt), dtype="<f4")
            if data.size != cnt:
                raise ValueError(f"{path}: truncated tensor {name}")
            out[name] = torch.from_numpy(data.astype(np.float32).reshape(dims))
    return out


def write_container(path, tensors):
    """magic[8] | u32 n | n x { u32 name_len | name | u32 ndim | u32 dims[ndim] | f32 data }.  `tensors`: (name, tensor) pairs
    or a mapping."""
    items = list(tensors.items()) if hasattr(tensors, "items") else list(tensors)
    with open(path, "wb") as f:
        f.write(b"SVADW001")
        f.write(struct.pack("<I", len(items)))
        for name, t in items:
            t = torch.as_tensor(t).detach().to("cpu", torch.float32)
            nb = name.encode()
            f.write(struct.pack("<I", len(nb)))
            f.write(nb)
            f.write(struct.pack("<I", t.dim()))
            f.write(struct.pack("<%dI" % t.dim(), *t.shape))
            f.write(t.contiguous().numpy().astype("<f4").tobytes())


def decoder_state_dict(sr, weights=None):
    """The six decoder tensors of one branch of a container, keyed as VADDecoderRNNJIT's state dict."""
    tm = read_container(weights or WEIGHTS)
    pre = _branch(sr) + ".decoder."
    try:
        return OrderedDict((k, tm[pre + k].clone()) for k in DECODER_SHAPES)
    except KeyError as ex:
        raise ValueError(f"container has no tensor {ex.args[0]}") from None


def save_tuned(path, decoder, sr, base=None):
    """Write the `base` container (default: the stock weights) with the decoder of branch `sr` replaced by `decoder`'s."""
    tm = read_container(base or WEIGHTS)
    sd = decoder.state_dict() if hasattr(decoder, "state_dict") else decoder
    pre = _branch(sr) + ".decoder."
    for k, shape in DECODER_SHAPES.items():
        if k not in sd:
            raise ValueError(f"decoder state has no {k}")
        t = sd[k].detach().to("cpu", torch.float32)
        if tuple(t.shape) != shape:
            raise ValueError(f"{k}: expected shape {shape}, got {tuple(t.shape)}")
        tm[pre + k] = t
    write_container(path, tm)
    return Path(path)


def export_weights(src, path):
    """Convert a TorchScript model file (such as the reference's tune.py saves), a torch.save'd state dict, or a state-dict mapping
    with the reference's keys into a container for SileroVADB200(weights=path).  The STFT basis buffers are dropped (the engine
    computes the STFT itself); every other key of the stock container must be present with its stock shape."""
    if hasattr(src, "items"):
        sd = src
    elif hasattr(src, "state_dict"):
        sd = src.state_dict()
    else:
        try:
            sd = torch.jit.load(str(src), map_location="cpu").state_dict()
        except RuntimeError:
            sd = torch.load(str(src), map_location="cpu")
    stock = read_container(WEIGHTS)
    keys = {k for k in sd if "forward_basis_buffer" not in k}
    if keys != set(stock):
        missing, extra = sorted(set(stock) - keys), sorted(keys - set(stock))
        raise ValueError(f"state dict does not match the model: missing {missing}, unexpected {extra}")
    out = OrderedDict()
    for k, ref in stock.items():
        t = sd[k].detach().to("cpu", torch.float32)
        if t.shape != ref.shape:
            raise ValueError(f"{k}: expected shape {tuple(ref.shape)}, got {tuple(t.shape)}")
        out[k] = t
    write_container(path, out)
    return Path(path)


# ---------------------------------------------------------------------------------------------------------------- features
def _segments(B, T, sms):
    """Chunks per segment S: the B streams are cut into B * ceil(T / S) rows so that the fp32 tile kernel (up to 32 rows per
    CTA, one CTA per SM) gets about one full wave of tiles instead of ceil(B / 32)."""
    nseg = max(1, min(T, -(-32 * sms // max(B, 1))))
    return -(-T // nseg)


def _features(engine, device, x, sr, S):
    n, ctx = (512, 64) if sr == 16000 else (256, 32)
    B, L = x.shape
    T = L // n
    nseg = -(-T // S)
    with torch.cuda.device(device):
        if nseg == 1 and S == T:
            xp, cx = x, None
        else:
            xp = torch.zeros(B, nseg * S * n, device=device)
            xp[:, :L] = x
            cx = torch.zeros(B, nseg, ctx, device=device)
            cx[:, 1:] = xp.view(B, nseg, S * n)[:, :-1, -ctx:]
        feat = torch.empty(B, nseg * S, 128, device=device)
        engine.features_device(sr, B * nseg, S * n, S * n, _ptr(xp), _ptr(cx), _ptr(feat), _stream(device))
    return feat if nseg * S == T else feat[:, :T].contiguous()


def encoder_features(model, x, sr):
    """Frozen STFT + encoder of `model` (a SileroVADB200) on fp32 audio x [B, L] (or [L]), L a multiple of the chunk size ->
    f32 [B, L / n, 128] on the model's device: the post-ReLU encoder output that the decoder's LSTM cell reads at each chunk,
    exactly as the reference's training loop computes it (pad(x, (ctx, 0)), windows of ctx + n)."""
    _branch(sr)
    n = 512 if sr == 16000 else 256
    x = torch.as_tensor(x)
    if x.dim() == 1:
        x = x.unsqueeze(0)
    if x.dim() != 2 or x.dtype != torch.float32:
        raise ValueError("encoder_features takes float32 audio [B, L]")
    if x.shape[1] == 0 or x.shape[1] % n:
        raise ValueError(f"audio length must be a positive multiple of {n} samples at {sr} Hz (got {x.shape[1]})")
    x = x.detach().to(model.device, torch.float32).contiguous()
    B, T = x.shape[0], x.shape[1] // n
    return _features(model.engine, model.device, x, sr, _segments(B, T, model.engine.sm_count))


# ---------------------------------------------------------------------------------------------------------------- decoder
class _DecoderScan(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, w_ih, w_hh, b_ih, b_hh, w_head, b_head, drop):
        B, T, _ = feat.shape
        dev = feat.device
        eng = _engine(dev)
        feat, w_ih, w_hh, b_ih, b_hh, w_head, b_head = (t.detach().contiguous() for t in (feat, w_ih, w_hh, b_ih, b_hh, w_head, b_head))
        need = any(ctx.needs_input_grad[1:7])
        L = _cabi.lib()
        with torch.cuda.device(dev):
            probs = torch.empty(B, T, device=dev)
            work = torch.empty(max(1, L.svad_decoder_workspace_bytes(B, T, 0)), dtype=torch.uint8, device=dev)
            tape = torch.empty(L.svad_decoder_tape_floats(B, T), device=dev) if need else None
            eng.decoder_forward_device(B, T, _ptr(feat), _ptr(w_ih), _ptr(w_hh), _ptr(b_ih), _ptr(b_hh), _ptr(w_head), _ptr(b_head),
                                       _ptr(drop), _ptr(probs), _ptr(tape), _ptr(work), _stream(dev))
        if need:
            ctx.save_for_backward(feat, w_hh, w_head, drop, probs, tape)
        return probs

    @staticmethod
    def backward(ctx, dprobs):
        feat, w_hh, w_head, drop, probs, tape = ctx.saved_tensors
        B, T, _ = feat.shape
        dev = feat.device
        dprobs = dprobs.detach().to(torch.float32).contiguous()
        with torch.cuda.device(dev):
            work = torch.empty(_cabi.lib().svad_decoder_workspace_bytes(B, T, 1), dtype=torch.uint8, device=dev)
            dw_ih = torch.empty(512, 128, device=dev)
            dw_hh = torch.empty(512, 128, device=dev)
            db = torch.empty(512, device=dev)
            dw_head = torch.empty(1, 128, 1, device=dev)
            db_head = torch.empty(1, device=dev)
            _engine(dev).decoder_backward_device(B, T, _ptr(feat), _ptr(w_hh), _ptr(w_head), _ptr(drop), _ptr(probs), _ptr(dprobs), _ptr(tape),
                                                 _ptr(work), _ptr(dw_ih), _ptr(dw_hh), _ptr(db), _ptr(dw_head), _ptr(db_head), _stream(dev))
        return None, dw_ih, dw_hh, db, db.clone(), dw_head, db_head, None


def decoder_scan(feat, w_ih, w_hh, b_ih, b_hh, w_head, b_head, drop=None):
    """probs [B, T] of the decoder over features [B, T, 128] from zero state (differentiable in the six parameters).
    drop: None or the f32 [B, T, 128] dropout multiplier of the head path."""
    if feat.dim() != 3 or feat.shape[2] != 128 or feat.dtype != torch.float32 or not feat.is_cuda:
        raise ValueError("decoder features must be a float32 CUDA tensor [B, T, 128]")
    params = (w_ih, w_hh, b_ih, b_hh, w_head, b_head)
    for p, shape in zip(params, DECODER_SHAPES.values()):
        if tuple(p.shape) != shape or p.dtype != torch.float32 or p.device != feat.device:
            raise ValueError(f"decoder parameter: expected float32 {shape} on {feat.device}, got {p.dtype} {tuple(p.shape)} on {p.device}")
    if drop is not None:
        if tuple(drop.shape) != tuple(feat.shape) or drop.dtype != torch.float32 or drop.device != feat.device:
            raise ValueError("dropout multiplier must be float32 like the features")
        drop = drop.detach().contiguous()
    return _DecoderScan.apply(feat, *params, drop)


class VADDecoderRNNJIT(nn.Module):
    """The reference's decoder module (tuning/utils.py): same submodules and parameter names, so state dicts move both ways.
    forward(feat [B, T, 128]) -> probs [B, T] runs the whole sequence from zero state on the GPU; in train() mode the head's
    Dropout(0.1) draws its mask with torch's generator on the device."""

    def __init__(self):
        super().__init__()
        self.rnn = nn.LSTMCell(128, 128)
        self.decoder = nn.Sequential(nn.Dropout(0.1), nn.ReLU(), nn.Conv1d(128, 1, kernel_size=1), nn.Sigmoid())

    def forward(self, feat):
        p = self.decoder[0].p
        drop = None
        if self.training and p > 0:
            drop = torch.empty_like(feat).bernoulli_(1.0 - p).div_(1.0 - p) if p < 1 else torch.zeros_like(feat)
        conv = self.decoder[2]
        return decoder_scan(feat, self.rnn.weight_ih, self.rnn.weight_hh, self.rnn.bias_ih, self.rnn.bias_hh, conv.weight, conv.bias, drop)


# ---------------------------------------------------------------------------------------------------------------- loops
class _Mean:
    def __init__(self):
        self.sum, self.count = 0.0, 0

    def update(self, val, n):
        self.sum += val * n
        self.count += n

    @property
    def avg(self):
        return self.sum / self.count if self.count else 0.0


def train(config, loader, model, decoder, criterion, optimizer, device):
    """One epoch (tuning/utils.py:206-249): features of every batch from the frozen encoder, decoder forward / backward on the
    GPU, loss (criterion(probs, targets) * masks).mean() in torch.  Returns the mean loss weighted by masks.numel()."""
    sr = 8000 if config.tune_8k else 16000
    losses = _Mean()
    decoder.train()
    with torch.enable_grad():
        for x, targets, masks in loader:
            targets, masks = targets.to(device), masks.to(device)
            feat = encoder_features(model, x, sr)
            probs = decoder(feat)
            loss = (criterion(probs, targets) * masks).mean()
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            losses.update(loss.item(), masks.numel())
    return losses.avg


def roc_auc(scores, labels):
    """ROC AUC from average ranks (ties share their mean rank), computed on the tensors' device in float64; equals
    sklearn.metrics.roc_auc_score for binary labels.  Raises ValueError when only one class is present, as sklearn does."""
    scores = torch.as_tensor(scores).to(torch.float64).flatten()
    labels = torch.as_tensor(labels, device=scores.device).flatten()
    srt, order = torch.sort(scores, stable=True)
    _, inv, counts = torch.unique_consecutive(srt, return_inverse=True, return_counts=True)
    ends = torch.cumsum(counts, 0).to(torch.float64)
    mean_rank = ends - (counts.to(torch.float64) - 1.0) / 2.0   # 1-based ranks start+1 .. end
    pos = labels[order] == 1
    n_pos = int(pos.sum())
    n_neg = scores.numel() - n_pos
    if n_pos == 0 or n_neg == 0:
        raise ValueError("Only one class present in y_true. ROC AUC score is not defined in that case.")
    r = float(mean_rank[inv][pos].sum())
    return (r - n_pos * (n_pos + 1) / 2.0) / (n_pos * n_neg)


def validate(config, loader, model, decoder, criterion, device):
    """tuning/utils.py:252-298: mean masked loss and round(ROC AUC, 3) over the chunks whose mask is non-zero."""
    sr = 8000 if config.tune_8k else 16000
    losses = _Mean()
    decoder.eval()
    preds, gts = [], []
    with torch.no_grad():
        for x, targets, masks in loader:
            targets, masks = targets.to(device), masks.to(device)
            probs = decoder(encoder_features(model, x, sr))
            keep = masks != 0
            preds.append(probs[keep])
            gts.append(targets[keep])
            loss = (criterion(probs, targets) * masks).mean()
            losses.update(loss.item(), masks.numel())
    score = roc_auc(torch.cat(preds), torch.cat(gts))
    return losses.avg, round(score, 3)


def predict(model, loader, device, sr):
    """tuning/utils.py:309-323: per file, the probabilities and targets of the chunks whose mask is non-zero (Python lists)."""
    all_predicts, all_gts = [], []
    with torch.no_grad():
        for x, targets, masks in loader:
            out = model.audio_forward(x, sr=sr)
            for i, out_chunk in enumerate(out):
                all_predicts.append(out_chunk[masks[i] != 0].cpu().tolist())
                all_gts.append(targets[i, masks[i] != 0].cpu().tolist())
    return all_predicts, all_gts


def calculate_best_thresholds(all_predicts, all_gts, device=None):
    """tuning/utils.py:326-356 with the 190 x files x chunks hysteresis scans in one kernel launch (integer match counts); the
    per-file rounding, the mean and the first-strictly-greater selection run here in the reference's order and arithmetic.
    Returns (enter, exit, accuracy).  Raises ValueError for empty input or when no pair has an accuracy above 0."""
    if len(all_predicts) == 0:
        raise ValueError("no predictions")
    if len(all_predicts) != len(all_gts) or any(len(p) != len(g) for p, g in zip(all_predicts, all_gts)):
        raise ValueError("predictions and targets differ in length")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    lens = [len(p) for p in all_predicts]
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    grid = np.linspace(0, 1, 20)
    with torch.cuda.device(dev):
        probs = torch.tensor([v for p in all_predicts for v in p], dtype=torch.float32).to(dev)
        gts = torch.tensor([v for g in all_gts for v in g], dtype=torch.float32).to(dev)
        if probs.numel() == 0:
            probs = gts = torch.zeros(1, device=dev)
        d_offs = torch.from_numpy(offs).to(dev)
        d_grid = torch.from_numpy(grid).to(dev)
        counts = torch.empty(len(lens), 190, dtype=torch.int64, device=dev)
        _cabi.check(_cabi.lib().svad_threshold_grid_device(_ptr(probs), _ptr(gts), _ptr(d_offs), len(lens), _ptr(d_grid), _ptr(counts),
                                                           _stream(dev)))
        counts = counts.cpu().tolist()
    best_acc, best = 0, None
    p = 0
    for a, ths_enter in enumerate(grid):
        for e, ths_exit in enumerate(grid):
            if ths_exit >= ths_enter:
                continue
            accs = [round(c[p] / n, 4) if n else float("nan") for c, n in zip(counts, lens)]
            mean_acc = round(np.mean(accs), 3)
            if mean_acc > best_acc:
                best_acc = mean_acc
                best = (round(ths_enter, 2), round(ths_exit, 2))
            p += 1
    if best is None:
        raise ValueError("no threshold pair reaches an accuracy above 0")
    return best[0], best[1], best_acc
