"""Decoder fine-tuning on the B200: encoder features, decoder forward / backward kernels against torch autograd, one training step,
validation AUC, tuned-weight round trip through every inference kernel, and the threshold-grid kernel."""
import importlib.util
import json

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import GOLDEN, REPO

pytestmark = pytest.mark.gpu
TOL = 1e-4
PARAM_NAMES = ["rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh", "decoder.2.weight", "decoder.2.bias"]


@pytest.fixture(scope="module")
def tune():
    return dict(np.load(GOLDEN / "tune.npz")), json.loads((GOLDEN / "tune.json").read_text())


@pytest.fixture(scope="module")
def model():
    from silero_vad_b200 import SileroVADB200
    return SileroVADB200(device=0)


def tuned_state_dict(sr, meta):
    """The seeded "tuned" decoder of the fixtures, recomputed by tools/gen_golden_tune.py's recipe and checked against its sum."""
    from silero_vad_b200 import decoder_state_dict
    spec = importlib.util.spec_from_file_location("gen_golden_tune", REPO / "tools" / "gen_golden_tune.py")
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    tuned = gen.tuned_decoder({k: v.numpy() for k, v in decoder_state_dict(sr).items()}, sr)
    assert gen.abs_sum(tuned) == meta[f"t{sr}_abs_sum"]
    return {k: torch.from_numpy(v) for k, v in tuned.items()}


def clips(fixtures, meta, sr):
    n = 512 if sr == 16000 else 256
    a = fixtures["test16k" if sr == 16000 else "aepyx8k"]["audio"]
    return np.stack([a[o:o + 64 * n] for o in meta[f"f{sr}_offsets"]]).copy()


class Twin(nn.Module):   # the reference decoder over a whole sequence (nn.LSTMCell + head), any dtype
    def __init__(self, sd, dtype):
        super().__init__()
        self.rnn = nn.LSTMCell(128, 128)
        self.decoder = nn.Sequential(nn.Dropout(0.0), nn.ReLU(), nn.Conv1d(128, 1, kernel_size=1), nn.Sigmoid())
        self.load_state_dict(sd)
        self.to("cuda", dtype)

    def forward(self, feat, drop=None):
        B, T, _ = feat.shape
        h = c = torch.zeros(B, 128, dtype=feat.dtype, device=feat.device)
        out = []
        for t in range(T):
            h, c = self.rnn(feat[:, t], (h, c))
            z = h if drop is None else h * drop[:, t]
            out.append(self.decoder(z.unsqueeze(-1)).squeeze(-1))
        return torch.cat(out, 1)


@pytest.mark.parametrize("sr", [16000, 8000])
def test_features_match_reference(model, tune, fixtures, sr):
    from silero_vad_b200 import encoder_features
    z, meta = tune
    feat = encoder_features(model, torch.from_numpy(clips(fixtures, meta, sr)), sr).cpu().numpy()
    err = float(np.abs(feat - z[f"f{sr}_feat"]).max())
    print(f"sr={sr}: max|feat_gpu - feat_ref| = {err:.3e}")
    assert err <= 1e-4


@pytest.mark.parametrize("B", [1, 3, 129])
@pytest.mark.parametrize("T", [1, 17, 250])
def test_features_segmented_equal_whole_stream(model, fixtures, B, T):
    from silero_vad_b200 import encoder_features, tuning
    for sr, name in ((16000, "test16k"), (8000, "aepyx8k")):
        n = 512 if sr == 16000 else 256
        a = fixtures[name]["audio"]
        x = torch.from_numpy(np.stack([a[(997 * b) % (len(a) - T * n):][: T * n] for b in range(B)]).copy())
        got = encoder_features(model, x, sr)
        assert got.shape == (B, T, 128)
        whole = tuning._features(model.engine, model.device, x.cuda(), sr, T)
        assert torch.equal(got, whole), (sr, B, T)
    with pytest.raises(ValueError):
        encoder_features(model, torch.zeros(2, 500), 16000)


@pytest.mark.parametrize("sr,name", [(16000, "test16k"), (8000, "aepyx8k")])
def test_stock_decoder_on_fixture_features(model, fixtures, sr, name):
    from silero_vad_b200 import VADDecoderRNNJIT, decoder_state_dict, encoder_features
    fx = fixtures[name]
    n = 512 if sr == 16000 else 256
    a = fx["audio"]
    x = torch.from_numpy(np.pad(a, (0, (-len(a)) % n)))
    dec = VADDecoderRNNJIT().cuda().eval()
    dec.load_state_dict(decoder_state_dict(sr))
    with torch.no_grad():
        p = dec(encoder_features(model, x, sr)).cpu().numpy()[0]
    ref = fx["probs"]
    err_ref = float(np.abs(p - ref).max())
    model.engine.set_kernel(0)
    model.engine.set_small_batch_max(0)
    try:
        af = model.audio_forward(torch.from_numpy(a), sr).numpy()[0]
    finally:
        model.engine.set_kernel(2)
        model.engine.set_small_batch_max(256)
    err_k0 = float(np.abs(p - af).max())
    print(f"{name}: decoder kernels vs reference {err_ref:.3e}, vs audio_forward kernel 0 {err_k0:.3e}")
    assert err_ref < TOL and err_k0 < 2e-5


def _rand_params(seed):
    g = torch.Generator().manual_seed(seed)
    from silero_vad_b200 import decoder_state_dict
    sd = decoder_state_dict(16000)
    return {k: v + 0.05 * v.abs().mean() * torch.randn(v.shape, generator=g) for k, v in sd.items()}


@pytest.mark.parametrize("B,T", [(5, 40), (200, 9), (300, 6)])
def test_forward_backward_against_float64_autograd(B, T):
    from silero_vad_b200 import VADDecoderRNNJIT
    torch.manual_seed(B)
    sd = _rand_params(B)
    feat = torch.relu(torch.randn(B, T, 128, device="cuda"))
    drop = (torch.rand(B, T, 128, device="cuda") >= 0.1).float() / 0.9
    targets = torch.randint(0, 2, (B, T), device="cuda").float()
    masks = torch.tensor([0.0, 0.5, 1.0], device="cuda")[torch.randint(0, 3, (B, T), device="cuda")]
    dec = VADDecoderRNNJIT().cuda()
    dec.load_state_dict(sd)
    from silero_vad_b200.tuning import decoder_scan
    conv = dec.decoder[2]
    params = [dec.rnn.weight_ih, dec.rnn.weight_hh, dec.rnn.bias_ih, dec.rnn.bias_hh, conv.weight, conv.bias]

    def run():
        for p in params:
            p.grad = None
        probs = decoder_scan(feat, *params, drop)
        loss = (nn.functional.binary_cross_entropy(probs, targets, reduction="none") * masks).mean()
        loss.backward()
        return probs.detach(), [p.grad.clone() for p in params]

    probs, grads = run()
    probs2, grads2 = run()
    assert torch.equal(probs, probs2)
    for g1, g2 in zip(grads, grads2):
        assert torch.equal(g1, g2)   # fixed-order reductions: bit-identical
    twin = Twin(sd, torch.float64)
    pt = twin(feat.double(), drop.double())
    lt = (nn.functional.binary_cross_entropy(pt, targets.double(), reduction="none") * masks.double()).mean()
    lt.backward()
    tg = [twin.rnn.weight_ih.grad, twin.rnn.weight_hh.grad, twin.rnn.bias_ih.grad, twin.rnn.bias_hh.grad, twin.decoder[2].weight.grad,
          twin.decoder[2].bias.grad]
    perr = float((probs.double() - pt.detach()).abs().max())
    print(f"B={B} T={T}: max|p - p64| = {perr:.3e}")
    assert perr < 1e-5
    for name, g, w in zip(PARAM_NAMES, grads, tg):
        rel = float((g.double() - w).norm() / w.norm())
        print(f"  {name}: relative Frobenius error {rel:.3e}")
        assert rel <= 1e-4, name


@pytest.mark.parametrize("sr", [16000, 8000])
def test_golden_loss_and_gradients(tune, sr):
    from silero_vad_b200 import VADDecoderRNNJIT, decoder_state_dict
    z, _ = tune
    dec = VADDecoderRNNJIT().cuda().eval()
    dec.load_state_dict(decoder_state_dict(sr))
    probs = dec(torch.from_numpy(z[f"f{sr}_feat"]).cuda())
    t, m = torch.from_numpy(z[f"g{sr}_targets"]).cuda(), torch.from_numpy(z[f"g{sr}_masks"]).cuda()
    loss = (nn.BCELoss(reduction="none")(probs, t) * m).mean()
    loss.backward()
    assert abs(loss.item() - float(z[f"g{sr}_loss"])) <= 1e-4 * abs(float(z[f"g{sr}_loss"]))
    for name, p in dec.named_parameters():
        key, g = f"g{sr}_{name.replace('.', '_')}", p.grad.cpu().double().numpy()
        if g.shape == (512, 128):   # stored as row sums, column sums and Frobenius norm
            for got, want in ((g.sum(axis=1), z[key + "_rowsum"]), (g.sum(axis=0), z[key + "_colsum"])):
                rel = float(np.linalg.norm(got - want) / np.linalg.norm(want))
                assert rel <= 1e-4, (name, rel)
            assert abs(np.linalg.norm(g) - float(z[key + "_norm"])) <= 1e-4 * float(z[key + "_norm"]), name
        else:
            want = z[key]
            rel = float(np.linalg.norm(g - want) / np.linalg.norm(want))
            assert rel <= 1e-4, (name, rel)


class _Cfg:
    def __init__(self, tune_8k):
        self.tune_8k = tune_8k


def _loader(fixtures, sr, B=6, T=32, seed=0):
    n = 512 if sr == 16000 else 256
    a = fixtures["test16k" if sr == 16000 else "aepyx8k"]["audio"]
    rng = np.random.default_rng(seed)
    x = torch.from_numpy(np.stack([a[o:o + T * n] for o in rng.integers(0, len(a) - T * n, B)]).copy())
    targets = torch.from_numpy(rng.integers(0, 2, (B, T)).astype(np.float32))
    masks = torch.from_numpy(rng.choice(np.array([0.0, 0.5, 1.0], np.float32), (B, T)))
    return [(x, targets, masks)]


@pytest.mark.parametrize("sr", [16000, 8000])
def test_train_step_with_sgd_matches_torch_twin(model, fixtures, sr):
    from silero_vad_b200 import VADDecoderRNNJIT, decoder_state_dict, encoder_features, train
    loader = _loader(fixtures, sr)
    dec = VADDecoderRNNJIT().cuda()
    dec.load_state_dict(decoder_state_dict(sr))
    dec.decoder[0].p = 0.0   # deterministic step: the twin runs without dropout too
    opt = torch.optim.SGD(dec.parameters(), lr=0.5)
    crit = nn.BCELoss(reduction="none")
    loss = train(_Cfg(sr == 8000), loader, model, dec, crit, opt, "cuda")
    twin = Twin(decoder_state_dict(sr), torch.float64)
    x, t, m = loader[0]
    feat = encoder_features(model, x, sr).double()
    lt = (nn.BCELoss(reduction="none")(twin(feat), t.cuda().double()) * m.cuda().double()).mean()
    topt = torch.optim.SGD(twin.parameters(), lr=0.5)
    topt.zero_grad()
    lt.backward()
    topt.step()
    assert abs(loss - lt.item()) <= 1e-4 * abs(lt.item())   # torch's float32 BCE vs float64
    tsd = twin.state_dict()
    for k, v in dec.state_dict().items():
        err = float((v.double() - tsd[k]).abs().max())
        assert err <= 1e-6, (k, err)


def test_validate_auc_equals_sklearn(model, fixtures):
    from silero_vad_b200 import VADDecoderRNNJIT, decoder_state_dict, encoder_features, validate
    from silero_vad_b200.tuning import roc_auc
    loader = _loader(fixtures, 16000, B=8, T=40, seed=3)
    dec = VADDecoderRNNJIT().cuda()
    dec.load_state_dict(decoder_state_dict(16000))
    loss, auc = validate(_Cfg(False), loader, model, dec, nn.BCELoss(reduction="none"), "cuda")
    x, t, m = loader[0]
    with torch.no_grad():
        p = dec.eval()(encoder_features(model, x, 16000)).cpu()
    keep = m != 0
    pr, gt = p[keep].tolist(), t[keep].tolist()
    tie_p = [round(v, 1) for v in pr]   # many ties
    try:
        from sklearn.metrics import roc_auc_score
    except ImportError:
        pytest.skip("sklearn not installed")
    assert auc == round(roc_auc_score(gt, pr), 3)
    assert abs(roc_auc(torch.tensor(pr, device="cuda"), torch.tensor(gt, device="cuda")) - roc_auc_score(gt, pr)) < 1e-12
    assert abs(roc_auc(torch.tensor(tie_p, device="cuda"), torch.tensor(gt, device="cuda")) - roc_auc_score(gt, tie_p)) < 1e-12


@pytest.mark.parametrize("sr", [16000, 8000])
def test_tuned_round_trip_through_every_kernel(tune, fixtures, tmp_path, sr):
    from silero_vad_b200 import SileroVADB200, get_speech_timestamps, save_tuned
    z, meta = tune
    sd = tuned_state_dict(sr, meta)
    path = save_tuned(tmp_path / "tuned.weights", sd, sr)
    m = SileroVADB200(device=0, weights=path)
    assert m.weights == path
    a = torch.from_numpy(fixtures[meta[f"t{sr}_fixture"]]["audio"])
    m.engine.set_small_batch_max(0)
    for k in (0, 1, 2):
        m.engine.set_kernel(k)
        p = m.audio_forward(a, sr).numpy()[0]
        err = float(np.abs(p - z[f"t{sr}_probs"]).max())
        print(f"sr={sr} kernel {k}: tuned model vs reference {err:.3e}")
        assert err < TOL
        segs = get_speech_timestamps(a, m, sampling_rate=sr)
        assert [[d["start"], d["end"]] for d in segs] == meta[f"t{sr}_segments"], k


def _best_thresholds_python(all_predicts, all_gts):
    """tuning/utils.py:326-356 transcribed (accuracy_score = fraction of equal labels)."""
    best_acc = 0
    for ths_enter in np.linspace(0, 1, 20):
        for ths_exit in np.linspace(0, 1, 20):
            if ths_exit >= ths_enter:
                continue
            accs = []
            for j, predict in enumerate(all_predicts):
                predict_bool = []
                is_speech = False
                for i in predict:
                    if i >= ths_enter:
                        is_speech = True
                        predict_bool.append(1)
                    elif i <= ths_exit:
                        is_speech = False
                        predict_bool.append(0)
                    else:
                        predict_bool.append(1 if is_speech else 0)
                accs.append(round(sum(g == p for g, p in zip(all_gts[j], predict_bool)) / len(predict_bool), 4))
            mean_acc = round(np.mean(accs), 3)
            if mean_acc > best_acc:
                best_acc = mean_acc
                best_ths_enter = round(ths_enter, 2)
                best_ths_exit = round(ths_exit, 2)
    return best_ths_enter, best_ths_exit, best_acc


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_threshold_search_equals_python_loop(seed):
    from silero_vad_b200 import calculate_best_thresholds
    rng = np.random.default_rng(seed)
    grid = np.linspace(0, 1, 20).astype(np.float32)
    special = np.concatenate([[0.0, 1.0], grid, np.nextafter(grid, np.float32(0)), np.nextafter(grid, np.float32(1))]).astype(np.float32)
    preds, gts = [], []
    for _ in range(int(rng.integers(5, 40))):
        L = int(rng.integers(1, 300))
        walk = np.clip(np.cumsum(rng.normal(0, 0.2, L)) % 2.0, 0, 1).astype(np.float32)
        pick = rng.random(L) < 0.3
        walk[pick] = rng.choice(special, int(pick.sum()))
        preds.append(walk.tolist())   # float32 widened to float like .tolist() of the model's output
        gts.append(rng.integers(0, 2, L).astype(np.float64).tolist())
    assert calculate_best_thresholds(preds, gts) == _best_thresholds_python(preds, gts)
