"""CPU tests of decoder fine-tuning (silero_vad_b200.tuning): the fp32 kernel's features mode run by the barrier-level emulator
against the reference's features, the training kernels' LSTM cell step against torch float64 autograd, tuned-weight containers
through the C oracle, and argument checks of the new C ABI functions."""
import ctypes
import importlib.util
import json
import subprocess

import numpy as np
import pytest
import torch

from conftest import GOLDEN, REPO

TOL = 1e-4


@pytest.fixture(scope="module")
def tune():
    return dict(np.load(GOLDEN / "tune.npz")), json.loads((GOLDEN / "tune.json").read_text())


def golden_recipe():
    """tools/gen_golden_tune.py: the seeded "tuned" decoder of the fixtures is recomputed, not stored."""
    spec = importlib.util.spec_from_file_location("gen_golden_tune", REPO / "tools" / "gen_golden_tune.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def tuned_state_dict(sr, meta):
    from silero_vad_b200 import tuning
    gen = golden_recipe()
    stock = {k: v.numpy() for k, v in tuning.decoder_state_dict(sr).items()}
    tuned = gen.tuned_decoder(stock, sr)
    assert gen.abs_sum(tuned) == meta[f"t{sr}_abs_sum"]
    return {k: torch.from_numpy(v) for k, v in tuned.items()}


def clips(fixtures, meta, sr):
    n = 512 if sr == 16000 else 256
    a = fixtures["test16k" if sr == 16000 else "aepyx8k"]["audio"]
    return np.stack([a[o:o + 64 * n] for o in meta[f"f{sr}_offsets"]]).copy()


@pytest.fixture(scope="module")
def emu_tune(tmp_path_factory):
    so = tmp_path_factory.mktemp("emu") / "libsvad_emu_tune.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", str(so), str(REPO / "tests" / "emu" / "svad_emu_tune.cpp")],
                   check=True)
    lib = ctypes.CDLL(str(so))
    fp = ctypes.c_void_p
    lib.svad_emu_features.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_long, fp, fp, fp]
    lib.svad_emu_cell_fwd.argtypes = [fp, ctypes.c_float, fp]
    lib.svad_emu_cell_fwd.restype = None
    lib.svad_emu_cell_bwd.argtypes = [fp, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, fp]
    lib.svad_emu_cell_bwd.restype = None
    return lib


def _emu_features(emu, sr, x, ctx_in=None, rm=8):
    from silero_vad_b200.model import WEIGHTS
    n = 512 if sr == 16000 else 256
    x = np.ascontiguousarray(x, np.float32)
    feat = np.full((x.shape[0], x.shape[1] // n, 128), np.nan, np.float32)
    rc = emu.svad_emu_features(str(WEIGHTS).encode(), sr, rm, x.shape[0], x.shape[1], x.ctypes.data,
                               None if ctx_in is None else ctx_in.ctypes.data, feat.ctypes.data)
    assert rc == 0
    return feat


@pytest.mark.parametrize("sr", [16000, 8000])
def test_emulated_features_match_reference(emu_tune, tune, fixtures, sr):
    z, meta = tune
    feat = _emu_features(emu_tune, sr, clips(fixtures, meta, sr))
    err = float(np.abs(feat - z[f"f{sr}_feat"]).max())
    print(f"sr={sr}: max|feat_emu - feat_ref| = {err:.3e}")
    assert err <= 1e-4


@pytest.mark.parametrize("sr", [16000, 8000])
def test_emulated_features_segmented_equal_whole(emu_tune, tune, fixtures, sr):
    """Rows of S chunks with the preceding ctx samples passed in give the whole-stream features bit for bit."""
    _, meta = tune
    n, ctx = (512, 64) if sr == 16000 else (256, 32)
    x = clips(fixtures, meta, sr)[:, : 24 * n]
    whole = _emu_features(emu_tune, sr, x, rm=4)
    S = 8
    rows = x.reshape(2 * 3, S * n).copy()
    cx = np.zeros((2, 3, ctx), np.float32)
    cx[:, 1:] = x.reshape(2, 3, S * n)[:, :-1, -ctx:]
    seg = _emu_features(emu_tune, sr, rows, np.ascontiguousarray(cx.reshape(6, ctx)), rm=4).reshape(2, 24, 128)
    assert np.array_equal(seg, whole)


def test_cell_step_matches_float64_autograd(emu_tune):
    rng = np.random.default_rng(7)
    for _ in range(20):
        pre = (rng.standard_normal(4) * 2).astype(np.float32)
        c_prev = np.float32(rng.standard_normal())
        dh, dc = np.float32(rng.standard_normal()), np.float32(rng.standard_normal())
        out = np.zeros(6, np.float32)
        emu_tune.svad_emu_cell_fwd(pre.ctypes.data, float(c_prev), out.ctypes.data)
        p = torch.tensor(pre, dtype=torch.float64, requires_grad=True)
        cp = torch.tensor(float(c_prev), dtype=torch.float64, requires_grad=True)
        i, f, g, o = torch.sigmoid(p[0]), torch.sigmoid(p[1]), torch.tanh(p[2]), torch.sigmoid(p[3])
        c = f * cp + i * g
        h = o * torch.tanh(c)
        want = torch.stack([i, f, g, o, c, h]).detach().numpy()
        assert np.abs(out - want).max() < 1e-6
        (h * float(dh) + c * float(dc)).backward()
        grads = np.zeros(5, np.float32)
        emu_tune.svad_emu_cell_bwd(out[:4].ctypes.data, float(c_prev), float(out[4]), float(dh), float(dc), grads.ctypes.data)
        want_g = np.concatenate([p.grad.numpy(), [cp.grad.item()]])
        assert np.abs(grads - want_g).max() < 1e-5 * max(1.0, np.abs(want_g).max())


def _oracle_with(path):
    from oracle.oracle import BASIS, Oracle
    o = Oracle()
    o.lib.svad_oracle_free(o.h)
    o.h = o.lib.svad_oracle_load(str(path).encode(), str(BASIS).encode())
    assert o.h
    return o


@pytest.mark.parametrize("sr", [16000, 8000])
def test_tuned_container_through_oracle(tune, fixtures, tmp_path, sr):
    from silero_vad_b200 import tuning
    z, meta = tune
    sd = tuned_state_dict(sr, meta)
    path = tuning.save_tuned(tmp_path / "tuned.weights", sd, sr)
    assert tuning.decoder_state_dict(sr, path)["rnn.weight_hh"].equal(sd["rnn.weight_hh"])
    other = 8000 if sr == 16000 else 16000
    assert tuning.decoder_state_dict(other, path)["rnn.weight_hh"].equal(tuning.decoder_state_dict(other)["rnn.weight_hh"])
    fx = fixtures[meta[f"t{sr}_fixture"]]
    p = _oracle_with(path).audio_forward(fx["audio"], sr, nthreads=8)[0]
    err = float(np.abs(p - z[f"t{sr}_probs"]).max())
    print(f"sr={sr}: oracle with the tuned container vs reference: {err:.3e}")
    assert err < TOL


def test_export_weights_round_trips_a_scripted_module(tmp_path):
    from silero_vad_b200 import tuning
    from silero_vad_b200.model import WEIGHTS
    stock = tuning.read_container(WEIGHTS)
    root = torch.nn.Module()
    for name, t in list(stock.items()) + [("_model.stft.forward_basis_buffer", torch.zeros(258, 1, 256))]:
        m = root
        for part in name.split(".")[:-1]:
            if not hasattr(m, part):
                m.add_module(part, torch.nn.Module())
            m = getattr(m, part)
        m.register_buffer(name.split(".")[-1], t.clone() + (1.0 if "decoder" in name else 0.0))
    torch.jit.save(torch.jit.script(root), str(tmp_path / "m.jit"))
    out = tuning.export_weights(tmp_path / "m.jit", tmp_path / "m.weights")
    back = tuning.read_container(out)
    assert list(back) == list(stock)
    for k in stock:
        assert back[k].equal(stock[k] + (1.0 if "decoder" in k else 0.0)), k
    bad = {k: v for k, v in stock.items() if k != "_model.decoder.rnn.bias_hh"}
    with pytest.raises(ValueError, match="missing"):
        tuning.export_weights(bad, tmp_path / "bad.weights")
    bad = dict(stock)
    bad["_model.decoder.rnn.bias_hh"] = torch.zeros(3)
    with pytest.raises(ValueError, match="shape"):
        tuning.export_weights(bad, tmp_path / "bad.weights")


def test_new_abi_functions_reject_bad_arguments_without_a_device():
    from silero_vad_b200 import _cabi
    L = _cabi.lib()
    EINVAL = -1
    dummy = ctypes.c_void_p(16)
    assert L.svad_features_device(None, 16000, 1, 512, 512, dummy, None, dummy, None) == EINVAL
    assert L.svad_decoder_tape_floats(-1, 5) == EINVAL and L.svad_decoder_tape_floats(2, 3) == 2 * 3 * 640
    assert L.svad_decoder_workspace_bytes(2, -1, 0) == EINVAL
    assert L.svad_decoder_forward_device(None, 1, 1, *([dummy] * 12)) == EINVAL
    assert L.svad_decoder_backward_device(None, 1, 1, *([dummy] * 14)) == EINVAL
    assert L.svad_threshold_grid_device(dummy, dummy, dummy, -1, dummy, dummy, None) == EINVAL
    assert L.svad_threshold_grid_device(None, dummy, dummy, 3, dummy, dummy, None) == EINVAL
    assert L.svad_threshold_grid_device(dummy, dummy, dummy, 3, None, dummy, None) == EINVAL
    assert "null" in L.svad_last_error().decode()


def test_threshold_search_rejects_empty_input():
    from silero_vad_b200 import calculate_best_thresholds
    with pytest.raises(ValueError):
        calculate_best_thresholds([], [])
    with pytest.raises(ValueError):
        calculate_best_thresholds([[0.1, 0.2]], [[0]])
