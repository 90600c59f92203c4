"""CPU tests of the drop-in boundary (SURVEY §8b): state_dict surface, parameter order, checkpoint
interchange, error behaviour, C-ABI symbols. No GPU compute."""
import ctypes
import importlib
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import wunet_oracle as wo
from wave_u_net_for_speech_enhancement_b200 import Model, _lib
from wave_u_net_for_speech_enhancement_b200 import build as wbuild

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def surface(golden_dir):
    return json.load(open(os.path.join(golden_dir, "state_dict_surface.json")))


def test_state_dict_matches_reference_surface(surface):
    m = Model()
    got = [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in m.state_dict().items()]
    assert got == surface["state_dict"]
    assert len(got) == 177


def test_parameter_order_and_count(surface):
    m = Model()
    got = [[k, list(v.shape)] for k, v in m.named_parameters()]
    assert got == surface["named_parameters"]          # Adam state is index-keyed (base_trainer.py:74,99)
    assert len(got) == 102
    assert sum(p.numel() for p in m.parameters()) == surface["n_params"] == 10132802


def test_plugin_loader_contract():
    """util/utils.py:55-72: importlib.import_module(cfg['module']) then getattr(mod, cfg['main'])(**cfg['args'])."""
    cfg = {"module": "wave_u_net_for_speech_enhancement_b200.unet_basic", "main": "Model", "args": {}}
    mod = importlib.import_module(cfg["module"])
    m = getattr(mod, cfg["main"])(**cfg["args"])
    assert m.n_layers == 12 and m.channels_interval == 24
    m2 = getattr(mod, cfg["main"])(n_layers=4, channels_interval=8)
    assert [k for k, _s, _d in wo.state_keys(4, 8)] == list(m2.state_dict().keys())


def test_strict_load_of_reference_format_checkpoint(tmp_path):
    """trainer/base_trainer.py:102-120 saves model.cpu().state_dict(); util/utils.py:11-21 loads .pth / .tar."""
    st = {k: torch.from_numpy(np.asarray(v)) for k, v in wo.make_state(12, 24, seed=0).items()}
    torch.save(st, tmp_path / "model_0001.pth")
    torch.save({"epoch": 1, "best_score": 0.0, "optimizer": {}, "model": st}, tmp_path / "latest_model.tar")
    m = Model()
    m.load_state_dict(torch.load(tmp_path / "model_0001.pth", map_location="cpu"), strict=True)
    m.load_state_dict(torch.load(tmp_path / "latest_model.tar", map_location="cpu")["model"], strict=True)
    for k, v in m.state_dict().items():
        assert torch.equal(v, st[k]), k
    m.cpu()                                              # .cpu()/.to() round trip must not break the module
    assert m._native.peek() is None                      # no native context was created on the way


def test_adam_state_round_trip():
    m = Model(n_layers=3, channels_interval=4, train_backend="torch")
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, betas=(0.9, 0.999))
    m.train()
    x = torch.randn(2, 1, 64)
    loss = torch.nn.functional.mse_loss(torch.zeros_like(x), m(x))     # loss(clean, enhanced), trainer.py:36
    loss.backward()
    opt.step()
    sd = opt.state_dict()
    assert len(sd["param_groups"][0]["params"]) == len(list(m.parameters()))
    opt2 = torch.optim.Adam(Model(n_layers=3, channels_interval=4).parameters())
    opt2.load_state_dict(sd)


def test_eval_forward_has_no_cpu_fallback():
    m = Model().eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 1, 16384))


def test_train_mode_backends():
    m = Model(n_layers=2, channels_interval=4)               # default: the native training step, CUDA only
    m.train()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 1, 16))
    m0 = Model(n_layers=2, channels_interval=4, train_backend="none").train()
    with pytest.raises(NotImplementedError):
        m0(torch.zeros(1, 1, 16))
    m2 = Model(n_layers=2, channels_interval=4, train_backend="torch").train()
    assert m2(torch.zeros(2, 1, 16)).shape == (2, 1, 16)


def test_bad_shapes_raise():
    m = Model().eval()
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 2, 16384))
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 1, 16384, dtype=torch.float64))
    with pytest.raises(ValueError):
        Model(precision="fp8")


def test_torch_training_path_matches_oracle_in_eval_semantics():
    """The opt-in composite path has the reference's semantics (checked in eval via module.eval())."""
    n, ci, B, T = 4, 8, 3, 256
    st = wo.make_state(n, ci, seed=11)
    m = Model(n, ci, train_backend="torch")
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in st.items()})
    m.eval()
    x = wo.make_input(B, T, seed=12)
    with torch.no_grad():
        y = m._forward_torch_reference_semantics(torch.from_numpy(x)).numpy()
    assert np.abs(y - wo.COracle(n, ci).forward(st, x)).max() <= 1e-5


def test_empty_batch_like_the_reference(golden_dir):
    """Zero frames: the reference's eval forward returns an empty [0, 1, T] tensor and still rejects a bad length; so does the
    drop-in, without touching the device (the C ABI itself takes B >= 1)."""
    m = Model(4, 8).eval()
    y = m(torch.zeros(0, 1, 256))
    assert y.shape == (0, 1, 256) and y.dtype == torch.float32
    assert m.forward_host(torch.zeros(0, 1, 256)).shape == (0, 1, 256)
    with pytest.raises(RuntimeError, match="not a multiple"):
        m(torch.zeros(0, 1, 100))
    ref = json.load(open(os.path.join(golden_dir, "empty_batch.json")))     # what the reference's Model(4, 8) returned
    assert (ref["n_layers"], ref["channels_interval"], ref["input_shape"]) == (4, 8, [0, 1, 256])
    assert list(y.shape) == ref["shape"] and str(y.dtype).replace("torch.", "") == ref["dtype"]


def test_library_builds_and_exports_header_symbols():
    so = wbuild.build()
    lib = ctypes.CDLL(so)
    header = open(os.path.join(ROOT, "include", "wunet_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(wunet_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no declarations parsed"
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/wunet_b200.h but not exported"
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared


def test_create_without_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib.load()
    ctx = ctypes.c_void_p()
    rc = lib.wunet_create(12, 24, 0, ctypes.byref(ctx))
    assert rc < 0 and b"no CUDA device" in lib.wunet_last_error()


def test_product_path_does_not_import_oracle():
    pkg = os.path.join(ROOT, "wave_u_net_for_speech_enhancement_b200")
    for dirpath, _d, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, fn)).read()
                assert "oracle" not in src.replace("no oracle", ""), f"{fn} references the oracle"
