"""Boundary test (SURVEY §8b recipe): the reference's UNCHANGED callers — `trainer/trainer.py:Trainer`, `trainer/base_trainer.py`
checkpointing, `util/utils.py:initialize_config / load_checkpoint` and the `enhancement.py` script — against the drop-in
module selected only by the config's "module" string.

The reference is not part of this repository, so what its callers produced is stored under tests/golden/
(oracle/gen_golden_callers.py runs them unchanged, with the drop-in or with the reference module): the checkpoint
base_trainer wrote while training the drop-in, the reference module's output with that checkpoint, the drop-in's
parameters after the Trainer ran one epoch over the drop-in Dataset plugin, a sample of what enhancement.py wrote for the
reference module, and a one-step Adam checkpoint of the reference module with its next step. The tests make the same
calls on the drop-in (trainer/trainer.py:34-38, util/utils.py:55-72, enhancement.py:53-71 as test_enhance.reference_loop)
and compare. Everything runs on the CPU: the drop-in trains with ``train_backend="torch"`` (the native kernels are
compared with it and with the float64 goldens on the B200 in tests/test_train_gpu.py), and for the enhancement run the ONE
native call (``Model._forward_native``) is replaced by the torch restatement of the same formulas. The checkpoints use 4
levels and 2 base filters to keep the stored files small."""
import importlib
import json
import os

import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

from oracle import wunet_oracle as wo
from test_enhance import reference_loop

DROPIN = "wave_u_net_for_speech_enhancement_b200.unet_basic"
N, CI = 4, 2
ENH_SEED = 5                 # wo.make_state seed of the 12 x 24 checkpoint enhancement.py runs with


def train_config(root, epochs):
    return {"seed": 0, "root_dir": str(root), "experiment_name": "boundary", "cudnn_deterministic": False,
            "trainer": {"module": "trainer.trainer", "main": "Trainer", "epochs": epochs, "save_checkpoint_interval": 1,
                        "validation": {"interval": 0, "find_max": True, "custom": {}}},
            "model": {"module": DROPIN, "main": "Model", "args": {"n_layers": N, "channels_interval": CI, "train_backend": "torch"}},
            "loss_function": {"module": "model.loss", "main": "mse_loss", "args": {}},
            "optimizer": {"lr": 0.001, "beta1": 0.9, "beta2": 0.999}}


def synthetic_loader(T=64, batches=3, B=4):
    g = torch.Generator().manual_seed(5)
    out = []
    for i in range(batches):
        clean = 0.1 * torch.randn(B, 1, T, generator=g)
        out.append((clean + 0.05 * torch.randn(B, 1, T, generator=g), clean, [f"f{i}_{j}" for j in range(B)]))
    return out


def probe_input():
    return torch.from_numpy((np.random.default_rng(4).standard_normal((2, 1, 64))).astype(np.float32))


def plugin_wavs(root):
    """Six noisy / clean int16 pairs and their list file (config/train/train.json:37-47 format); returns the list path."""
    import scipy.io.wavfile as wavfile
    os.makedirs(root, exist_ok=True)
    rng = np.random.default_rng(2)
    lines = []
    for i in range(6):
        n = 400 + 13 * i
        clean = rng.integers(-8000, 8000, n, dtype=np.int16)
        noisy = (clean + rng.integers(-900, 900, n)).astype(np.int16)
        wavfile.write(os.path.join(root, f"c{i}.wav"), 16000, clean)
        wavfile.write(os.path.join(root, f"n{i}.wav"), 16000, noisy)
        lines.append(f"{os.path.join(root, f'n{i}.wav')} {os.path.join(root, f'c{i}.wav')}")
    lst = os.path.join(root, "train.txt")
    with open(lst, "w") as f:
        f.write("\n".join(lines) + "\n")
    return lst


def plugin_stanza(lst):
    return {"module": "wave_u_net_for_speech_enhancement_b200.dataset", "main": "Dataset",
            "args": {"dataset": lst, "limit": None, "offset": 0, "sample_length": 64, "mode": "train"}}


def plugin_initial_state():
    return {k: torch.from_numpy(np.asarray(v)) for k, v in wo.make_state(N, CI, seed=31).items()}


def enhancement_clips():
    rng = np.random.default_rng(0)
    return [(0.3 * rng.standard_normal(16384 + 4000)).astype(np.float32),    # padded to 2 chunks, trimmed
            (0.3 * rng.standard_normal(16384)).astype(np.float32)]           # exactly one chunk


def after_step_atol(key):
    """Tolerance of a state entry after Adam steps against the stored reference run. A conv bias that feeds a train-mode
    BatchNorm has a zero gradient; what autograd returns for it is rounding noise whose value depends on the CPU's
    summation order, and Adam scales any nonzero gradient to a step of up to ~1.4 lr per step. Those biases agree only to
    within that, and the running mean of the BatchNorm after them, which moves by momentum (0.1) times the batch mean of
    a later step, to within a tenth of it; every other entry agrees to 1e-7."""
    if key.endswith(".main.0.bias") or key == "middle.0.bias":
        return 3e-3
    return 3e-4 if key.endswith(".1.running_mean") else 1e-7


def train_epoch(model, optimizer, loader):
    """trainer/trainer.py:32-38"""
    loss_function = torch.nn.MSELoss()                                   # model/loss.py
    for mixture, clean, _name in loader:
        optimizer.zero_grad()
        loss = loss_function(clean, model(mixture))
        loss.backward()
        optimizer.step()


def adam(model):
    return torch.optim.Adam(params=model.parameters(), lr=0.001, betas=(0.9, 0.999))      # train.py:31-35


def test_unchanged_trainer_trains_checkpoints_and_resumes_the_dropin(golden_dir, tmp_path):
    """The latest_model.tar the unchanged base_trainer wrote after two epochs of the drop-in loads strictly into a fresh
    drop-in, which computes what the reference module computed with it; resuming from it (base_trainer.py:62-81) restores the
    model and the index-keyed optimizer state and training continues; the nn.DataParallel form keeps `.module` the drop-in."""
    ck = torch.load(os.path.join(golden_dir, f"trainer_latest_model_n{N}_c{CI}.tar"), map_location="cpu")
    g = np.load(os.path.join(golden_dir, "callers.npz"))
    assert {"epoch", "optimizer", "model"} <= set(ck) and ck["epoch"] == 2
    torch.manual_seed(0)
    init = importlib.import_module(DROPIN).Model(N, CI, train_backend="torch")
    assert list(init.state_dict()) == list(ck["model"])
    assert any(not torch.equal(a, b) for a, b in zip(init.state_dict().values(), ck["model"].values())), \
        "optimizer never moved the parameters"

    drop = importlib.import_module(DROPIN).Model(N, CI, train_backend="torch")
    drop.load_state_dict(ck["model"])                                               # strict
    drop.eval()
    with torch.no_grad():
        y = drop._forward_torch_reference_semantics(torch.from_numpy(g["trainer_x"]))
    assert np.abs(y.numpy() - g["trainer_y"]).max() <= 1e-6

    # resume: model and optimizer state come back, training continues at epoch 3
    t2 = importlib.import_module(DROPIN).Model(N, CI, train_backend="torch")
    opt = adam(t2)
    t2.load_state_dict(ck["model"])
    opt.load_state_dict(ck["optimizer"])
    assert ck["epoch"] + 1 == 3
    for a, b in zip(t2.state_dict().values(), ck["model"].values()):
        assert torch.equal(a, b)
    assert len(opt.state_dict()["state"]) == len(list(t2.parameters()))
    before = [p.detach().clone() for p in t2.parameters()]
    t2.train()
    train_epoch(t2, opt, synthetic_loader())
    assert any(not torch.equal(a, b) for a, b in zip(before, t2.parameters()))

    # the nn.DataParallel branches of save / resume (base_trainer.py:76-77, 102-103): `.module` is the drop-in
    dp = torch.nn.DataParallel(t2)
    torch.save({"epoch": 4, "optimizer": opt.state_dict(), "model": dp.module.cpu().state_dict()}, tmp_path / "latest_model.tar")
    back = torch.load(tmp_path / "latest_model.tar", map_location="cpu")
    opt.load_state_dict(back["optimizer"])
    dp.module.load_state_dict(back["model"])
    assert back["epoch"] + 1 == 5 and type(dp.module).__module__ == DROPIN


def test_adam_state_written_with_the_reference_model_continues_on_the_dropin(golden_dir):
    """Adam's state is keyed by parameter INDEX (base_trainer.py:74,99): a run started with the reference module and resumed
    with the drop-in must continue exactly as the reference would have. The reference's checkpoint after one step, its next
    batch, and its loss and state after that second step are stored (4 levels, 2 base filters)."""
    g = np.load(os.path.join(golden_dir, "adam_resume_n4_c2.npz"))
    n, ci = int(g["n_layers"]), int(g["channels_interval"])
    model_sd = {k[len("model:"):]: torch.from_numpy(g[k]) for k in g.files if k.startswith("model:")}
    state = {}
    for k in (k for k in g.files if k.startswith("opt:")):
        _, i, name = k.split(":")
        state.setdefault(int(i), {})[name] = torch.from_numpy(g[k])
    opt_sd = {"state": state, "param_groups": json.loads(str(g["opt_param_groups"]))}
    mixture, clean = torch.from_numpy(g["mixture"]), torch.from_numpy(g["clean"])
    drop = importlib.import_module(DROPIN).Model(n, ci, train_backend="torch").train()
    drop.load_state_dict(model_sd)
    opt2 = torch.optim.Adam(drop.parameters(), lr=1e-3, betas=(0.9, 0.999))
    opt2.load_state_dict(opt_sd)
    opt2.zero_grad()
    loss = torch.nn.MSELoss()(clean, drop(mixture))
    loss.backward()
    opt2.step()
    got, want = float(loss.detach()), float(g["loss"])
    assert abs(got - want) <= 1e-7 * abs(want)
    final = [k for k in g.files if k.startswith("final:")]
    assert [k[len("final:"):] for k in final] == list(drop.state_dict().keys())
    for k, b in zip(final, drop.state_dict().values()):
        assert torch.allclose(torch.from_numpy(g[k]).float(), b.float(), atol=after_step_atol(k[len("final:"):])), k


def test_unchanged_enhancement_script_runs_the_dropin(golden_dir, tmp_path, monkeypatch):
    """enhancement.py's calls (plugin loading, strict checkpoint load, `.to()/.eval()`, the [1,1,16384] chunk calls,
    `.detach().cpu()`, trimming) on the drop-in give what the unchanged script wrote for the reference module with the same
    checkpoint and inputs (a seeded sample of the samples is stored)."""
    drop_mod = importlib.import_module(DROPIN)
    monkeypatch.setattr(drop_mod.Model, "_forward_native", lambda self, x: self._forward_torch_reference_semantics(x).detach())
    ckpt = tmp_path / "model_0001.pth"
    torch.save({k: torch.from_numpy(np.asarray(v)) for k, v in wo.make_state(12, 24, seed=ENH_SEED).items()}, ckpt)
    cfg = {"module": DROPIN, "main": "Model", "args": {}}                               # the enhancement config's "model"
    model = getattr(importlib.import_module(cfg["module"]), cfg["main"])(**cfg["args"])
    model.load_state_dict(torch.load(ckpt, map_location="cpu"))                        # strict
    model.to(torch.device("cpu"))
    model.eval()
    g = np.load(os.path.join(golden_dir, "callers.npz"))
    for name, clip in zip(("a", "b"), enhancement_clips()):
        y = reference_loop(lambda chunk: model(chunk).detach().cpu(), clip, 16384)
        assert y.shape == clip.shape and len(y) == int(g[f"enh_{name}_len"])
        assert np.abs(y[g[f"enh_{name}_idx"]] - g[f"enh_{name}_val"]).max() <= 1e-6, name


def test_dataset_plugin_is_selected_by_the_config_stanza_and_feeds_the_unchanged_trainer(golden_dir, tmp_path):
    """config/train/train.json:37-47 with only the "module" string changed: the plugin loader builds the drop-in Dataset, a
    stock DataLoader batches it (train.py:15-27), and one epoch of training on those batches ends where the unchanged
    Trainer's epoch ended."""
    stanza = plugin_stanza(plugin_wavs(str(tmp_path)))
    dataset = getattr(importlib.import_module(stanza["module"]), stanza["main"])(**stanza["args"])     # train.py:15
    assert type(dataset).__module__ == "wave_u_net_for_speech_enhancement_b200.dataset" and len(dataset) == 6
    np.random.seed(0)
    loader = DataLoader(dataset=dataset, batch_size=3, num_workers=0, shuffle=False)
    batches = list(loader)
    assert len(batches) == 2 and batches[0][0].shape == (3, 1, 64) and batches[0][0].dtype == torch.float32
    assert list(batches[1][2]) == ["n3", "n4", "n5"]
    model = importlib.import_module(DROPIN).Model(N, CI, train_backend="torch")
    model.load_state_dict(plugin_initial_state())
    model.train()
    opt = adam(model)
    before = [p.detach().clone() for p in model.parameters()]
    train_epoch(model, opt, loader)
    assert any(not torch.equal(a, b) for a, b in zip(before, model.parameters()))
    g = np.load(os.path.join(golden_dir, "callers.npz"))
    for k, v in model.state_dict().items():
        assert torch.allclose(torch.from_numpy(g["plugin:" + k]).float(), v.float(), atol=after_step_atol(k)), k
