"""
oracle/gen_golden_callers.py — generates the golden vectors that stand in for the reference in the caller-side tests.

Needs a checkout of the reference project; point WUNET_REFERENCE at it:

    WUNET_REFERENCE=<checkout> python oracle/gen_golden_callers.py

What is recorded from the unmodified reference, for the tests that used to import it directly:

* ``dataset_items.json`` — what ``dataset/waveform_dataset.py:Dataset`` returns (name, shape and a sha256 of the exact
  float32 samples of every item, train and validation mode) for the seeded wav files of tests/test_dataset_cpu.py, with
  ``librosa.load`` stubbed by that test's soundfile-like reader (tests/test_dataset_cpu.py).
* ``adam_resume_n4_c2.npz`` — a checkpoint written after one Adam step of ``model/unet_basic.py:Model`` (model state and
  the index-keyed optimizer state), the next batch, and the loss and model state after the reference's second step
  (tests/test_boundary_callers.py).  4 levels like the other caller tests, 2 base filters to keep the file small.
* ``empty_batch.json`` — the shape and dtype the reference's eval forward returns for zero frames
  (tests/test_module_surface.py).
* ``trainer_latest_model_n4_c2.tar`` and ``callers.npz`` — the reference's own callers driving the drop-in or the
  reference module (tests/test_boundary_callers.py): the ``latest_model.tar`` that ``trainer/base_trainer.py`` wrote after
  two epochs of the drop-in, the reference module's output with that checkpoint, the drop-in's parameters after the
  unchanged Trainer ran one epoch over the drop-in Dataset plugin, and a seeded sample of what ``enhancement.py`` wrote for
  the reference module.  The packages the reference imports but this image lacks (json5, librosa, pesq, pystoi,
  matplotlib) are stubbed; the reference itself is imported unchanged.
"""
import copy
import hashlib
import importlib
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden")
REF = os.environ.get("WUNET_REFERENCE")
if not REF or not os.path.isdir(os.path.join(REF, "model")):
    sys.exit("set WUNET_REFERENCE to a checkout of the reference project")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, REF)


def sha256(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def dataset_items():
    import test_dataset_cpu as tdc                          # the wav files and the librosa stand-in the test uses
    sys.modules["librosa"] = types.SimpleNamespace(load=lambda path, sr=None: tdc.soundfile_like(path))
    for name in ("pesq", "pystoi", "pystoi.stoi"):
        m = types.ModuleType(name)
        m.pesq = m.stoi = lambda *a, **k: 0.0
        sys.modules[name] = m
    sys.modules["pystoi"].stoi = sys.modules["pystoi.stoi"]
    ref_ds = importlib.import_module("dataset.waveform_dataset")
    out = {"seed": 7, "sample_length": 16384}
    with tempfile.TemporaryDirectory() as d:
        import pathlib
        lst, _lines = tdc._pair_files(pathlib.Path(d))
        for mode in ("train", "validation"):
            r = ref_ds.Dataset(lst, sample_length=16384, mode=mode)
            np.random.seed(7)
            items = [r[i] for i in range(len(r))]
            out[mode] = [{"name": n, "shape": list(m.shape), "dtype": str(m.dtype), "mixture_sha256": sha256(m),
                          "clean_sha256": sha256(c)} for m, c, n in items]
    with open(os.path.join(OUT, "dataset_items.json"), "w") as f:
        json.dump(out, f, indent=1)


def adam_resume(n=4, ci=2):
    from model.unet_basic import Model
    g = torch.Generator().manual_seed(5)
    batches = []
    for _ in range(2):
        clean = 0.1 * torch.randn(4, 1, 64, generator=g)
        batches.append((clean + 0.05 * torch.randn(4, 1, 64, generator=g), clean))
    loss_fn = torch.nn.MSELoss()

    def one_step(model, optimizer, batch):
        optimizer.zero_grad()
        loss = loss_fn(batch[1], model(batch[0]))
        loss.backward()
        optimizer.step()
        return float(loss.detach())

    torch.manual_seed(1)
    ref = Model(n_layers=n, channels_interval=ci).train()
    opt = torch.optim.Adam(ref.parameters(), lr=1e-3, betas=(0.9, 0.999))
    one_step(ref, opt, batches[0])
    rec = {"n_layers": n, "channels_interval": ci, "mixture": batches[1][0].numpy(), "clean": batches[1][1].numpy()}
    rec.update({"model:" + k: v.numpy().copy() for k, v in ref.state_dict().items()})
    osd = copy.deepcopy(opt.state_dict())
    for i, s in osd["state"].items():
        for name, v in s.items():
            rec[f"opt:{i}:{name}"] = v.numpy()
    rec["opt_param_groups"] = np.array(json.dumps(osd["param_groups"]))
    rec["loss"] = np.float64(one_step(ref, opt, batches[1]))
    rec.update({"final:" + k: v.numpy().copy() for k, v in ref.state_dict().items()})
    np.savez_compressed(os.path.join(OUT, f"adam_resume_n{n}_c{ci}.npz"), **rec)


def empty_batch():
    from model.unet_basic import Model
    y = Model(4, 8).eval()(torch.zeros(0, 1, 256))
    with open(os.path.join(OUT, "empty_batch.json"), "w") as f:
        json.dump({"n_layers": 4, "channels_interval": 8, "input_shape": [0, 1, 256], "shape": list(y.shape),
                   "dtype": str(y.dtype).replace("torch.", "")}, f, indent=1)


def stub_reference_imports(wavs, written):
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m
    mod("json5", dumps=lambda o, **k: json.dumps(o, default=str), dump=lambda o, f, **k: json.dump(o, f, default=str),
        load=json.load, loads=json.loads)
    librosa = mod("librosa", load=lambda path, sr=None: (wavs[path].copy(), 16000),
                  stft=lambda y, **k: np.zeros((161, 4), np.complex64), magphase=lambda d: (np.abs(d), d),
                  amplitude_to_db=lambda m: m)
    librosa.output = mod("librosa.output", write_wav=lambda path, y, sr: written.__setitem__(path, np.asarray(y).copy()))
    librosa.display = mod("librosa.display", waveplot=lambda *a, **k: None, specshow=lambda *a, **k: None)
    mod("pesq", pesq=lambda sr, a, b, mode: 2.0)
    pystoi = mod("pystoi")
    pystoi.stoi = mod("pystoi.stoi", stoi=lambda a, b, sr, extended=False: 0.5)
    plt = mod("matplotlib.pyplot", switch_backend=lambda *a: None, subplots=lambda *a, **k: (None, None), tight_layout=lambda: None)
    mod("matplotlib", pyplot=plt)
    for name in [k for k in sys.modules if k.split(".")[0] in ("trainer", "util", "model", "dataset")]:
        sys.modules.pop(name)


def callers():
    import pathlib
    import runpy
    import scipy.io.wavfile as wavfile
    from torch.utils.data import DataLoader
    import test_boundary_callers as tb                      # N, CI, DROPIN, configs, the synthetic loader and the wavs
    from oracle import wunet_oracle as wo
    wavs, written = {}, {}
    stub_reference_imports(wavs, written)
    utils = importlib.import_module("util.utils")
    ref_model_cls = importlib.import_module("model.unet_basic").Model
    rec = {}

    def trainer(cfg, resume, model, loader):
        optimizer = torch.optim.Adam(params=model.parameters(), lr=cfg["optimizer"]["lr"],
                                     betas=(cfg["optimizer"]["beta1"], cfg["optimizer"]["beta2"]))
        cls = utils.initialize_config(cfg["trainer"], pass_args=False)
        return cls(config=cfg, resume=resume, model=model, loss_function=utils.initialize_config(cfg["loss_function"]),
                   optimizer=optimizer, train_dataloader=loader, validation_dataloader=[])

    with tempfile.TemporaryDirectory() as d:
        d = pathlib.Path(d)
        # train.py:29-49 for two epochs of the drop-in: the checkpoint base_trainer writes
        torch.manual_seed(0)
        cfg = tb.train_config(d / "t", 2)
        trainer(cfg, False, utils.initialize_config(cfg["model"]), tb.synthetic_loader()).train()
        ck = d / "t" / "boundary" / "checkpoints"
        sd_pth = utils.load_checkpoint(str(ck / "model_0002.pth"), torch.device("cpu"))
        sd_tar = utils.load_checkpoint(str(ck / "latest_model.tar"), torch.device("cpu"))
        assert list(sd_pth) == list(sd_tar) and all(torch.equal(sd_pth[k], sd_tar[k]) for k in sd_pth)
        with open(ck / "latest_model.tar", "rb") as f, open(os.path.join(OUT, f"trainer_latest_model_n{tb.N}_c{tb.CI}.tar"), "wb") as g:
            g.write(f.read())
        ref = ref_model_cls(n_layers=tb.N, channels_interval=tb.CI)
        ref.load_state_dict(sd_pth)
        ref.eval()
        x = tb.probe_input()
        with torch.no_grad():
            rec["trainer_x"], rec["trainer_y"] = x.numpy(), ref(x).numpy()

        # config/train/train.json:37-47 with the drop-in Dataset plugin, a stock DataLoader, one epoch of the unchanged Trainer
        lst = tb.plugin_wavs(d / "p")
        dataset = utils.initialize_config(tb.plugin_stanza(lst))
        assert type(dataset).__module__ == "wave_u_net_for_speech_enhancement_b200.dataset"
        np.random.seed(0)
        loader = DataLoader(dataset=dataset, batch_size=3, num_workers=0, shuffle=False)
        list(loader)
        cfg = tb.train_config(d / "p", 1)
        model = utils.initialize_config(cfg["model"])
        model.load_state_dict(tb.plugin_initial_state())
        trainer(cfg, False, model, loader).train()
        rec.update({"plugin:" + k: v.detach().cpu().numpy().copy() for k, v in model.state_dict().items()})

        # enhancement.py end to end for the reference module (its default 12 x 24 plan)
        ckpt = d / "model_0001.pth"
        torch.save({k: torch.from_numpy(np.asarray(v)) for k, v in wo.make_state(12, 24, seed=tb.ENH_SEED).items()}, ckpt)
        listing = d / "list.txt"
        paths = [str(d / "a.wav"), str(d / "b.wav")]
        for p, clip in zip(paths, tb.enhancement_clips()):
            wavs[p] = clip
        listing.write_text("\n".join(paths) + "\n")
        cfg = {"model": {"module": "model.unet_basic", "main": "Model", "args": {}},
               "dataset": {"module": "dataset.waveform_dataset_enhancement", "main": "WaveformDataset",
                           "args": {"dataset": str(listing), "limit": None, "offset": 0, "sample_length": 16384}},
               "custom": {"sample_length": 16384}}
        (d / "enh.json").write_text(json.dumps(cfg))
        (d / "enh").mkdir()
        argv = sys.argv
        sys.argv = ["enhancement.py", "-C", str(d / "enh.json"), "-D", "-1", "-O", str(d / "enh"), "-M", str(ckpt)]
        try:
            runpy.run_path(os.path.join(REF, "enhancement.py"), run_name="__main__")
        finally:
            sys.argv = argv
        for p in paths:
            name = os.path.splitext(os.path.basename(p))[0]
            y = written[str(d / "enh" / f"{name}.wav")]
            idx = np.unique(np.concatenate([np.arange(16), np.arange(len(y) - 16, len(y)),         # both ends + 1024 seeded
                                            np.random.default_rng(9).choice(len(y), 1024, replace=False)]))
            rec[f"enh_{name}_len"], rec[f"enh_{name}_idx"], rec[f"enh_{name}_val"] = np.int64(len(y)), idx, y[idx]
    np.savez_compressed(os.path.join(OUT, "callers.npz"), **rec)


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    dataset_items()
    adam_resume()
    empty_batch()
    callers()
    for fn in ("dataset_items.json", "adam_resume_n4_c2.npz", "empty_batch.json", "trainer_latest_model_n4_c2.tar", "callers.npz"):
        print(f"  {fn}: {os.path.getsize(os.path.join(OUT, fn)) / 1024:.1f} KiB")


if __name__ == "__main__":
    main()
