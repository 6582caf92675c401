"""The drop-in claim of INTEGRATION.md: the reference's loader and inferencer steps, driven by its shipped config/inference.toml
after changing ONE string (``[model] path``), work unchanged with ``fsnplus_b200.model.FullSubNet_Plus``.

  reference code on this path: audio_zen/utils.py:63-99 (initialize_module: dotted path -> class(**args)),
  audio_zen/inferencer/base_inferencer.py:97-110 (_load_model: initialize_module + torch.load + load_state_dict + .to(device) +
  .eval()), :133-160 (__call__: one clip per call, int16 scaling) and fullsubnet_plus/inferencer/inferencer.py:140-165
  (mag_complex_full_band_crm_mask).

What the reference did on this path is stored in tests/golden/reference_inferencer.npz (tests/golden/make_golden.py
``inferencer``): the state-dict keys and shapes of the reference class built from that TOML, the model calls its inferencer
makes, and the int16 waveforms it writes for synthetic clips 0 and 1 with the reference model and the same checkpoint.

CPU test: everything up to the forward (construction from the TOML's [model.args], strict checkpoint load, eval, the reference
class's keys and shapes) and the documented error on CPU tensors.  GPU test: the inferencer's per-clip loop with the model on
the B200, its int16 waveforms compared with those the all-reference inferencer wrote.
"""
import importlib
import os

import numpy as np
import pytest
import torch

from oracle import fsn_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
REF_TOML = os.path.join(HERE, "golden", "inference_reference.toml")


def _config(tmp_path):
    from fsnplus_b200.tools import inference as T
    cfg = T.load_toml(REF_TOML)
    assert cfg["model"]["path"] == "fullsubnet_plus.model.fullsubnet_plus.FullSubNet_Plus"
    cfg["model"]["path"] = "fsnplus_b200.model.FullSubNet_Plus"          # <- the one-string swap of INTEGRATION.md
    ckpt = tmp_path / "ckpt.tar"
    params = O.make_params_plus(O.default_plus_config(), seed=0)
    torch.save({"model": {k: torch.from_numpy(v) for k, v in params.items()}, "epoch": 7}, ckpt)
    return cfg, ckpt


def _initialize_module(path, args):
    """What a dotted [model] path means to the reference loader: import the module, instantiate the class with the args."""
    module, cls = path.rsplit(".", 1)
    return getattr(importlib.import_module(module), cls)(**args)


def _load_model(model_config, checkpoint_path, device):
    """The steps of the reference's _load_model: build from the TOML, load ``ckpt["model"]`` strictly, move, eval."""
    model = _initialize_module(model_config["path"], model_config["args"])
    ckpt = torch.load(checkpoint_path, map_location="cpu")
    model.load_state_dict(ckpt["model"])
    model.to(device)
    model.eval()
    return model, ckpt["epoch"]


def test_reference_loader_builds_and_loads_the_dropin_class(tmp_path, built_lib, golden):
    g = golden("reference_inferencer")
    cfg, ckpt = _config(tmp_path)
    from fsnplus_b200.model import FullSubNet_Plus
    m = _initialize_module(cfg["model"]["path"], cfg["model"]["args"])
    assert isinstance(m, FullSubNet_Plus)
    model, epoch = _load_model(cfg["model"], ckpt, torch.device("cpu"))     # strict load_state_dict inside
    assert isinstance(model, FullSubNet_Plus) and epoch == 7 and not model.training
    assert sum(p.numel() for p in model.parameters()) == 8675102                           # SURVEY.md 8a
    # same keys, in the same order, and shapes as the reference class built from the same TOML section
    sd = model.state_dict()
    assert list(sd.keys()) == list(g["state_dict_keys"])
    assert all(list(sd[k].shape) == [d for d in s if d >= 0] for k, s in zip(sd, g["state_dict_shapes"]))
    x = torch.zeros(1, 1, 257, 10)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(x, x, x)


@pytest.mark.gpu
def test_reference_inferencer_runs_the_dropin_model_on_gpu(tmp_path, built_lib, golden):
    """The reference inferencer's loop, one clip per call: STFT -> model(mag, real, imag) -> decompress_cIRM x spectrum -> iSTFT
    -> int16, with the drop-in model on the B200; every call has the shapes the reference inferencer used."""
    from fsnplus_b200 import inference as H
    from fsnplus_b200.model import FullSubNet_Plus
    from fsnplus_b200.tools import inference as T
    g = golden("reference_inferencer")
    clips = O.synth_clips(2).astype(np.float32)
    cfg, ckpt = _config(tmp_path)
    dev = torch.device("cuda:0")
    model, epoch = _load_model(cfg["model"], ckpt, dev)
    assert isinstance(model, FullSubNet_Plus) and epoch == 7
    assert [os.path.basename(f) for f in g["files"]] == ["clip0.wav", "clip1.wav"]
    assert all(os.path.dirname(f) == f"enhanced_{str(epoch).zfill(4)}" for f in g["files"])
    ac = cfg["acoustics"]
    stft_args = (ac["n_fft"], ac["hop_length"], ac["win_length"])
    for i, clip in enumerate(clips):
        noisy = torch.from_numpy(clip)[None].to(dev)
        X = H.stft(noisy, *stft_args)
        ins = (X.abs().unsqueeze(1), X.real.unsqueeze(1).contiguous(), X.imag.unsqueeze(1).contiguous())
        with torch.no_grad():
            crm = model(*ins)
        assert [list(x.shape) for x in ins] + [list(crm.shape)] == g["model_calls"][i].tolist()
        enhanced = H.istft(H.apply_cirm(crm, X), *stft_args, length=noisy.size(-1))[0].cpu().numpy()
        pcm, want = T.to_int16(enhanced), g["pcm"][i]
        assert pcm.dtype == np.int16 and pcm.shape == want.shape
        err = O.rel_l2(pcm.astype(np.float64), want.astype(np.float64))
        print(f"\n[reference inferencer loop + drop-in model] clip{i} int16 waveform vs all-reference inferencer: rel-L2 {err:.3e}, "
              f"max |diff| {np.abs(pcm.astype(int) - want.astype(int)).max()} LSB")
        assert err < 2e-3
