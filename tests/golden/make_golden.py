"""Generate the committed golden vectors from the UNMODIFIED reference.

Run where a checkout of the reference is available (found by
oracle/ref_loader.py); the tests only read the fixtures:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [causal|inferencer]

The reference is imported read-only (librosa stubbed, SURVEY.md 8c), loaded with
the deterministic numpy parameters of ``oracle.fsn_oracle.make_params_*`` through
``load_state_dict(strict=True)`` (which also pins the state-dict key/shape
contract), run in float64 one sample at a time (the only batch size the
reference inference supports, SURVEY.md 0.4), and its outputs are written as
float32 ``.npz`` fixtures next to this script.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402

ref_loader.setup()                                  # the reference on sys.path, librosa / soundfile stubbed (never called)

import torch  # noqa: E402

from oracle import fsn_oracle as O  # noqa: E402
from fullsubnet_plus.model.fullsubnet_plus import FullSubNet_Plus  # noqa: E402
from fullsubnet.model.fullsubnet import Model as FSNModel  # noqa: E402
from audio_zen.model.module.sequence_model import SequenceModel  # noqa: E402
from audio_zen.acoustics.feature import stft as ref_stft, istft as ref_istft  # noqa: E402
from audio_zen.acoustics.mask import decompress_cIRM as ref_decompress  # noqa: E402

torch.set_grad_enabled(False)


def load(model, params):
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in params.items()}
    model.load_state_dict(sd, strict=True)
    return model.double().eval()


def hooks(model, names):
    cap = {}
    hs = []
    for n in names:
        mod = getattr(model, n)
        hs.append(mod.register_forward_hook(lambda m, i, o, n=n: cap.__setitem__(n, o.detach().numpy().copy())))
    return cap, hs


def run_plus(cfg, params, mag, real, imag):
    """Reference forward, B=1 per call, float64. Returns out [B,2,F,T] + stage captures."""
    model = load(causal_plus(cfg) if cfg.get("causal_tcn") else FullSubNet_Plus(**cfg), params)
    names = ["channel_attention", "channel_attention_real", "channel_attention_imag",
             "fb_model", "fb_model_real", "fb_model_imag"]
    outs, fb_in, fb_out = [], [], []
    for b in range(mag.shape[0]):
        cap, hs = hooks(model, names)
        t = lambda x: torch.from_numpy(np.asarray(x[b:b + 1], np.float64))
        y = model(t(mag), t(real), t(imag))
        for h in hs:
            h.remove()
        outs.append(y.numpy().copy())
        Fq, Tq = cap[names[1]][0].shape                 # subband_num > 1: the mag attention runs on [(F + pad) / sub, T * sub]
        fb_in.append(np.stack([cap[n][0].reshape(-1, Tq)[:Fq] for n in names[:3]]))
        fb_out.append(np.stack([cap[n][0] for n in names[3:]]))
    return np.concatenate(outs), np.stack(fb_in, 1), np.stack(fb_out, 1)      # [B,2,F,T], [3,B,F,T'], [3,B,F,T']


def causal_plus(cfg):
    """The reference FullSubNet_Plus with every full-band TCNBlock rebuilt as TCNBlock(causal=True) (causal_conv.py:67-117; the
    constructor of SequenceModel("TCN") never passes causal, so the variant is assembled from the reference's own block class;
    parameter names and shapes are unchanged)."""
    from audio_zen.model.module.causal_conv import TCNBlock
    kw = {k: v for k, v in cfg.items() if k != "causal_tcn"}
    model = FullSubNet_Plus(**kw)
    for sfx in ("", "_real", "_imag"):
        seq = getattr(model, "fb_model" + sfx).sequence_model
        for i, d in enumerate((1, 2, 5, 9, 1, 2, 5, 9)):
            seq[i] = TCNBlock(in_channels=cfg["num_freqs"], out_channels=cfg["num_freqs"], dilation=d, causal=True)
    return model


def run_fsn(cfg, params, mag):
    model = load(FSNModel(**cfg), params)
    outs, fb_out = [], []
    for b in range(mag.shape[0]):
        cap, hs = hooks(model, ["fb_model"])
        y = model(torch.from_numpy(np.asarray(mag[b:b + 1], np.float64)))
        for h in hs:
            h.remove()
        outs.append(y.numpy().copy()); fb_out.append(cap["fb_model"][0])
    return np.concatenate(outs), np.stack(fb_out)


def spectra(clips, n_fft=512, hop=256):
    X = ref_stft(torch.from_numpy(clips), n_fft, hop, n_fft)
    return X.abs().numpy()[:, None], X.real.numpy()[:, None], X.imag.numpy()[:, None], X.numpy()


def save(name, **kw):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **{k: (v.astype(np.float32) if isinstance(v, np.ndarray) and v.dtype == np.float64 else v)
                                 for k, v in kw.items()})
    print(f"  wrote {name}.npz  {os.path.getsize(path) / 1e6:.2f} MB")


def small_plus_cfg():
    c = O.default_plus_config()
    c.update(num_freqs=33, sb_num_neighbors=3, sb_model_hidden_size=32)
    return c


def small_fsn_cfg(norm="offline_laplace_norm"):
    c = O.default_fsn_config()
    c.update(num_freqs=33, sb_num_neighbors=3, sb_model_hidden_size=32, fb_model_hidden_size=48, norm_type=norm)
    return c


def small_inputs(B, F, T, seed):
    rng = np.random.default_rng(seed)
    real = rng.standard_normal((B, 1, F, T)) * 0.05 + 0.004
    imag = rng.standard_normal((B, 1, F, T)) * 0.05 - 0.003
    mag = np.sqrt(real ** 2 + imag ** 2)
    return mag.astype(np.float32), real.astype(np.float32), imag.astype(np.float32)


def main():
    # ---- 1. default config (config/inference.toml), one 3 s synthetic clip --------------------
    cfg = O.default_plus_config()
    clips = O.synth_clips(1)
    mag, real, imag, X = spectra(clips)
    # the oracle's numpy STFT must reproduce the reference's torch.stft
    Xo = O.stft(clips)
    print("stft oracle-vs-reference rel-L2:", O.rel_l2(np.abs(Xo), mag[:, 0]))
    for tag, scale in (("plus_default", 1.0), ("plus_default_stress", 3.0)):
        params = O.make_params_plus(cfg, seed=0, lstm_scale=scale)
        out, fb_in, fb_out = run_plus(cfg, params, mag, real, imag)
        st = {}
        oo = O.fullsubnet_plus_forward(params, cfg, mag, real, imag, stages=st)
        print(f"{tag}: oracle-vs-reference rel-L2 out={O.rel_l2(oo, out):.2e} "
              f"fb_in={O.rel_l2(st['fb_in'], fb_in):.2e} fb_out={O.rel_l2(st['fb_out'], fb_out):.2e}")
        m32 = load(FullSubNet_Plus(**cfg), params).float()
        o32 = m32(torch.from_numpy(mag), torch.from_numpy(real), torch.from_numpy(imag)).numpy()
        print(f"   reference fp32-vs-fp64 rel-L2 = {O.rel_l2(o32, out):.2e}")
        if scale == 1.0:
            enh = ref_istft(torch.stack([torch.from_numpy(O.enhance(X, out).real),
                                         torch.from_numpy(O.enhance(X, out).imag)], -1).float(), 512, 256, 512,
                            length=clips.shape[1]).numpy()
            dref = ref_decompress(torch.from_numpy(out).permute(0, 2, 3, 1)).numpy()
            print("   decompress oracle-vs-ref:", O.rel_l2(O.decompress_cIRM(out).transpose(0, 2, 3, 1), dref))
            # three files, each under 1 MB; tests/conftest.py merges "<name>.<part>.npz" into "<name>"
            save(tag, mag=mag, real=real, imag=imag, seed=0, lstm_scale=scale)
            save(tag + ".outputs", out=out, enhanced=enh)
            save(tag + ".stages", fb_in=fb_in, fb_out=fb_out)
        else:
            save(tag, out=out, seed=0, lstm_scale=scale)

    # ---- 2. fullsubnet.Model default config ---------------------------------------------------
    fcfg = O.default_fsn_config()
    params = O.make_params_fsn(fcfg, seed=1)
    out, fb_out = run_fsn(fcfg, params, mag)
    st = {}
    oo = O.fullsubnet_forward(params, fcfg, mag, stages=st)
    print(f"fsn_default: oracle-vs-reference rel-L2 out={O.rel_l2(oo, out):.2e} fb_out={O.rel_l2(st['fb_out'], fb_out):.2e}")
    save("fsn_default", out=out, fb_out=fb_out, seed=1)

    # ---- 3. small configs with every stage, B=3 (per-sample reference) -----------------------
    scfg = small_plus_cfg()
    m, r, i = small_inputs(3, 33, 20, 7)
    params = O.make_params_plus(scfg, seed=3)
    out, fb_in, fb_out = run_plus(scfg, params, m, r, i)
    st = {}
    oo = O.fullsubnet_plus_forward(params, scfg, m, r, i, stages=st)
    print(f"plus_small: oracle-vs-reference rel-L2 out={O.rel_l2(oo, out):.2e}")
    save("plus_small", mag=m, real=r, imag=i, out=out, fb_in=fb_in, fb_out=fb_out, sb_in=st["sb_in"], seed=3)

    for attn in ("SE", "ECA", "CBAM"):                                     # fullsubnet_plus.py:52-70
        acfg = dict(scfg, channel_attention_model=attn)
        params = O.make_params_plus(acfg, seed=5)
        out, fb_in, fb_out = run_plus(acfg, params, m, r, i)
        oo = O.fullsubnet_plus_forward(params, acfg, m, r, i)
        print(f"plus_small[{attn}]: oracle-vs-reference rel-L2 out={O.rel_l2(oo, out):.2e}")
        save(f"plus_small_{attn}", out=out, fb_in=fb_in, seed=5)

    # subband_num > 1 (fullsubnet_plus.py:146-153) runs in the reference only with the channel-agnostic ECA attention;
    # F = 33: subband_num = 2 pads one bin, subband_num = 3 pads a whole extra group (33 % 3 == 0)
    for sub in (2, 3):
        bcfg = dict(scfg, channel_attention_model="ECA", subband_num=sub)
        params = O.make_params_plus(bcfg, seed=5)
        out, fb_in, fb_out = run_plus(bcfg, params, m, r, i)
        print(f"plus_small[ECA, subband_num={sub}]: oracle-vs-reference rel-L2 out="
              f"{O.rel_l2(O.fullsubnet_plus_forward(params, bcfg, m, r, i), out):.2e}")
        save(f"plus_small_ECA_sub{sub}", out=out, fb_in=fb_in, seed=5)

    # fb_num_neighbors > 0: the full-band outputs are unfolded too (fullsubnet_plus.py:167-179, fullsubnet.py:90-91)
    ncfg = dict(scfg, fb_num_neighbors=1)
    params = O.make_params_plus(ncfg, seed=6)
    out, fb_in, fb_out = run_plus(ncfg, params, m, r, i)
    print(f"plus_small[fb_num_neighbors=1]: oracle-vs-reference rel-L2 out={O.rel_l2(O.fullsubnet_plus_forward(params, ncfg, m, r, i), out):.2e}")
    save("plus_small_fbn1", out=out, seed=6)
    ncfg = dict(small_fsn_cfg(), fb_num_neighbors=2)
    params = O.make_params_fsn(ncfg, seed=6)
    out, fb_out = run_fsn(ncfg, params, m)
    print(f"fsn_small[fb_num_neighbors=2]: oracle-vs-reference rel-L2 out={O.rel_l2(O.fullsubnet_forward(params, ncfg, m), out):.2e}")
    save("fsn_small_fbn2", out=out, seed=6)

    # sequence_model = "GRU" (sequence_model.py:39-46): FullSubNet+ sub-band GRU, fullsubnet.Model full-band + sub-band GRU
    gcfg = dict(scfg, sequence_model="GRU")
    params = O.make_params_plus(gcfg, seed=8, lstm_scale=2.0)
    out, fb_in, fb_out = run_plus(gcfg, params, m, r, i)
    print(f"plus_small[GRU]: oracle-vs-reference rel-L2 out={O.rel_l2(O.fullsubnet_plus_forward(params, gcfg, m, r, i), out):.2e}")
    save("plus_small_GRU", out=out, seed=8, lstm_scale=2.0)
    gcfg = dict(small_fsn_cfg(), sequence_model="GRU")
    params = O.make_params_fsn(gcfg, seed=8, lstm_scale=2.0)
    out, fb_out = run_fsn(gcfg, params, m)
    print(f"fsn_small[GRU]: oracle-vs-reference rel-L2 out={O.rel_l2(O.fullsubnet_forward(params, gcfg, m), out):.2e}")
    save("fsn_small_GRU", out=out, fb_out=fb_out, seed=8, lstm_scale=2.0)

    for norm in ("offline_laplace_norm", "cumulative_laplace_norm", "offline_gaussian_norm", "cumulative_layer_norm"):
        c = small_fsn_cfg(norm)
        params = O.make_params_fsn(c, seed=4)
        out, fb_out = run_fsn(c, params, m)
        oo = O.fullsubnet_forward(params, c, m)
        print(f"fsn_small[{norm}]: oracle-vs-reference rel-L2 out={O.rel_l2(oo, out):.2e}")
        save(f"fsn_small_{norm}", mag=m, out=out, fb_out=fb_out, seed=4)

    # ---- 4. 3-layer sub-band LSTM (BASELINE config #5 building block; not reachable through
    #         the reference constructors, SURVEY.md 0.5 -> SequenceModel(num_layers=3) directly)
    rng = np.random.default_rng(11)
    x = rng.standard_normal((6, 10, 25))                                   # [N, I, T]
    p3 = O._lstm_params(np.random.default_rng(12), "sb_model", 10, 16, 3, 2)
    sm = SequenceModel(input_size=10, output_size=2, hidden_size=16, num_layers=3, bidirectional=False,
                       sequence_model="LSTM", output_activate_function=False)
    sm.load_state_dict({k[len("sb_model."):]: torch.from_numpy(v) for k, v in p3.items()}, strict=True)
    y = sm.double()(torch.from_numpy(x)).numpy()
    print("lstm3: oracle-vs-reference rel-L2:", O.rel_l2(O.seq_lstm(x, p3, "sb_model", 3, False), y))
    save("lstm3_small", x=x, out=y, seed=12)


def main_inferencer():
    """The reference's own inferencer (tools/inference.py:11-18: initialize_module(inferencer path) -> Inferencer(config, ckpt,
    out)()) with the reference model on the CPU, driven by its shipped config/inference.toml and a reference-format checkpoint
    of the seed-0 parameters: the int16 waveforms it writes for synthetic clips 0 and 1, the model calls it makes, and the
    state-dict keys and shapes of the reference class built from that TOML.  tests/test_reference_dropin.py checks the
    drop-in class against these."""
    import tempfile
    import toml
    from oracle import ref_loader
    root = ref_loader.reference_root()
    _, sf = ref_loader._stubs()
    sys.path.insert(0, os.path.dirname(HERE))                              # tests/dropin_dataset.py
    from audio_zen.utils import initialize_module
    cfg = toml.load(os.path.join(root, "config", "inference.toml"))
    params = O.make_params_plus(O.default_plus_config(), seed=0)
    calls = []
    with tempfile.TemporaryDirectory() as tmp:
        np.save(os.path.join(tmp, "clips.npy"), O.synth_clips(2).astype(np.float32))
        cfg["dataset"] = {"path": "dropin_dataset.Dataset", "args": {"npy_path": os.path.join(tmp, "clips.npy"), "sr": 16000}}
        torch.save({"model": {k: torch.from_numpy(v) for k, v in params.items()}, "epoch": 7}, os.path.join(tmp, "ckpt.tar"))
        inferencer = initialize_module(cfg["inferencer"]["path"], initialize=False)(cfg, os.path.join(tmp, "ckpt.tar"), os.path.join(tmp, "out"))
        inferencer.model.register_forward_hook(lambda m, i, o: calls.append([list(x.shape) for x in i] + [list(o.shape)]))
        sf.written.clear()
        inferencer()
        written = {os.path.relpath(k, os.path.join(tmp, "out")): v for k, v in sf.written.items()}
    names = sorted(written)
    assert names == ["enhanced_0007/clip0.wav", "enhanced_0007/clip1.wav"], names
    assert all(written[n][1] == 16000 and written[n][0].dtype == np.int16 for n in names)
    sd = FullSubNet_Plus(**cfg["model"]["args"]).state_dict()
    shapes = np.full((len(sd), 4), -1, np.int64)
    for j, v in enumerate(sd.values()):
        shapes[j, :v.dim()] = v.shape
    print(f"reference inferencer: {len(calls)} model calls {calls[0]}, wrote {names}")
    save("reference_inferencer", pcm=np.stack([written[n][0] for n in names]), files=np.array(names),
         model_calls=np.array(calls, np.int64), state_dict_keys=np.array(list(sd)), state_dict_shapes=shapes, seed=0)


def main_causal():
    """Round 2: the causal FullSubNet+ variant (SURVEY.md 8f rank 2): TCNBlock(causal=True) in all three full-band models."""
    ccfg = dict(small_plus_cfg(), causal_tcn=True)
    m, r, i = small_inputs(3, 33, 20, 7)
    params = O.make_params_plus(ccfg, seed=14)
    out, fb_in, fb_out = run_plus(ccfg, params, m, r, i)
    st = {}
    oo = O.fullsubnet_plus_forward(params, ccfg, m, r, i, stages=st)
    print(f"plus_small[causal TCN]: oracle-vs-reference rel-L2 out={O.rel_l2(oo, out):.2e} fb_out={O.rel_l2(st['fb_out'], fb_out):.2e}")
    nc = O.fullsubnet_plus_forward(params, dict(ccfg, causal_tcn=False), m, r, i)
    print(f"   (non-causal output differs by {O.rel_l2(nc, out):.2e})")
    save("plus_small_causal", out=out, fb_out=fb_out, seed=14)


if __name__ == "__main__":
    if "causal" in sys.argv[1:]:
        main_causal()
    elif "inferencer" in sys.argv[1:]:
        main_inferencer()
    else:
        main()
        main_causal()
        main_inferencer()
