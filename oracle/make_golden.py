"""Generate tests/golden/*.npz by running the REFERENCE itself (imported from /root/reference
with stubs for its missing optional dependencies, SURVEY.md Appendix A) on seeded inputs and
the oracle's deterministic sensitised weights.

Run in the build container only (needs /root/reference):

    python oracle/make_golden.py            # writes tests/golden/, prints oracle-vs-reference errors

The GPU box never runs this; it only reads the committed fixtures.
"""
from __future__ import annotations

import argparse
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("FDBM_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, HERE)


def import_reference():
    sys.path.insert(0, REF)

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m

    stub("pesq", pesq=lambda *a, **k: 0.0)
    stub("pystoi", stoi=lambda *a, **k: 0.0)

    class _LM(nn.Module):
        def save_hyperparameters(self, *a, **k):
            pass

    stub("pytorch_lightning", LightningModule=_LM,
         LightningDataModule=type("LDM", (), {"__init__": lambda s: None}))
    # fdbm.model additionally imports these (only BridgeModel._loss is used from it, as an unbound function)
    stub("torch_ema", ExponentialMovingAverage=object)
    stub("librosa", resample=None)
    stub("soundfile", write=None)
    stub("torch_pesq", PesqLoss=object)
    try:
        import torchaudio  # noqa: F401
    except Exception:
        stub("torchaudio", load=None)
    from fdbm.bridge import Bridge
    from fdbm.backbones import BackboneRegistry
    from fdbm.data_module import SpecsDataModule
    from fdbm.util.other import pad_spec, si_sdr
    return Bridge, BackboneRegistry, SpecsDataModule, pad_spec, si_sdr


def rel(a, b):
    a = torch.as_tensor(a); b = torch.as_tensor(b)
    return float((a - b).abs().pow(2).sum().sqrt() / b.abs().pow(2).sum().sqrt().clamp_min(1e-30))


def c2n(t):
    return t.detach().cpu().numpy()


class reference_tf32_convs:
    """Run the REFERENCE the way it runs on any Ampere-or-later GPU: cuDNN convolutions in TF32
    (torch.backends.cudnn.allow_tf32 defaults to True), i.e. both operands of every nn.Conv2d rounded to a 10-bit
    mantissa, fp32 accumulation; matmuls / einsum stay fp32 (allow_tf32 for matmul defaults to False).  On the CPU this
    is emulated by rounding the operands (round-to-nearest-even, the most favourable reading of TF32) in front of
    torch.nn.functional.conv2d.  The deviation of this run from the fp32 run is the yardstick for what a 16-bit-operand
    implementation may deviate: tests/golden/ref_tf32_deviation.json."""

    def __enter__(self):
        import fdbm_oracle as O
        import torch.nn.functional as F
        self.F, self.orig = F, F.conv2d

        def conv2d(x, w, *a, **k):
            return self.orig(O.round_tf32(x), O.round_tf32(w), *a, **k)
        F.conv2d = conv2d
        return self

    def __exit__(self, *a):
        self.F.conv2d = self.orig


class fixed_noise:
    """torch.randn_like replaced by a fixed sequence of draws (the samplers call it once per prior / step)."""

    def __init__(self, zs):
        self.zs = zs

    def __enter__(self):
        seq = iter(self.zs)
        self.orig = torch.randn_like
        torch.randn_like = lambda x, **k: next(seq)

    def __exit__(self, *a):
        torch.randn_like = self.orig


def main():
    import fdbm_oracle as O
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    Bridge, BackboneRegistry, SpecsDataModule, ref_pad_spec, ref_si_sdr = import_reference()
    os.makedirs(OUT, exist_ok=True)
    dm = SpecsDataModule(base_dir="/unused", n_fft=512, hop_length=256, num_frames=256,
                         window="sqrthann", gpu=False)
    scfg = O.SpecConfig()

    # ---- (1) spectral front/back end on synthetic utterances -------------------------------
    clean, noisy = O.synth_pair(0, n_samples=16000)           # 1 s -> 63 frames -> padded 64
    y = (noisy / noisy.abs().max())[None]
    S_ref = dm.stft(y)
    Y_ref = dm.spec_fwd(S_ref)
    Yp_ref = ref_pad_spec(Y_ref[None], mode="reflection")
    Yz_ref = ref_pad_spec(Y_ref[None], mode="zero_pad")
    wav_ref = dm.istft(dm.spec_back(Yp_ref.squeeze()), 16000)
    S_or = O.stft(y, scfg)
    Y_or = O.spec_fwd(S_or, scfg)
    Yp_or = O.pad_spec(Y_or[None], "reflection")
    wav_or = O.istft(O.spec_back(Yp_or.squeeze(), scfg), scfg, 16000)
    print("stft      oracle vs ref: max abs", float((S_or - S_ref).abs().max()), "bit-equal", bool(torch.equal(S_or, S_ref)))
    print("spec_fwd  oracle vs ref:", rel(Y_or, Y_ref))
    print("pad_spec  oracle vs ref: equal", bool(torch.equal(Yp_or, Yp_ref)),
          bool(torch.equal(O.pad_spec(Y_or[None], 'zero_pad'), O.pad_spec(Y_ref[None], 'zero_pad'))))
    print("istft     oracle vs ref:", rel(wav_or, wav_ref), float((wav_or - wav_ref).abs().max()))
    Yr_ref = ref_pad_spec(Y_ref[None], mode="replication")
    assert torch.equal(O.pad_spec(Y_or[None], "replication"), Yr_ref)
    np.savez_compressed(os.path.join(OUT, "spectral_1s.npz"),
                        wave=c2n(y), stft=c2n(S_ref), spec=c2n(Y_ref), spec_reflect=c2n(Yp_ref),
                        spec_zero=c2n(Yz_ref), spec_replicate=c2n(Yr_ref), wave_back=c2n(wav_ref))

    # ---- (2) coefficient tables --------------------------------------------------------------
    tables = {}
    for path, kw in (("sb", dict(noise_schedule="bb")), ("sb", dict(noise_schedule="ve")),
                     ("sb", dict(noise_schedule="vp")), ("sb", dict(noise_schedule="gmax")),
                     ("fm", dict())):
        for st in ("ode_ei", "sde_ei"):
            if path == "fm" and st == "sde_ei":
                continue
            for N in (1, 5, 10, 30):
                rb = Bridge(path, N=N, sampler_type=st, **kw)
                ob = O.Bridge(path, N=N, sampler_type=st, **kw)
                ts = torch.linspace(rb.start_time, rb.end_time, N + 1)
                rows = []
                tp = ts[0] * torch.ones(1)
                for t in ts[1:]:
                    tt = t * torch.ones(1)
                    if st == "ode_ei":
                        w = rb.path.sampling_param_ode_ei(tt, tp, 1, "cpu")
                    else:
                        w = list(rb.path.sampling_param_sde_ei(tt, tp, 1, "cpu"))
                        if t == ts[-1]:
                            w[2] = torch.zeros_like(w[2])
                    rows.append(torch.stack([w[0][0], w[1][0], w[2][0]]))
                    tp = tt
                tab = torch.stack(rows)
                key = f"{path}_{kw.get('noise_schedule', 'ot')}_{st}_N{N}"
                tables[key] = c2n(tab)
                same = torch.equal(tab, ob.coefficient_table())
                if not same:
                    print("coefficient table MISMATCH", key, (tab - ob.coefficient_table()).abs().max())
                # prior + path params
                tq = torch.tensor([0.03, 0.25, 0.5, 0.9999, 1.0])
                pr = rb.path.path_param(tq); po = ob.path.path_param(tq)
                assert all(torch.equal(a, b) for a, b in zip(pr, po)), key
                tables[key + "_pathparam"] = c2n(torch.stack(pr))
    print("coefficient tables:", len(tables), "entries, oracle bit-identical")
    np.savez_compressed(os.path.join(OUT, "coeff_tables.npz"), **tables)

    # ---- (3) FIR resampling identities vs the reference's upfirdn2d_native ---------------------
    from fdbm.backbones.ncsnpp_utils import up_or_down_sampling as uds
    xx = torch.randn(2, 3, 8, 12)
    print("fir_down2 vs ref:", float((O.fir_down2(xx) - uds.downsample_2d(xx, (1, 3, 3, 1), factor=2)).abs().max()))
    print("fir_up2   vs ref:", float((O.fir_up2(xx) - uds.upsample_2d(xx, (1, 3, 3, 1), factor=2)).abs().max()))
    np.savez_compressed(os.path.join(OUT, "fir.npz"), x=c2n(xx),
                        down=c2n(uds.downsample_2d(xx, (1, 3, 3, 1), factor=2)),
                        up=c2n(uds.upsample_2d(xx, (1, 3, 3, 1), factor=2)))

    # ---- (4) backbone + sampler at T=64 frames with sensitised weights -------------------------
    for name, pred in (("ncsnpp_v2", False), ("ncsnpp_v2_predictive", True)):
        cfg = O.NcsnppConfig(predictive=pred)
        sd = O.sensitised_state_dict(cfg, seed=0)
        net = BackboneRegistry.get_by_name(name)().eval()
        ref_sd = net.state_dict()
        assert set(ref_sd.keys()) == set(sd.keys()), (set(ref_sd) ^ set(sd))
        for k in ref_sd:
            assert tuple(ref_sd[k].shape) == tuple(sd[k].shape), k
        net.load_state_dict(sd, strict=True)
        g = torch.Generator().manual_seed(7)
        Y = Yp_ref.clone()                                                     # [1,1,257,64]
        with torch.no_grad():
            if pred:
                D_ref = net(Y)
                D_or = O.ncsnpp_forward(sd, cfg, Y)
                print(name, "forward oracle vs ref:", rel(D_or, D_ref), "out std", float(D_ref.abs().std()))
                np.savez_compressed(os.path.join(OUT, "predictive_T64.npz"), Y=c2n(Y), D=c2n(D_ref))
                continue
            xt = Y + 0.3 * torch.view_as_complex(torch.randn(1, 1, 257, 64, 2, generator=g))
            t = torch.tensor([0.6])
            D_ref = net(xt, Y, t)
            D_or = O.ncsnpp_forward(sd, cfg, xt, Y, t)
            print(name, "forward oracle vs ref:", rel(D_or, D_ref), "out std", float(D_ref.abs().std()))
            out = dict(Y=c2n(Y), xt=c2n(xt), t=c2n(t), D=c2n(D_ref))
            for path, st in (("sb", "ode_ei"), ("sb", "sde_ei"), ("fm", "ode_ei")):
                rb = Bridge(path, N=5, sampler_type=st)
                ob = O.Bridge(path, N=5, sampler_type=st)
                # deterministic noise: patch torch.randn_like through a shared generator sequence
                zg = torch.Generator().manual_seed(11)
                zs = [torch.view_as_complex(torch.randn(1, 1, 257, 64, 2, generator=zg)) * (0.5 ** 0.5)
                      for _ in range(6)]
                seq = iter(zs)
                orig = torch.randn_like
                torch.randn_like = lambda x, **k: next(seq)
                try:
                    s_ref = rb.sampler(lambda a, b, c: net(a, b, c), Y)
                finally:
                    torch.randn_like = orig
                s_or = ob.sampler(lambda a, b, c: O.ncsnpp_forward(sd, cfg, a, b, c), Y, z0=zs[0], zs=zs[1:])
                w_ref = dm.istft(dm.spec_back(s_ref.squeeze()), 16000)
                w_or = O.istft(O.spec_back(s_or.squeeze(), scfg), scfg, 16000)
                print(f"{name} sampler {path}/{st}: spec rel {rel(s_or, s_ref):.3e}  wave rel {rel(w_or, w_ref):.3e}")
                out[f"sample_{path}_{st}"] = c2n(s_ref)
                out[f"wave_{path}_{st}"] = c2n(w_ref)
                if st != "ode_ei" or path == "fm":
                    out[f"noise_{path}_{st}"] = c2n(torch.stack(zs))
            np.savez_compressed(os.path.join(OUT, "bridge_T64.npz"), **out)

            # ---- (4b) the other schedules and step counts the reference offers, same weights / input ----------------
            more = {}
            f_ref = lambda a, b, c: net(a, b, c)
            f_or = lambda a, b, c: O.ncsnpp_forward(sd, cfg, a, b, c)
            zg = torch.Generator().manual_seed(13)
            zs31 = [torch.view_as_complex(torch.randn(1, 1, 257, 64, 2, generator=zg)) * (0.5 ** 0.5) for _ in range(31)]
            for tag, path, st, N, kw in (("sb_ve_ode_ei_N5", "sb", "ode_ei", 5, dict(noise_schedule="ve")),
                                         ("sb_vp_ode_ei_N5", "sb", "ode_ei", 5, dict(noise_schedule="vp", c=0.3)),
                                         ("sb_gmax_ode_ei_N5", "sb", "ode_ei", 5, dict(noise_schedule="gmax")),
                                         ("sb_ve_sde_ei_N5", "sb", "sde_ei", 5, dict(noise_schedule="ve")),
                                         ("sb_bb_ode_ei_N1", "sb", "ode_ei", 1, {}),
                                         ("sb_bb_ode_ei_N10", "sb", "ode_ei", 10, {}),
                                         ("sb_bb_ode_ei_N30", "sb", "ode_ei", 30, {})):
                rb = Bridge(path, N=N, sampler_type=st, **kw)
                ob = O.Bridge(path, N=N, sampler_type=st, **kw)
                with fixed_noise(zs31):
                    s_ref = rb.sampler(f_ref, Y)
                s_or = ob.sampler(f_or, Y, z0=zs31[0], zs=zs31[1:])
                print(f"{name} sampler {tag}: oracle vs ref spec rel {rel(s_or, s_ref):.3e}")
                more["sample_" + tag] = c2n(s_ref)
            more["noise"] = c2n(torch.stack(zs31[:6]))
            np.savez_compressed(os.path.join(OUT, "bridge_T64_more.npz"), **more)

            # ---- (4c) the reference in ITS OWN reduced precision (TF32 convolutions) vs its fp32 run -------------------
            dev = {}
            with reference_tf32_convs():
                D_tf = net(xt, Y, t)
            with O.operand_rounding("tf32"):
                D_tf_or = O.ncsnpp_forward(sd, cfg, xt, Y, t)
            dev["forward_T64"] = rel(D_tf, D_ref)
            dev["forward_T64_oracle_emulation_vs_reference_emulation"] = rel(D_tf_or, D_tf)
            for path, st in (("sb", "ode_ei"), ("sb", "sde_ei"), ("fm", "ode_ei")):
                rb = Bridge(path, N=5, sampler_type=st)
                with fixed_noise(zs):
                    s32 = rb.sampler(f_ref, Y)
                with fixed_noise(zs), reference_tf32_convs():
                    stf = rb.sampler(f_ref, Y)
                dev[f"sampler_{path}_{st}_N5_T64"] = rel(stf, s32)
            # the other schedules / step counts of (4b), same inputs and noise draws
            for tag, path, st, N, kw in (("sb_ve_ode_ei_N5", "sb", "ode_ei", 5, dict(noise_schedule="ve")),
                                         ("sb_vp_ode_ei_N5", "sb", "ode_ei", 5, dict(noise_schedule="vp", c=0.3)),
                                         ("sb_gmax_ode_ei_N5", "sb", "ode_ei", 5, dict(noise_schedule="gmax")),
                                         ("sb_ve_sde_ei_N5", "sb", "sde_ei", 5, dict(noise_schedule="ve")),
                                         ("sb_bb_ode_ei_N1", "sb", "ode_ei", 1, {}),
                                         ("sb_bb_ode_ei_N10", "sb", "ode_ei", 10, {}),
                                         ("sb_bb_ode_ei_N30", "sb", "ode_ei", 30, {})):
                rb = Bridge(path, N=N, sampler_type=st, **kw)
                with fixed_noise(zs31), reference_tf32_convs():
                    stf = rb.sampler(f_ref, Y)
                dev[f"sampler_{tag}_T64"] = rel(stf, torch.from_numpy(more["sample_" + tag]))
            # BASELINE's own size: 4 s = 256 frames (utterance 0 of the synthetic set, reflection padding), default sampler and
            # the step sweep of configs[4]
            _, noisy4 = O.synth_pair(0)
            Y4 = ref_pad_spec(dm.spec_fwd(dm.stft((noisy4 / noisy4.abs().max())[None]))[None], mode="reflection")
            assert Y4.shape == (1, 1, 257, 256)
            for N in (5, 1, 10, 30):
                rb = Bridge("sb", N=N, sampler_type="ode_ei")
                s32 = rb.sampler(f_ref, Y4)
                with reference_tf32_convs():
                    stf = rb.sampler(f_ref, Y4)
                dev[f"sampler_sb_ode_ei_N{N}_T256"] = rel(stf, s32)
                print(f"  4 s, N={N}: reference TF32 vs fp32 {dev[f'sampler_sb_ode_ei_N{N}_T256']:.3e}", flush=True)
            import json
            dev["what"] = ("relative L2 deviation of the reference run with TF32 convolutions (its default GPU precision; emulated on the CPU "
                           "by rounding both operands of every nn.Conv2d to 10 mantissa bits, RNE) from the same reference run in fp32; "
                           "sensitised weights seed 0, inputs of bridge_T64.npz")
            with open(os.path.join(OUT, "ref_tf32_deviation.json"), "w") as fjs:
                json.dump(dev, fjs, indent=1)
            print("reference TF32-vs-fp32 deviations:", {k: (f"{v:.3e}" if isinstance(v, float) else "") for k, v in dev.items()})
    # ---- (5) the training loss head: BridgeModel._loss 'data_prediction_hybrid' (model.py:187-218) and its gradient ----
    import types as _types
    import fdbm.model as ref_model
    gl = torch.Generator().manual_seed(21)

    def spec(B=2, T=64):
        mag = torch.rand(B, 1, 257, T, generator=gl) ** 3 * 0.6
        ph = 2 * 3.14159265 * torch.rand(B, 1, 257, T, generator=gl)
        return torch.polar(mag, ph)
    x = spec()
    x_hat = x + 0.3 * spec()
    x_hat[:, :, 256] = 0
    fake_self = _types.SimpleNamespace(loss_type="data_prediction_hybrid", pesq_weight=0.0, data_module=dm,
                                       _backward_transform=dm.spec_back,
                                       to_audio=lambda s, length=None: dm.istft(dm.spec_back(s), length))
    leaf = x_hat.clone().requires_grad_(True)
    loss_ref = ref_model.BridgeModel._loss(fake_self, leaf, None, None, None, None, x)
    (g_ref,) = torch.autograd.grad(loss_ref, leaf)
    leaf2 = x_hat.clone().requires_grad_(True)
    loss_or = O.hybrid_loss(leaf2, x, scfg)
    (g_or,) = torch.autograd.grad(loss_or, leaf2)
    g_ref = torch.nan_to_num(g_ref); g_or = torch.nan_to_num(g_or)          # d angle / d z at the exact zeros of row 256
    print(f"hybrid loss reference {float(loss_ref):.6f} oracle {float(loss_or):.6f}; gradient oracle vs ref {rel(g_or, g_ref):.3e}")
    np.savez_compressed(os.path.join(OUT, "hybrid_loss.npz"), x=c2n(x), x_hat=c2n(x_hat), loss=np.float64(loss_ref.item()),
                        grad=c2n(g_ref))
    loss_goldens_data_prediction(ref_model, dm, x, x_hat, scfg)
    tfgridnet_goldens(BackboneRegistry)
    variant_goldens(BackboneRegistry)
    print("golden fixtures written to", OUT)
    for f in sorted(os.listdir(OUT)):
        print("  ", f, os.path.getsize(os.path.join(OUT, f)) // 1024, "KiB")


def loss_goldens_data_prediction(ref_model=None, dm=None, x=None, x_hat=None, scfg=None):
    """BridgeModel._loss 'data_prediction' (model.py:163-185, the argparse default; l1_weight 0.001, pesq_weight 0) and its gradient.
    Stand-alone: `python oracle/make_golden.py loss`."""
    import types as _types
    import fdbm_oracle as O
    if ref_model is None:
        import_reference()
        import fdbm.model as ref_model
        from fdbm.data_module import SpecsDataModule
        dm = SpecsDataModule(base_dir="/unused", n_fft=512, hop_length=256, num_frames=64, window="sqrthann", gpu=False)
        scfg = O.SpecConfig()
        gl = torch.Generator().manual_seed(21)

        def spec(B=2, T=64):
            mag = torch.rand(B, 1, 257, T, generator=gl) ** 3 * 0.6
            ph = 2 * 3.14159265 * torch.rand(B, 1, 257, T, generator=gl)
            return torch.polar(mag, ph)
        x = spec()
        x_hat = x + 0.3 * spec()
        x_hat[:, :, 256] = 0
    T = x.shape[-1]
    fake_dm = _types.SimpleNamespace(num_frames=T, hop_length=dm.hop_length)
    fake_self = _types.SimpleNamespace(loss_type="data_prediction", pesq_weight=0.0, l1_weight=0.001, data_module=fake_dm,
                                       to_audio=lambda s, length=None: dm.istft(dm.spec_back(s), length))
    leaf = x_hat.clone().requires_grad_(True)
    loss_ref = ref_model.BridgeModel._loss(fake_self, leaf, None, None, None, None, x)
    (g_ref,) = torch.autograd.grad(loss_ref, leaf)
    leaf2 = x_hat.clone().requires_grad_(True)
    loss_or = O.data_prediction_loss(leaf2, x, scfg, 0.001)
    (g_or,) = torch.autograd.grad(loss_or, leaf2)
    g_ref = torch.nan_to_num(g_ref); g_or = torch.nan_to_num(g_or)
    print(f"data_prediction loss reference {float(loss_ref):.6f} oracle {float(loss_or):.6f}; gradient oracle vs ref {rel(g_or, g_ref):.3e}")
    np.savez_compressed(os.path.join(OUT, "data_prediction_loss.npz"), x=c2n(x), x_hat=c2n(x_hat), loss=np.float64(loss_ref.item()),
                        grad=c2n(g_ref))


def loss_goldens_mel(seed=23):
    """BridgeModel._loss 'data_prediction_mel' / 'data_prediction_melphase' (model.py:220-251) through the reference's own
    MelSpectrogramLoss / PhaseLoss classes (loss.py), and their gradients.  The one substitution: `librosa.filters.mel` (absent
    here) is the oracle's restatement `mel_filterbank`, so these fixtures pin everything except the filterbank formula.
    Stand-alone: `python oracle/make_golden.py mel`."""
    import types as _types
    import fdbm_oracle as O
    import_reference()
    lib_filters = types.ModuleType("librosa.filters")
    lib_filters.mel = lambda sr, n_fft, n_mels, fmin=0.0, fmax=None: O.mel_filterbank(sr, n_fft, n_mels, fmin, fmax).numpy()
    sys.modules["librosa.filters"] = lib_filters
    sys.modules["librosa"].filters = lib_filters
    import fdbm.model as ref_model
    import fdbm.loss as ref_loss
    from fdbm.data_module import SpecsDataModule
    T = 64
    dm = SpecsDataModule(base_dir="/unused", n_fft=512, hop_length=256, num_frames=T, window="sqrthann", gpu=False)
    scfg = O.SpecConfig()
    gl = torch.Generator().manual_seed(seed)

    def spec(B=2):
        mag = torch.rand(B, 1, 257, T, generator=gl) ** 3 * 0.6
        ph = 2 * 3.14159265 * torch.rand(B, 1, 257, T, generator=gl)
        return torch.polar(mag, ph)
    x = spec()
    x_hat = x + 0.3 * spec()
    x_hat[:, :, 256] = 0
    mel_args = dict(n_mels=list(O.MEL_N_MELS), win_lengths=list(O.MEL_N_FFTS), hop_lengths=[n // 4 for n in O.MEL_N_FFTS],
                    n_ffts=list(O.MEL_N_FFTS), mag_weight=0.0, log_weight=1.0)
    out = {"x": c2n(x), "x_hat": c2n(x_hat)}
    for kind, with_phase in (("data_prediction_mel", False), ("data_prediction_melphase", True)):
        fake_dm = _types.SimpleNamespace(num_frames=T, hop_length=dm.hop_length, n_fft=512)
        fake_self = _types.SimpleNamespace(loss_type=kind, pesq_weight=0.0, l1_weight=0.001, data_module=fake_dm,
                                           to_audio=lambda s, length=None: dm.istft(dm.spec_back(s), length),
                                           loss_fn=ref_loss.MelSpectrogramLoss(**mel_args), loss_fn_mel=ref_loss.MelSpectrogramLoss(**mel_args),
                                           loss_fn_phase=ref_loss.PhaseLoss(nfreqs=257, frames=T))
        leaf = x_hat.clone().requires_grad_(True)
        loss_ref = ref_model.BridgeModel._loss(fake_self, leaf, None, None, None, None, x)
        (g_ref,) = torch.autograd.grad(loss_ref, leaf)
        leaf2 = x_hat.clone().requires_grad_(True)
        loss_or = O.data_prediction_mel_loss(leaf2, x, scfg, with_phase)
        (g_or,) = torch.autograd.grad(loss_or, leaf2)
        g_ref = torch.nan_to_num(g_ref); g_or = torch.nan_to_num(g_or)
        print(f"{kind}: loss reference {float(loss_ref):.6f} oracle {float(loss_or):.6f}; gradient oracle vs ref {rel(g_or, g_ref):.3e}")
        tag = "melphase" if with_phase else "mel"
        out["loss_" + tag] = np.float64(loss_ref.item()); out["grad_" + tag] = c2n(g_ref)
    np.savez_compressed(os.path.join(OUT, "mel_loss.npz"), **out)


def tfgridnet_goldens(BackboneRegistry=None):
    """(6) TF-GridNet: the reference's tfgridnet_5l32c100 / _predictive forward on [2,1,257,24] with the oracle's fixed weights,
    and the deviation a 10-bit-mantissa-operand run has from fp32 (cuDNN runs the reference's LSTMs and convolutions in TF32 on
    a GPU; emulated by the oracle's fp16-operand mode, whose NCSN++ counterpart is validated against the reference above)."""
    import json
    import fdbm_oracle as O
    if BackboneRegistry is None:
        BackboneRegistry = import_reference()[1]
    torch.set_num_threads(os.cpu_count())
    g = torch.Generator().manual_seed(5)
    Y = torch.view_as_complex(torch.randn(2, 1, 257, 24, 2, generator=g)) * 0.3
    X = Y + 0.2 * torch.view_as_complex(torch.randn(2, 1, 257, 24, 2, generator=g))
    t = torch.tensor([0.6, 0.31])
    out = dict(Y=c2n(Y), X=c2n(X), t=c2n(t))
    dev_path = os.path.join(OUT, "ref_tf32_deviation.json")
    dev = json.load(open(dev_path)) if os.path.exists(dev_path) else {}
    for name, pred in (("tfgridnet_5l32c100", False), ("tfgridnet_5l32c100_predictive", True)):
        cfg = O.TFGridNetConfig(predictive=pred)
        sd = O.tfgridnet_state_dict(cfg, seed=0)
        net = BackboneRegistry.get_by_name(name)().eval()
        assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}
        net.load_state_dict(sd, strict=True)
        with torch.no_grad():
            want = net(Y) if pred else net(X, Y, t)
            got = O.tfgridnet_forward(sd, cfg, Y) if pred else O.tfgridnet_forward(sd, cfg, X, Y, t)
            with O.operand_rounding("fp16"):
                low = O.tfgridnet_forward(sd, cfg, Y) if pred else O.tfgridnet_forward(sd, cfg, X, Y, t)
        print(f"{name}: oracle vs ref {rel(got, want):.3e}; 10-bit-operand emulation vs fp32 {rel(low, got):.3e}; out std {float(want.abs().std()):.3f}")
        out["D_pred" if pred else "D"] = c2n(want)
        dev[name + "_forward_T24"] = rel(low, got)
    np.savez_compressed(os.path.join(OUT, "tfgridnet_T24.npz"), **out)
    json.dump(dev, open(dev_path, "w"), indent=1)


def variant_goldens(BackboneRegistry=None):
    """(7) the nf = 64 size variant ncsnpp_v2_16M (ncsnpp_v2.py:418-433): reference forward at T = 64 with sensitised weights."""
    import fdbm_oracle as O
    if BackboneRegistry is None:
        BackboneRegistry = import_reference()[1]
    torch.set_num_threads(os.cpu_count())
    cfg = O.NcsnppConfig(nf=64, attn_resolutions=(0,))
    sd = O.sensitised_state_dict(cfg, seed=0)
    net = BackboneRegistry.get_by_name("ncsnpp_v2_16M")().eval()
    assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}
    net.load_state_dict(sd, strict=True)
    g = np.load(os.path.join(OUT, "bridge_T64.npz"))
    xt, Y, t = (torch.from_numpy(g[k]) for k in ("xt", "Y", "t"))
    with torch.no_grad():
        want = net(xt, Y, t)
        got = O.ncsnpp_forward(sd, cfg, xt, Y, t)
    print(f"ncsnpp_v2_16M forward oracle vs ref: {rel(got, want):.3e}  out std {float(want.abs().std()):.3f}  params {sum(v.numel() for v in sd.values())}")
    np.savez_compressed(os.path.join(OUT, "ncsnpp_16M_T64.npz"), D=c2n(want))
    # the nf = 96 variants ncsnpp_v2_5M (ncsnpp_v2.py:404-415) and ncsnpp_v2_37M (:436-448): 96 / 192-channel tensors, GroupNorm
    # groups of 4, 6, 9 and 12 channels
    out = {}
    for name, cfg in (("ncsnpp_v2_5M", O.NcsnppConfig(nf=96, ch_mult=(1, 1, 1, 1), num_res_blocks=1, attn_resolutions=(0,))),
                      ("ncsnpp_v2_37M", O.NcsnppConfig(nf=96))):
        sd = O.sensitised_state_dict(cfg, seed=0)
        net = BackboneRegistry.get_by_name(name)().eval()
        assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}
        net.load_state_dict(sd, strict=True)
        with torch.no_grad():
            want = net(xt, Y, t)
            got = O.ncsnpp_forward(sd, cfg, xt, Y, t)
        print(f"{name} forward oracle vs ref: {rel(got, want):.3e}  out std {float(want.abs().std()):.3f}  params {sum(v.numel() for v in sd.values())}")
        out[name] = c2n(want)
    np.savez_compressed(os.path.join(OUT, "ncsnpp_nf96_T64.npz"), **out)


DROPIN_PATHS = {"sb_bb": ("sb", dict(noise_schedule="bb")), "sb_ve": ("sb", dict(noise_schedule="ve")),
                "sb_vp": ("sb", dict(noise_schedule="vp", c=0.3)), "sb_gmax": ("sb", dict(noise_schedule="gmax")), "fm_ot": ("fm", dict())}
DROPIN_T = [0.03, 0.2, 0.55, 0.9999, 1.0]
DROPIN_PC = [(c, k, p) for c, k in (("ald", 1), ("langevin", 2), ("none", 1)) for p in ("euler_maruyama", "none")]


def argparse_defaults(cls):
    pa = argparse.ArgumentParser()
    cls.add_argparse_args(pa)
    return vars(pa.parse_args([]))


def dropin_soup(backbone_defaults):
    """The kwargs dictionary train.py hands a backbone (model.py:47-48 passes the values of ALL argparse groups at once)."""
    return dict(backbone_defaults, lr=1e-4, ema_decay=0.999, N=5, T=1.0, sampler_type="ode_ei", noise_schedule="bb",
                base_dir="/x", batch_size=8, n_fft=512, hop_length=256, gpus=1, loss_type="data_prediction_hybrid")


def dropin_bridge_inputs():
    g = torch.Generator().manual_seed(1)
    return tuple(torch.view_as_complex(torch.randn(5, 1, 9, 4, 2, generator=g)) for _ in range(3))     # s, y, x


def dropin_sampler_inputs():
    """A cheap stand-in model (B = 1, as the reference's broadcasting requires), its conditioning and a fixed noise sequence."""
    g = torch.Generator().manual_seed(3)
    y = torch.view_as_complex(torch.randn(1, 1, 17, 8, 2, generator=g)) * 0.3
    zs = [torch.view_as_complex(torch.randn(1, 1, 17, 8, 2, generator=g)) * 0.5 ** 0.5 for _ in range(40)]
    model = lambda x, yy, t: 0.6 * x + 0.3 * yy * torch.cos(t)[:, None, None, None] + 0.05 * x.abs()
    return y, zs, model


def dropin_record(Bridge, BackboneRegistry, SpecsDataModule):
    """What tests/test_reference_dropin.py compares against the original project's objects, computed with the classes given:
    argparse defaults, state_dict layout, requires_grad flags and per-tensor init statistics of the backbones, Bridge attributes
    and the scalar path maths on seeded inputs, pc / ode_int sampler outputs with a stand-in model, SpecsDataModule attributes.
    Returns {name: array}; the JSON-able facts are one JSON string under "meta"."""
    import itertools
    import json
    meta, out = {}, {}
    cls = BackboneRegistry.get_by_name("ncsnpp_v2")
    meta["ncsnpp_v2_args"] = argparse_defaults(cls)
    net = cls(**dropin_soup(meta["ncsnpp_v2_args"]))
    meta["ncsnpp_v2_shapes"] = {k: list(v.shape) for k, v in net.state_dict().items()}
    meta["ncsnpp_v2_requires_grad"] = [[n, p.requires_grad] for n, p in net.named_parameters()]
    torch.manual_seed(0)
    meta["ncsnpp_v2_init_std"] = {n: float(p.detach().std()) for n, p in cls().named_parameters() if p.numel() > 4096}
    meta["ncsnpp_v2_predictive_shapes"] = {k: list(v.shape) for k, v in
                                           BackboneRegistry.get_by_name("ncsnpp_v2_predictive")().state_dict().items()}
    meta["bridge_args"] = argparse_defaults(Bridge)
    s, y, x = dropin_bridge_inputs()
    t, t1 = torch.tensor(DROPIN_T), torch.tensor([0.4])
    for tag, (path, kw) in DROPIN_PATHS.items():
        b = Bridge(path, N=7, sampler_type="sde_ei", sampling_eps=1e-3, **kw)
        meta[tag] = {"attrs": {a: getattr(b, a) for a in ("N", "T", "sampler_type", "start_time", "end_time")},
                     "sampling_direction": b.path.sampling_direction, "path_T": b.path.T, "path_args": argparse_defaults(type(b.path))}
        vals = {"path_param": b.path.path_param(t), "std": [b._std(t)], "probability_path": b.probability_path(s, y, t),
                "score_fn": [b.score_fn(t, x, s, y)], "ode": [b.path.ode(t1, x[:1], s[:1], y[:1])]}
        if path == "sb":
            vals.update(sde=b.path.sde(t1, x[:1], s[:1], y[:1]), auxiliary_param=b.path.auxiliary_param(t1),
                        sampling_param_ode_ei=b.path.sampling_param_ode_ei(t1 * 0.5, t1, 1, "cpu"),
                        sampling_param_sde_ei=b.path.sampling_param_sde_ei(t1 * 0.5, t1, 1, "cpu"))
        for name, vs in vals.items():
            for i, v in enumerate(vs):
                out[f"{tag}_{name}_{i}"] = c2n(torch.as_tensor(v))
    y, zs, model = dropin_sampler_inputs()
    for corrector, steps, predictor in DROPIN_PC:
        with fixed_noise(zs):
            out[f"pc_{corrector}_{predictor}"] = c2n(Bridge("sb", N=4, sampler_type="pc").sampler(
                model, y, predictor_name=predictor, corrector_name=corrector, snr=0.3, corrector_steps=steps))
    with fixed_noise(itertools.repeat(zs[0])):
        out["ode_int_fm"] = c2n(Bridge("fm", sampler_type="ode_int").sampler(model, y, rtol=1e-6, atol=1e-6))
    dm = SpecsDataModule(base_dir="/unused", n_fft=512, hop_length=256, num_frames=256, window="sqrthann", gpu=False)
    meta["data_module"] = {a: getattr(dm, a) for a in ("normalize", "n_fft", "hop_length", "num_frames", "spec_factor",
                                                        "spec_abs_exponent", "transform_type")}
    meta["data_module_stft_kwargs"] = sorted(dm.stft_kwargs)
    out["data_module_window"] = c2n(dm.window)
    out["meta"] = np.array(json.dumps(meta, sort_keys=True))
    return out


def dropin_goldens():
    """(8) tests/golden/dropin.npz: dropin_record run on the original project's Bridge, BackboneRegistry and SpecsDataModule."""
    Bridge, BackboneRegistry, SpecsDataModule = import_reference()[:3]
    np.savez_compressed(os.path.join(OUT, "dropin.npz"), **dropin_record(Bridge, BackboneRegistry, SpecsDataModule))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "dropin":
        dropin_goldens()
    elif len(sys.argv) > 1 and sys.argv[1] == "tfgridnet":
        os.makedirs(OUT, exist_ok=True)
        tfgridnet_goldens()
    elif len(sys.argv) > 1 and sys.argv[1] == "mel":
        loss_goldens_mel()
    elif len(sys.argv) > 1 and sys.argv[1] == "loss":
        loss_goldens_data_prediction()
    elif len(sys.argv) > 1 and sys.argv[1] == "variants":
        variant_goldens()
    else:
        main()
