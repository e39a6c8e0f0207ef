"""Kernel-level parity: each C-ABI building block against the CPU oracle (torch fp32) on seeded
inputs.  Runs on the B200 only (`-m gpu`)."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import load_npz, nchw_to_ntfc, ntfc_to_nchw, rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from fdbm_b200 import _lib
    lb = _lib.load()
    _lib.check(lb.fdbm_check_device(), "fdbm_check_device")
    return lb


def _h16():
    from fdbm_b200 import _lib
    return _lib.operand_dtype()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check(lib, rc):
    assert rc == 0, lib.fdbm_last_error().decode()


# ------------------------------------------------------------------------------------------------
# spectral front / back end
# ------------------------------------------------------------------------------------------------
def test_framing_is_bit_exact(lib):
    """With an all-ones window and transform 'none' the DC bin of every frame is the plain sum of the
    framed samples; a one-hot 'window' returns the framed sample itself -> framing/reflection indices
    are checked bit-exactly against the oracle's index table."""
    import fdbm_oracle as O
    from fdbm_b200 import SpecsDataModule
    g = torch.Generator().manual_seed(3)
    for n in (4000, 16000, 16001):
        x = torch.randn(2, n, generator=g)
        idx = torch.from_numpy(O.frame_index(n, 512, 256))
        dm = SpecsDataModule(n_fft=512, hop_length=256, window="sqrthann")
        for tap in (0, 1, 255, 256, 511):
            w = torch.zeros(512); w[tap] = 1.0
            dm.windows.clear(); dm.window = w
            S = dm.stft(x.cuda())                       # [2, 257, M]
            got = S[:, 0, :].real.cpu()                 # DC bin = sum_k x[idx[m,k]] w[k] = x[idx[m,tap]]
            want = x[:, idx[:, tap]]
            assert torch.equal(got, want), (n, tap)


def test_stft_compress_matches_golden(lib, golden_dir):
    from fdbm_b200 import SpecsDataModule, pad_spec
    g = load_npz(f"{golden_dir}/spectral_1s.npz")
    dm = SpecsDataModule(n_fft=512, hop_length=256, window="sqrthann")
    y = torch.from_numpy(g["wave"]).cuda()
    S = dm.stft(y)
    ref = torch.from_numpy(g["stft"])
    assert float((S.cpu() - ref).abs().max()) <= 2e-5 * float(ref.abs().max())
    assert rel_l2(S, ref) < 1e-6
    Y = dm.spec_fwd(S)
    assert rel_l2(Y, g["spec"]) < 1e-6
    assert rel_l2(pad_spec(Y[None], "reflection"), g["spec_reflect"]) < 1e-6
    fused = dm.stft_compress(y, pad_mode="reflection")
    assert fused.shape == (1, 1, 257, 64)
    assert rel_l2(fused, g["spec_reflect"]) < 1e-6
    assert rel_l2(dm.stft_compress(y, pad_mode="zero_pad"), g["spec_zero"]) < 1e-6
    assert rel_l2(fused[..., 63], fused[..., 61]) < 1e-6        # reflection: frame 63 mirrors frame 61


def test_istft_matches_golden_and_roundtrip(lib, golden_dir):
    from fdbm_b200 import SpecsDataModule
    g = load_npz(f"{golden_dir}/spectral_1s.npz")
    dm = SpecsDataModule(n_fft=512, hop_length=256, window="sqrthann")
    Yp = torch.from_numpy(g["spec_reflect"]).cuda()
    w = dm.to_audio(Yp[0, 0], 16000)
    assert rel_l2(w, g["wave_back"].reshape(-1)) < 2e-6
    # unfused reference call sequence gives the same thing
    w2 = dm.istft(dm.spec_back(Yp[0, 0]), 16000)
    assert rel_l2(w2, w) < 1e-6
    # round trip at the BASELINE size (4 s, batch 8) and at 30 s: istft(stft(x)) == x
    for n, B in ((64000, 8), (480000, 2)):
        x = torch.randn(B, n, generator=torch.Generator().manual_seed(n)).cuda()
        back = dm.to_audio(dm.stft_compress(x, pad_mode="zero_pad")[:, 0], n)
        assert rel_l2(back, x) < 5e-6


def test_hop128_and_log_transform(lib):
    import fdbm_oracle as O
    from fdbm_b200 import SpecsDataModule
    x = torch.randn(3, 9000, generator=torch.Generator().manual_seed(5))
    # hop 512 is outside the fast STFT kernels: it runs the first-generation STFT
    for hop, tt in ((128, "exponent"), (256, "log"), (128, "none"), (512, "exponent")):
        cfg = O.SpecConfig(n_fft=512, hop_length=hop, window="hann", transform_type=tt)
        dm = SpecsDataModule(n_fft=512, hop_length=hop, window="hann", transform_type=tt)
        ref = O.spec_fwd(O.stft(x, cfg), cfg)
        got = dm.spec_fwd(dm.stft(x.cuda()))
        assert rel_l2(got, ref) < 2e-6, (hop, tt)
        if hop == 512:
            continue                          # frames without overlap: the Hann window's zeros make the iSTFT undefined
        wref = O.istft(O.spec_back(ref, cfg), cfg, 9000)
        wgot = dm.to_audio(got, 9000)
        assert rel_l2(wgot, wref) < 5e-6, (hop, tt)


# ------------------------------------------------------------------------------------------------
# bridge arithmetic
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_samples", [16000, 16001, 64000, 5000, 70001])
def test_stft_istft_various_lengths_vs_oracle(lib, n_samples):
    """Frame counts that are odd / even / not multiples of the 16-frame block, every pad mode, batch 3: the fused kernels
    against the oracle (data_module.py:173-229, other.py:76-90); iSTFT round trip reproduces the waveform."""
    import fdbm_oracle as O
    from fdbm_b200 import SpecsDataModule
    sc = O.SpecConfig()
    g = torch.Generator().manual_seed(n_samples)
    x = torch.randn(3, n_samples, generator=g) * torch.tensor([1.0, 0.03, 7.0])[:, None]
    dm = SpecsDataModule(n_fft=512, hop_length=256, window="sqrthann")
    S = dm.stft(x.cuda())
    want = O.stft(x, sc)
    assert S.shape == want.shape and rel_l2(S, want) < 2e-6
    n_pad = (64 - want.shape[-1] % 64) % 64
    modes = ("zero_pad", "reflection", "replication") if n_pad < want.shape[-1] else ("zero_pad", "replication")   # reflection needs pad < frames
    for mode in modes:
        got = dm.stft_compress(x.cuda(), pad_mode=mode)
        ref = O.pad_spec(O.spec_fwd(want, sc)[:, None], mode)
        assert got.shape == ref.shape and rel_l2(got, ref) < 2e-6, mode
        if mode == "zero_pad" and ref.shape[-1] > want.shape[-1]:
            assert float(got[..., want.shape[-1]:].abs().max()) == 0.0            # pad frames are exact zeros
    back = dm.to_audio(got[:, 0], n_samples)
    ref_back = O.istft(O.spec_back(ref[:, 0], sc), sc, n_samples)
    assert rel_l2(back, ref_back) < 3e-6
    y = dm.istft(S, n_samples)
    assert rel_l2(y, x) < 3e-6


def test_fused_normalise_rescale_clip(lib):
    """The elementwise glue of `enhance` folded into the kernels (infer_single.py:83-97, infer_folder.py:119-120): peak
    normalisation inside the STFT, `* norm` and the peak of the result inside the iSTFT, the clip rule as one kernel --
    against the reference's op sequence in torch, fixed- and variable-length batches."""
    import fdbm_oracle as O
    from fdbm_b200 import SpecsDataModule
    sc = O.SpecConfig()
    g = torch.Generator().manual_seed(11)
    lens = [40000, 33333, 25601, 40000]
    x = torch.zeros(4, 40000)
    for i, n in enumerate(lens):
        x[i, :n] = torch.randn(n, generator=g) * (0.2 + 3 * i)
    dm = SpecsDataModule(n_fft=512, hop_length=256, window="sqrthann")
    xd = x.cuda()
    lengths = torch.tensor(lens, dtype=torch.int32, device="cuda")
    norm = dm.wave_absmax(xd, lengths)
    assert torch.equal(norm.cpu(), x.abs().amax(1))
    assert torch.equal(dm.wave_absmax(xd).cpu(), x.abs().amax(1))
    Y = dm.stft_compress_var(xd, lengths, min(lens), max(lens), pad_mode="reflection", norm=norm)
    for i, n in enumerate(lens):
        yi = x[i:i + 1, :n] / x[i, :n].abs().max()
        ref = O.pad_spec(O.spec_fwd(O.stft(yi, sc), sc)[:, None], "reflection")
        T = ref.shape[-1]
        assert rel_l2(Y[i:i + 1, ..., :T], ref) < 2e-6, i
    # inverse with rescale + peak, then the clip rule
    spec = Y[:, 0] * 1.7                                             # push some rows above |x| = 1 after the rescale
    wave, peak = dm.to_audio_ex(spec, max(lens), lengths=lengths, norm=norm, want_peak=True)
    plain = dm.to_audio_var(spec, lengths, max(lens))
    want = plain * norm[:, None]
    assert rel_l2(wave, want) < 1e-6
    for i, n in enumerate(lens):
        assert float(wave[i, n:].abs().max() if n < max(lens) else 0.0) == 0.0
    assert torch.allclose(peak, wave.abs().amax(1), rtol=0, atol=0)
    clipped = dm.clip_rescale_(wave.clone(), peak, 0.95, lengths)
    ref_clip = torch.where(peak[:, None] > 1.0, wave / peak[:, None] * 0.95, wave)
    assert float(peak.max()) > 1.0 and torch.equal(clipped, ref_clip)


def test_bridge_step_bit_exact(lib):
    g = torch.Generator().manual_seed(1)
    shape = (2, 1, 257, 64)
    x = torch.view_as_complex(torch.randn(*shape, 2, generator=g))
    d = torch.view_as_complex(torch.randn(*shape, 2, generator=g))
    y = torch.view_as_complex(torch.randn(*shape, 2, generator=g))
    for coef in ((3999.45, 0.19994, -3998.65), (0.8166, 0.31001, -0.12661)):
        w = torch.tensor(coef, dtype=torch.float32)
        want = w[0] * x + w[1] * d + w[2] * y                       # bridge.py:83, CPU fp32
        dd, yd, wd = d.cuda(), y.cuda(), w.cuda()                   # keep alive: pointers are passed raw
        xs = x.clone().cuda()
        _check(lib, lib.fdbm_bridge_step(xs.data_ptr(), dd.data_ptr(), yd.data_ptr(), wd.data_ptr(),
                                         0, 0, 0, xs.numel(), _stream()))
        assert torch.equal(xs.cpu(), want)
        xs = x.clone().cuda()                                       # SDE with supplied noise, bridge.py:109
        _check(lib, lib.fdbm_bridge_step(xs.data_ptr(), dd.data_ptr(), yd.data_ptr(), wd.data_ptr(),
                                         1, 0, 0, xs.numel(), _stream()))
        assert torch.equal(xs.cpu(), want)


def test_prior_and_philox_noise(lib):
    from fdbm_b200 import Bridge
    y = torch.view_as_complex(torch.randn(4, 1, 257, 64, 2, generator=torch.Generator().manual_seed(2))).cuda()
    assert torch.equal(Bridge("sb").prior_sampling(y), y)           # SB: x_start == y exactly (sigma = 0, b = 1)
    br = Bridge("fm", noise="philox", seed=9)
    x0 = br.prior_sampling(y)
    z = (x0 - y * (1 - 1e-4)) / br.path.sigma_t(torch.tensor(1e-4)).item()
    zr = torch.view_as_real(z).flatten().cpu().double()
    assert abs(zr.mean()) < 5e-3 and abs(zr.var() - 0.5) < 5e-3     # complex normal: N(0, 1/2) per component
    assert abs((zr ** 4).mean() / zr.var() ** 2 - 3.0) < 0.05       # Gaussian kurtosis
    x1 = Bridge("fm", noise="philox", seed=9).prior_sampling(y)
    assert torch.equal(x0, x1)                                      # same seed, same stream -> same draw
    x2 = Bridge("fm", noise="philox", seed=10).prior_sampling(y)
    assert not torch.equal(x0, x2)


# ------------------------------------------------------------------------------------------------
# backbone building blocks
# ------------------------------------------------------------------------------------------------
def test_fir_resample(lib, golden_dir):
    g = load_npz(f"{golden_dir}/fir.npz")
    x = torch.from_numpy(g["x"])                                    # [2,3,8,12] NCHW (H=F, W=T)
    xin = nchw_to_ntfc(x).cuda()
    B, T, Fq, Cc = xin.shape
    for mode, key in ((1, "down"), (2, "up")):
        To, Fo = (T // 2, Fq // 2) if mode == 1 else (T * 2, Fq * 2)
        out = torch.empty(B, To, Fo, Cc, device="cuda")
        _check(lib, lib.fdbm_fir_resample(xin.data_ptr(), B, T, Fq, Cc, mode, out.data_ptr(), _stream()))
        assert float((ntfc_to_nchw(out).cpu() - torch.from_numpy(g[key])).abs().max()) < 1e-6


def _gn_ref(x, gamma, beta, silu):
    C_ = x.shape[1]
    y = F.group_norm(x, min(C_ // 4, 32), gamma, beta, eps=1e-6)
    return F.silu(y) if silu else y


@pytest.mark.parametrize("C1,C2,mode", [(128, 0, 0), (256, 128, 0), (256, 256, 0), (128, 0, 1), (256, 0, 2), (256, 128, 2)])
def test_groupnorm_act(lib, C1, C2, mode):
    import fdbm_oracle as O
    g = torch.Generator().manual_seed(C1 + C2 + mode)
    B, T, Fq = 2, 12, 16
    Cc = C1 + C2
    x = torch.randn(B, Cc, Fq, T, generator=g) * 1.5 + 0.3
    gamma = 1 + 0.1 * torch.randn(Cc, generator=g)
    beta = 0.1 * torch.randn(Cc, generator=g)
    act = _gn_ref(x, gamma, beta, True)
    raw = x
    if mode == 1:
        act, raw = O.fir_down2(act), O.fir_down2(raw)
    elif mode == 2:
        act, raw = O.fir_up2(act), O.fir_up2(raw)
    s1 = nchw_to_ntfc(x[:, :C1]).cuda()
    s2 = nchw_to_ntfc(x[:, C1:]).cuda() if C2 else None
    sums1 = torch.empty(B, C1, 2, dtype=torch.float64, device="cuda")
    _check(lib, lib.fdbm_channel_stats(s1.data_ptr(), B, T, Fq, C1, sums1.data_ptr(), _stream()))
    want = torch.stack([x[:, :C1].double().sum((2, 3)), x[:, :C1].double().pow(2).sum((2, 3))], -1)
    assert rel_l2(sums1, want) < 1e-6
    sums2 = None
    if C2:
        sums2 = torch.empty(B, C2, 2, dtype=torch.float64, device="cuda")
        _check(lib, lib.fdbm_channel_stats(s2.data_ptr(), B, T, Fq, C2, sums2.data_ptr(), _stream()))
    To, Fo = act.shape[3], act.shape[2]
    a_out = torch.empty(B, To, Fo, Cc, dtype=_h16(), device="cuda")
    r_out = torch.empty_like(a_out)
    gd, bd = gamma.cuda(), beta.cuda()
    _check(lib, lib.fdbm_groupnorm_act(s1.data_ptr(), sums1.data_ptr(), C1, s2.data_ptr() if C2 else None,
                                       sums2.data_ptr() if C2 else None, C2, gd.data_ptr(),
                                       bd.data_ptr(), B, T, Fq, 1, mode, a_out.data_ptr(), r_out.data_ptr(),
                                       _stream()))
    assert rel_l2(ntfc_to_nchw(a_out.float()), act) < 4e-3            # 16-bit output rounding
    assert rel_l2(ntfc_to_nchw(r_out.float()), raw) < 4e-3
    assert float((ntfc_to_nchw(a_out.float()).cpu() - act).abs().max()) < 0.03


@pytest.mark.parametrize("C1,C2,mode,T,Fq", [(128, 0, 1, 12, 16), (256, 0, 1, 36, 8), (256, 0, 2, 12, 16), (256, 128, 2, 20, 6),
                                             (256, 256, 2, 4, 4), (128, 0, 1, 4, 4)])
def test_gn_resample_h16(lib, C1, C2, mode, T, Fq):
    """Resampling blocks' input pass from the 16-bit stream (layerspp.py:242-257 with up/down): compared with
    torch GroupNorm -> SiLU -> FIR on the same 16-bit input."""
    import fdbm_oracle as O
    g = torch.Generator().manual_seed(C1 + C2 + mode + T)
    B = 2
    Cc = C1 + C2
    x = (torch.randn(B, Cc, Fq, T, generator=g) * 1.5 + 0.3).to(_h16()).float()
    gamma = 1 + 0.1 * torch.randn(Cc, generator=g)
    beta = 0.1 * torch.randn(Cc, generator=g)
    act = _gn_ref(x, gamma, beta, True)
    act, raw = (O.fir_down2(act), O.fir_down2(x)) if mode == 1 else (O.fir_up2(act), O.fir_up2(x))
    s1 = nchw_to_ntfc(x[:, :C1]).to(_h16()).cuda()
    s2 = nchw_to_ntfc(x[:, C1:]).to(_h16()).cuda() if C2 else None
    sums1 = torch.stack([x[:, :C1].double().sum((2, 3)), x[:, :C1].double().pow(2).sum((2, 3))], -1).cuda()
    sums2 = torch.stack([x[:, C1:].double().sum((2, 3)), x[:, C1:].double().pow(2).sum((2, 3))], -1).cuda() if C2 else None
    To, Fo = act.shape[3], act.shape[2]
    a_out = torch.full((B, To, Fo, Cc), float("nan"), dtype=_h16(), device="cuda")
    r_out = torch.full_like(a_out, float("nan"))
    gd, bd = gamma.cuda(), beta.cuda()
    table = torch.empty(B * Cc * 2, device="cuda")
    _check(lib, lib.fdbm_gn_resample_h16(s1.data_ptr(), sums1.data_ptr(), C1, s2.data_ptr() if C2 else None,
                                         sums2.data_ptr() if C2 else None, C2, gd.data_ptr(), bd.data_ptr(), table.data_ptr(),
                                         B, T, Fq, mode, a_out.data_ptr(), r_out.data_ptr(), _stream()))
    assert rel_l2(ntfc_to_nchw(r_out.float()), raw) < 1e-3            # 16-bit output rounding only
    assert rel_l2(ntfc_to_nchw(a_out.float()), act) < 4e-3            # + packed 16-bit SiLU
    assert float((ntfc_to_nchw(a_out.float()).cpu() - act).abs().max()) < 0.03


def _conv_case(lib, B, T, Fq, C1, k, C2, Cout, residual, bias_b, seed):
    g = torch.Generator().manual_seed(seed)
    x1 = torch.randn(B, C1, Fq, T, generator=g).to(_h16()).float()
    w1 = (torch.randn(Cout, C1, k, k, generator=g) / (C1 * k * k) ** 0.5).to(_h16()).float()
    bias = torch.randn(Cout, generator=g)
    ref = F.conv2d(x1.double(), w1.double(), None, padding=k // 2)
    x2 = w2 = None
    if C2:
        x2 = torch.randn(B, C2, Fq, T, generator=g).to(_h16()).float()
        w2 = (torch.randn(Cout, C2, 1, 1, generator=g) / C2 ** 0.5).to(_h16()).float()
        ref = ref + F.conv2d(x2.double(), w2.double())
    ref = ref + bias.double()[None, :, None, None]
    bb = res = None
    if bias_b:
        bb = torch.randn(B, Cout, generator=g)
        ref = ref + bb.double()[:, :, None, None]
    if residual:
        res = torch.randn(B, Cout, Fq, T, generator=g)
        ref = ref + res.double()
    scale = 0.70710678118654752 if residual or C2 else 1.0
    ref = (ref * scale).float()

    nbytes = C.c_int64()
    _check(lib, lib.fdbm_pack_conv_weights(None, C1, k, None, C2, Cout, None, C.byref(nbytes), None))
    wpack = torch.empty(nbytes.value // 2, dtype=_h16(), device="cuda")
    w1d = w1.cuda()
    w2d = w2.cuda() if C2 else None
    _check(lib, lib.fdbm_pack_conv_weights(w1d.data_ptr(), C1, k, w2d.data_ptr() if C2 else None, C2, Cout,
                                           wpack.data_ptr(), None, _stream()))
    in1 = nchw_to_ntfc(x1).to(_h16()).cuda()
    in2 = nchw_to_ntfc(x2).to(_h16()).cuda() if C2 else None
    out = torch.full((B, T, Fq, Cout), float("nan"), device="cuda")
    out16 = torch.empty(B, T, Fq, Cout, dtype=_h16(), device="cuda")
    sums = torch.empty(B, Cout, 2, dtype=torch.float64, device="cuda")
    biasd = bias.cuda()
    bbd = bb.cuda() if bias_b else None
    resd = nchw_to_ntfc(res).cuda() if residual else None
    _check(lib, lib.fdbm_conv_igemm(in1.data_ptr(), C1, k, in2.data_ptr() if C2 else None, C2, wpack.data_ptr(),
                                    biasd.data_ptr(), bbd.data_ptr() if bias_b else None,
                                    resd.data_ptr() if residual else None, scale, B, T, Fq, Cout, out.data_ptr(),
                                    out16.data_ptr(), sums.data_ptr(), _stream()))
    torch.cuda.synchronize()
    got = ntfc_to_nchw(out).cpu()
    assert torch.isfinite(got).all()
    err = rel_l2(got, ref)
    assert err < 2e-5, f"fp32-accumulated conv differs from the fp64 reference: rel L2 {err}"
    assert rel_l2(ntfc_to_nchw(out16.float()), ref) < 4e-3
    want = torch.stack([ref.double().sum((2, 3)), ref.double().pow(2).sum((2, 3))], -1)
    assert rel_l2(sums, want) < 1e-4


@pytest.mark.parametrize("B,T,Fq,C1,k,C2,Cout,residual,bias_b", [
    (1, 16, 8, 64, 3, 0, 128, False, False),        # one M-tile, one K-block: the minimal case
    (1, 32, 16, 128, 3, 0, 128, False, True),       # Conv_0 shape class (FiLM bias)
    (2, 16, 16, 128, 3, 0, 128, True, False),       # Conv_1 with identity shortcut
    (1, 16, 16, 256, 3, 128, 256, False, False),    # Conv_1 + fused Conv_2 1x1, two N blocks
    (3, 20, 12, 128, 3, 0, 128, False, False),      # ragged tiles in both directions, odd tile count
    (2, 4, 4, 256, 3, 0, 256, True, False),         # bottleneck-sized image (smaller than one tile)
    (1, 16, 16, 256, 1, 0, 256, True, False),       # NIN / 1x1 with residual
    (1, 64, 64, 512, 3, 0, 256, False, True),       # up-path Conv_0 (concat input), many tiles, phase wrap
])
def test_conv_igemm(lib, B, T, Fq, C1, k, C2, Cout, residual, bias_b):
    _conv_case(lib, B, T, Fq, C1, k, C2, Cout, residual, bias_b, seed=B * 1000 + T + C1)


@pytest.mark.parametrize("B,T,Fq,C1,k,Cout,silu", [
    (2, 16, 16, 128, 3, 128, 1),       # GroupNorm_1 + SiLU + Conv_1 shape class
    (1, 20, 12, 256, 3, 256, 1),       # ragged tiles: halo pixels outside the image must stay exactly zero
    (2, 16, 16, 256, 1, 256, 0),       # attention GroupNorm (no activation) + NIN
])
def test_gn_table_then_conv_igemm_ex_on_load(lib, B, T, Fq, C1, k, Cout, silu):
    """conv(act(GroupNorm(x))) with the normalisation applied to the operand tile in shared memory
    (layerspp.py:242-246): fdbm_gn_table builds the (scale, shift) table, fdbm_conv_igemm_ex applies it on load.
    Compared with torch GroupNorm -> SiLU -> conv2d in fp64 on the same 16-bit x."""
    g = torch.Generator().manual_seed(B * 100 + T + C1 + k)
    x = (torch.randn(B, C1, Fq, T, generator=g) * 1.7 + 0.4).to(_h16()).float()
    gamma = 1 + 0.1 * torch.randn(C1, generator=g)
    beta = 0.1 * torch.randn(C1, generator=g)
    w = (torch.randn(Cout, C1, k, k, generator=g) / (C1 * k * k) ** 0.5).to(_h16()).float()
    bias = torch.randn(Cout, generator=g)
    a = F.group_norm(x.double(), 32, gamma.double(), beta.double(), eps=1e-6)
    if silu:
        a = F.silu(a)
    ref = (F.conv2d(a, w.double(), bias.double(), padding=k // 2)).float()

    nbytes = C.c_int64()
    _check(lib, lib.fdbm_pack_conv_weights(None, C1, k, None, 0, Cout, None, C.byref(nbytes), None))
    wpack = torch.empty(nbytes.value // 2, dtype=_h16(), device="cuda")
    wd = w.cuda()
    _check(lib, lib.fdbm_pack_conv_weights(wd.data_ptr(), C1, k, None, 0, Cout, wpack.data_ptr(), None, _stream()))
    xd = nchw_to_ntfc(x).to(_h16()).cuda()
    sums1 = torch.stack([x.double().sum((2, 3)), x.double().pow(2).sum((2, 3))], -1).cuda()
    gd, bd, biasd = gamma.cuda(), beta.cuda(), bias.cuda()
    table = torch.empty(B * C1 * 2, device="cuda")
    out = torch.full((B, T, Fq, Cout), float("nan"), device="cuda")
    sums = torch.empty(B, Cout, 2, dtype=torch.float64, device="cuda")
    from fdbm_b200 import _lib
    _check(lib, lib.fdbm_gn_table(sums1.data_ptr(), C1, None, 0, gd.data_ptr(), bd.data_ptr(), 0, B, T * Fq, table.data_ptr(),
                                  None, _stream()))
    d = _lib.ConvDesc(n_seg=1, wpack=wpack.data_ptr(), bias=biasd.data_ptr(), scale=1.0, B=B, T=T, F=Fq, Cout=Cout,
                      out_f32=out.data_ptr(), sums=sums.data_ptr())
    d.seg[0] = _lib.ConvSeg(in_=xd.data_ptr(), C=C1, taps=k * k, norm_tab=table.data_ptr(), tab_stride=C1, act=silu)
    _check(lib, lib.fdbm_conv_igemm_ex(C.byref(d), _stream()))
    torch.cuda.synchronize()
    got = ntfc_to_nchw(out).cpu()
    assert torch.isfinite(got).all()
    err = rel_l2(got, ref)
    assert err < 1e-3, f"normalise-on-load conv differs from GroupNorm->SiLU->conv2d: rel L2 {err}"   # operand rounding 2^-12
    want = torch.stack([ref.double().sum((2, 3)), ref.double().pow(2).sum((2, 3))], -1)
    assert rel_l2(sums, want) < 2e-3


def test_attention(lib):
    g = torch.Generator().manual_seed(4)
    B, L, Cc = 2, 96, 256
    q, k, v = (torch.randn(B, L, Cc, generator=g).to(_h16()) for _ in range(3))
    w = torch.softmax(torch.einsum("bqc,bkc->bqk", q.float(), k.float()) * Cc ** -0.5, dim=-1)
    ref = torch.einsum("bqk,bkc->bqc", w, v.float())
    o = torch.empty(B, L, Cc, dtype=_h16(), device="cuda")
    qd, kd, vd = q.cuda(), k.cuda(), v.cuda()
    _check(lib, lib.fdbm_attention(qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), B, L, Cc, o.data_ptr(), _stream()))
    assert rel_l2(o.float(), ref) < 5e-3


# ------------------------------------------------------------------------------------------------
# training step: convolution gradients vs torch autograd (fp64) on the same 16-bit operands
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,T,Fq,Cin,k,Cout", [
    (1, 16, 8, 64, 3, 128),          # one pixel tile, one 64-channel box: the minimal MN-major case
    (2, 16, 16, 128, 3, 128),        # ResnetBlock Conv_0 / Conv_1 class
    (2, 20, 12, 256, 3, 128),        # ragged tiles (zero-filled halo and tile tails), two Cin blocks
    (1, 32, 32, 128, 1, 256),        # 1x1 shortcut (Conv_2), two Cout blocks
    (3, 64, 64, 128, 3, 128),        # many tiles per split
])
def test_conv_wgrad(lib, B, T, Fq, Cin, k, Cout):
    g = torch.Generator().manual_seed(7 * B + T + Cin + k)
    x = torch.randn(B, Cin, Fq, T, generator=g).to(_h16()).double()
    dy = torch.randn(B, Cout, Fq, T, generator=g).to(_h16()).double()
    w = torch.zeros(Cout, Cin, k, k, dtype=torch.float64, requires_grad=True)
    F.conv2d(x, w, None, padding=k // 2).backward(dy)
    ref = w.grad.float()
    xd = nchw_to_ntfc(x.float()).to(_h16()).cuda()
    dyd = nchw_to_ntfc(dy.float()).to(_h16()).cuda()
    ws = torch.empty(lib.fdbm_conv_wgrad_workspace_bytes(Cout, Cin, k, B, T, Fq) // 4, device="cuda")
    dw = torch.full((Cout, Cin, k, k), 0.5, device="cuda")                 # accumulates: dw += scale * grad
    _check(lib, lib.fdbm_conv_wgrad(dyd.data_ptr(), Cout, xd.data_ptr(), Cin, k, B, T, Fq, 2.0, dw.data_ptr(),
                                    ws.data_ptr(), _stream()))
    torch.cuda.synchronize()
    got = (dw.cpu() - 0.5) / 2.0
    err = rel_l2(got, ref)
    assert err < 2e-5, f"wgrad differs from autograd: rel L2 {err}"


@pytest.mark.parametrize("B,T,Fq,Cin,k,Cout", [
    (2, 16, 16, 128, 3, 128),
    (1, 20, 12, 256, 3, 128),        # ragged tiles; Cin (= dgrad output channels) in two N blocks
    (1, 16, 16, 128, 1, 256),        # 1x1
])
def test_conv_dgrad(lib, B, T, Fq, Cin, k, Cout):
    """dX = conv(dY, W transposed + flipped) through the forward tcgen05 kernel, accumulated onto an existing gradient."""
    g = torch.Generator().manual_seed(11 * B + T + Cin + k)
    w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5).to(_h16()).double()
    dy = torch.randn(B, Cout, Fq, T, generator=g).to(_h16()).double()
    x = torch.zeros(B, Cin, Fq, T, dtype=torch.float64, requires_grad=True)
    F.conv2d(x, w, None, padding=k // 2).backward(dy)
    prev = torch.randn(B, Cin, Fq, T, generator=g)
    ref = (x.grad + prev.double()).float()
    nbytes = C.c_int64()
    _check(lib, lib.fdbm_pack_conv_weights_dgrad(None, Cout, Cin, k, None, C.byref(nbytes), None))
    wpack = torch.empty(nbytes.value // 2, dtype=_h16(), device="cuda")
    wd = w.float().cuda()
    _check(lib, lib.fdbm_pack_conv_weights_dgrad(wd.data_ptr(), Cout, Cin, k, wpack.data_ptr(), None, _stream()))
    dyd = nchw_to_ntfc(dy.float()).to(_h16()).cuda()
    acc = nchw_to_ntfc(prev).cuda().contiguous()
    zero_bias = torch.zeros(Cin, device="cuda")
    _check(lib, lib.fdbm_conv_igemm(dyd.data_ptr(), Cout, k, None, 0, wpack.data_ptr(), zero_bias.data_ptr(), None,
                                    acc.data_ptr(), 1.0, B, T, Fq, Cin, acc.data_ptr(), None, None, _stream()))
    torch.cuda.synchronize()
    err = rel_l2(ntfc_to_nchw(acc).cpu(), ref)
    assert err < 2e-5, f"dgrad differs from autograd: rel L2 {err}"


# ------------------------------------------------------------------------------------------------
# the skinny layers of NCSN++ (SURVEY 8 A7e / A7f) at kernel level, against the torch ops the reference runs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c_in", [4, 2])
def test_pack_and_im2col_input_first_convolution(lib, c_in):
    """ncsnpp_v2.py:247-250 + :278 (ncsnpp_v2_predictive.py for 2 channels): input packing (bit-exact), the im2col K-block (exact up to
    the 16-bit rounding of its entries) and the whole 3x3 input convolution through fdbm_conv_igemm against F.conv2d."""
    g = torch.Generator().manual_seed(11)
    B, T, Fb, nf = 2, 48, 257, 128
    x = torch.view_as_complex(torch.randn(B, 1, Fb, T, 2, generator=g)).cuda()
    y = torch.view_as_complex(torch.randn(B, 1, Fb, T, 2, generator=g)).cuda()
    packed = torch.empty(B, T, 256, c_in, device="cuda")
    _check(lib, lib.fdbm_pack_input(torch.view_as_real(x).data_ptr(), torch.view_as_real(y).data_ptr() if c_in == 4 else None, B, T, Fb, 256, c_in,
                                    packed.data_ptr(), _stream()))
    parts = (x.real, x.imag, y.real, y.imag) if c_in == 4 else (x.real, x.imag)
    h_in = torch.cat(parts, dim=1)[:, :, :256, :]                                # [B, c_in, 256, T]
    assert torch.equal(packed, nchw_to_ntfc(h_in))
    cols = torch.empty(B, T, 256, 64, dtype=_h16(), device="cuda")
    _check(lib, lib.fdbm_im2col_input(packed.data_ptr(), c_in, B, T, 256, cols.data_ptr(), _stream()))
    ref_cols = F.unfold(h_in, 3, padding=1).reshape(B, c_in, 9, 256, T)           # [B, ci, kf*3+kt, F, T]
    ref_cols = ref_cols.permute(0, 4, 3, 2, 1).reshape(B, T, 256, 9 * c_in)       # k = tap * c_in + ci
    torch.cuda.synchronize()
    assert torch.equal(cols[..., :9 * c_in].float(), ref_cols.to(_h16()).float()) and not cols[..., 9 * c_in:].any()
    # the convolution: weights OIHW (H = frequency, W = frames) packed with ksize -2, one 64-wide K-block
    w = (torch.randn(nf, c_in, 3, 3, generator=g) * 0.2).cuda(); bias = torch.randn(nf, generator=g).cuda()
    nb = C.c_int64(); lib.fdbm_pack_conv_weights(None, c_in, -2, None, 0, nf, None, C.byref(nb), None)
    wp = torch.empty(nb.value // 2, dtype=_h16(), device="cuda")
    _check(lib, lib.fdbm_pack_conv_weights(w.data_ptr(), c_in, -2, None, 0, nf, wp.data_ptr(), C.byref(nb), _stream()))
    out = torch.empty(B, T, 256, nf, device="cuda")
    _check(lib, lib.fdbm_conv_igemm(cols.data_ptr(), 64, 1, None, 0, wp.data_ptr(), bias.data_ptr(), None, None, 1.0, B, T, 256, nf,
                                    out.data_ptr(), None, None, _stream()))
    want = F.conv2d(h_in.double(), w.double(), bias.double(), padding=1).float()
    err = rel_l2(ntfc_to_nchw(out), want)
    print(f"input convolution {c_in} -> {nf}: rel L2 {err:.2e}")
    assert err < 1e-3


def test_time_embedding_and_film_rows(lib):
    """layerspp.py:32-41 + ncsnpp_v2.py:252-270 + layerspp.py:263: Fourier features of log t, the two-layer MLP, and all Dense_0 FiLM
    rows at once, in fp32 against the same torch ops."""
    g = torch.Generator().manual_seed(12)
    B, nf, rows = 5, 128, 49 * 128 + 64
    t = (0.03 + 0.97 * torch.rand(B, generator=g)).cuda()
    W = (torch.randn(nf, generator=g) * 16).cuda()
    w1 = (torch.randn(4 * nf, 2 * nf, generator=g) * 0.05).cuda(); b1 = torch.randn(4 * nf, generator=g).cuda() * 0.1
    w2 = (torch.randn(4 * nf, 4 * nf, generator=g) * 0.05).cuda(); b2 = torch.randn(4 * nf, generator=g).cuda() * 0.1
    act = torch.empty(B, 4 * nf, device="cuda")
    _check(lib, lib.fdbm_time_embedding(t.data_ptr(), W.data_ptr(), nf, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), B,
                                        act.data_ptr(), _stream()))
    proj = torch.log(t)[:, None] * W[None, :] * 2 * np.pi
    emb = torch.cat([torch.sin(proj), torch.cos(proj)], dim=-1)
    temb = F.linear(F.silu(F.linear(emb, w1, b1)), w2, b2)
    want = F.silu(temb)
    e1 = rel_l2(act, want)
    dw = (torch.randn(rows, 4 * nf, generator=g) * 0.05).cuda(); db = torch.randn(rows, generator=g).cuda()
    film = torch.empty(B, rows, device="cuda")
    _check(lib, lib.fdbm_film_rows(act.data_ptr(), dw.data_ptr(), db.data_ptr(), B, 4 * nf, rows, film.data_ptr(), _stream()))
    e2 = rel_l2(film, F.linear(act, dw, db))
    print(f"time embedding rel L2 {e1:.2e}, FiLM rows {e2:.2e}")
    # |2 pi W log t| reaches ~1e2 rad: an fp32 rounding of the argument is ~1e-5 rad, which is what sin / cos can agree to
    assert e1 < 2e-4 and e2 < 1e-5


@pytest.mark.parametrize("c_pyr", [4, 2])
def test_combine_and_output_layer(lib, c_pyr):
    """layerspp.py:52-59 (Combine, 'sum') and ncsnpp_v2.py:392-399 (output 1x1 convolution, un-packing to the complex layout with the
    zero Nyquist row) against F.conv2d."""
    g = torch.Generator().manual_seed(13)
    B, T, Fq, Cc = 2, 40, 64, 256
    h = torch.randn(B, Cc, Fq, T, generator=g).cuda(); pyr = torch.randn(B, c_pyr, Fq, T, generator=g).cuda()
    w = (torch.randn(Cc, c_pyr, 1, 1, generator=g) * 0.3).cuda(); b = torch.randn(Cc, generator=g).cuda()
    hk = nchw_to_ntfc(h); pk = nchw_to_ntfc(pyr)
    _check(lib, lib.fdbm_combine(hk.data_ptr(), pk.data_ptr(), c_pyr, w.reshape(Cc, c_pyr).contiguous().data_ptr(), b.data_ptr(), B, T, Fq, Cc, _stream()))
    # (fp64 references: cuDNN convolutions run in TF32 by default, these kernels are fp32 FMA)
    e1 = rel_l2(ntfc_to_nchw(hk), (F.conv2d(pyr.double(), w.double(), b.double()) + h.double()).float())
    T2, Fq2 = 72, 256
    pyr2 = torch.randn(B, c_pyr, Fq2, T2, generator=g).cuda()
    wo = (torch.randn(2, c_pyr, 1, 1, generator=g) * 0.5).cuda(); bo = torch.randn(2, generator=g).cuda()
    out = torch.full((B, 1, 257, T2), 7.0, dtype=torch.complex64, device="cuda")
    _check(lib, lib.fdbm_output_layer(nchw_to_ntfc(pyr2).data_ptr(), c_pyr, wo.reshape(2, c_pyr).contiguous().data_ptr(), bo.data_ptr(), B, T2, Fq2, 257,
                                      torch.view_as_real(out).data_ptr(), _stream()))
    o = F.conv2d(pyr2.double(), wo.double(), bo.double()).float()
    want = torch.view_as_complex(o.permute(0, 2, 3, 1).contiguous())[:, None]
    e2 = rel_l2(out[:, :, :256], want)
    print(f"combine rel L2 {e1:.2e}, output layer {e2:.2e}")
    assert e1 < 1e-6 and e2 < 1e-6 and not torch.view_as_real(out[:, :, 256]).any()
