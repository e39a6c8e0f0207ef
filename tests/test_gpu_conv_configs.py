"""Every convolution configuration the backbone plans launch (csrc/plan.cu), driven through fdbm_conv_igemm_ex with the
same descriptor a plan builds, against fp64 references.  Runs on the B200 only (`-m gpu`).

Two tiers:
- exact: dyadic inputs (activations k/2, weights k/16, biases / residuals / pyramids k/16, power-of-two GroupNorm scales
  with non-zero integer shifts), no SiLU.  Every product and partial sum is then representable in fp32, so the fp32
  output must EQUAL the fp64 reference and the 16-bit output its round-to-nearest.  Any indexing, tiling, halo, table,
  utterance or epilogue-routing error shows up bit for bit.
- realistic: Gaussian data, GroupNorm tables built by fdbm_gn_table from fp64 sums, SiLU, scale 1/sqrt(2), against torch
  fp64 group_norm -> SiLU -> conv2d; bounded in rel L2 and per output element.
Activations are [B,T,F,C] (kernel layout); the reference works in NCHW with H = F, W = T (weights OIHW).
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
SHAPES = {                     # B, T, F
    "aligned": (2, 32, 16),    # whole 16 x 8 tiles
    "ragged": (2, 20, 12),     # T, F not multiples of 16 / 8: partial tiles, zero halo inside the box
    "tiny": (2, 4, 4),         # the bottom level: an image smaller than one tile (one M-tile per utterance)
    "odd": (3, 48, 8),         # three M-tiles per utterance: the tile pairs of an item straddle utterances
}


@pytest.fixture(scope="module")
def lib():
    from fdbm_b200 import _lib
    lb = _lib.load()
    _lib.check(lb.fdbm_check_device(), "fdbm_check_device")
    return lb


def _op():
    from fdbm_b200 import _lib
    return _lib.operand_dtype()


def _unit():
    """unit round-off of the 16-bit operand format"""
    return 2.0 ** -8 if _op() == torch.bfloat16 else 2.0 ** -11


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check(lib, rc):
    assert rc == 0, lib.fdbm_last_error().decode()


def _ptr(t):
    return None if t is None else t.data_ptr()


def _nchw(x):
    return x.permute(0, 3, 2, 1)


def _ntfc(x):
    return x.permute(0, 3, 2, 1)


def _n_items(B, T, Fq, Cout, narrow=False):
    """the persistent grid's work items, as launch_conv_igemm counts them: pairs of 16 x 8 M-tiles x MMA-N blocks"""
    bn = 16 if narrow else (64 if Cout == 64 else 128)
    n_mtiles = B * math.ceil(T / 16) * math.ceil(Fq / 8)
    return math.ceil(n_mtiles / 2) * (Cout // bn)


# ------------------------------------------------------------------------------------------------
# configurations: what each plan.cu call site puts into ConvArgs
# ------------------------------------------------------------------------------------------------
# main   channels of the leading segments, all `taps` taps, normalised on load when `norm` (sharing one table over their
#        concatenation, as Conv_0's two inputs do); packed as w1
# side   channels of the raw 1-tap segments behind them (the fused Conv_2 shortcut), packed as the concatenated w2
def _spec(name, shape):
    s = dict(main=[], taps=9, norm=True, act=1, side=[], Cout=0, bias_b=False, film_uniform=False, residual=None,
             comb_C=0, pyr_C=0, pyr_prev=False, nin=False, sums=True, prezeroed=False, scale_exact=1.0, scale_real=1.0)
    if name == "conv0_film":                  # plan.cu:485-493 up-path Conv_0: two 9-tap GroupNorm + SiLU segments, FiLM
        s["main"], s["Cout"] = {"aligned": ([256, 256], 256), "ragged": ([256, 128], 256), "tiny": ([128, 128], 128),
                                "odd": ([256, 128], 256)}[shape]
        s["bias_b"] = True
    elif name == "conv0_uniform_t":           # plan.cu:406, 411: FiLM row 0 for every utterance, statistics added on
        s.update(main=[256, 128], Cout=256, bias_b=True, film_uniform=True, prezeroed=True)
    elif name in ("conv1_shortcut", "conv1_combine"):   # plan.cu:510-524 Conv_1: GroupNorm_1 + SiLU on load, raw Conv_2 operands
        cout, side = {"aligned": (256, [256, 256]), "ragged": (256, [256, 128]), "tiny": (256, [128]),
                      "odd": (128, [128, 128])}[shape]
        s.update(main=[cout], side=side, Cout=cout, scale_exact=0.5, scale_real=0.5 ** 0.5)
        if name == "conv1_combine":           # last block of a level: Combine in the epilogue
            s["comb_C"] = 4 if shape in ("aligned", "tiny") else 2
    elif name == "conv1_identity":            # plan.cu:521 Conv_1 with the 16-bit identity shortcut
        c = 256 if shape in ("aligned", "tiny") else 128
        s.update(main=[c], Cout=c, residual="h16", scale_exact=0.5, scale_real=0.5 ** 0.5)
    elif name == "attn_nin3":                 # plan.cu:644-649 attention output NIN_3 + 16-bit shortcut
        s.update(main=[256], taps=1, norm=False, Cout=256, residual="h16", scale_exact=0.5, scale_real=0.5 ** 0.5)
    elif name == "attn_qkv":                  # plan.cu:631-635 q/k/v: 1-tap GroupNorm without activation, Cout = 3C, no sums
        s.update(main=[256], taps=1, act=0, Cout=768, nin=True, sums=False)
    elif name == "pyramid":                   # plan.cu:873-877 C -> 4 / 2 with the FIR-upsampled coarser level
        s.update(main=[256 if shape in ("aligned", "odd") else 128], Cout=16, pyr_C=4 if shape in ("aligned", "tiny") else 2,
                 pyr_prev=True, sums=False)
    elif name == "pyramid_coarsest":          # the first pyramid level has no coarser one
        s.update(main=[256], Cout=16, pyr_C=4 if shape != "ragged" else 2, sums=False)
    elif name == "cout64":                    # ncsnpp_v2_16M: Cout = 64 layers (MMA N = 64)
        s.update(main=[64], Cout=64, bias_b=True, residual="f32", scale_exact=0.5, scale_real=0.5 ** 0.5)
    else:
        raise KeyError(name)
    return s


CONFIGS = ["conv0_film", "conv0_uniform_t", "conv1_shortcut", "conv1_combine", "conv1_identity", "attn_nin3", "attn_qkv",
           "pyramid", "pyramid_coarsest", "cout64"]
EXACT_CASES = [(c, sh) for c in CONFIGS for sh in SHAPES if not (c == "pyramid_coarsest" and sh in ("aligned", "odd"))]
REAL_CASES = [(c, sh) for c in CONFIGS for sh in ("ragged", "odd") if c != "pyramid_coarsest"]


def _dyadic(shape, lo, hi, den, g):
    return (torch.randint(lo, hi + 1, shape, generator=g, dtype=torch.int32).double() / den).to(DEV)


class _Case:
    """inputs, packed weights and the descriptor of one configuration; `ref` is computed in fp64"""

    def __init__(self, lib, s, B, T, Fq, exact, seed):
        self.lib, self.s, self.B, self.T, self.Fq, self.exact = lib, s, B, T, Fq, exact
        g = torch.Generator().manual_seed(seed)
        op = _op()
        cout = s["Cout"]
        n_out = s["pyr_C"] if s["pyr_C"] else cout          # real output channels (pyramid: pyr_C of the 16 MMA columns)

        def act_in(c):                                      # 16-bit activation [B,T,F,c], returned as fp64
            if exact:
                return _dyadic((B, T, Fq, c), -4, 4, 2, g)
            return (torch.randn(B, T, Fq, c, generator=g) * 1.5 + 0.3).to(op).double().to(DEV)

        def wts(*shape, fan):
            if exact:
                return _dyadic(shape, -8, 8, 16, g)
            return (torch.randn(*shape, generator=g) / fan ** 0.5).to(op).double().to(DEV)

        def small(*shape, real_scale=1.0):                  # biases, residuals, pyramids: k/16 in [-2, 2], or Gaussian
            if exact:
                return _dyadic(shape, -32, 32, 16, g)
            return (torch.randn(*shape, generator=g) * real_scale).double().to(DEV)

        self.x_main = [act_in(c) for c in s["main"]]
        self.x_side = [act_in(c) for c in s["side"]]
        cm, cs, k = sum(s["main"]), sum(s["side"]), 3 if s["taps"] == 9 else 1
        self.w_main = wts(n_out, cm, k, k, fan=cm * k * k + cs)
        self.w_side = wts(n_out, cs, fan=cm * k * k + cs) if cs else None
        self.bias = small(cout)
        self.bias_b = small(1 if s["film_uniform"] else B, cout) if s["bias_b"] else None
        self.residual = small(B, T, Fq, cout) if s["residual"] else None
        if s["residual"] == "h16":
            self.residual = self.residual.to(op).double()
        self.comb = None
        if s["comb_C"]:
            self.comb = (small(B, T, Fq, s["comb_C"]), small(cout, s["comb_C"], real_scale=0.3), small(cout))
        self.pyr_prev = small(B, T // 2, Fq // 2, s["pyr_C"]) if s["pyr_prev"] else None

        # GroupNorm (scale, shift) table over the concatenation of the normalised segments: [B, cm] pairs
        self.table = None
        if s["norm"]:
            if exact:
                # power-of-two scales per (utterance, channel) and non-zero integer shifts: x * scale + shift stays on a
                # 1/4 grid within +-16 (exact in fp16 and bf16), and a shift leaking into the zero padding is visible
                sc = 2.0 ** torch.randint(-1, 2, (B, cm), generator=g).double()
                sh = torch.randint(1, 4, (B, cm), generator=g).double() * (torch.randint(0, 2, (B, cm), generator=g) * 2 - 1)
                self.table = torch.stack([sc, sh], -1).to(DEV)
            else:
                self.gamma = (1 + 0.1 * torch.randn(cm, generator=g)).to(DEV)
                self.beta = (0.1 * torch.randn(cm, generator=g)).to(DEV)

        # device operands
        self.in_main = [x.to(op) for x in self.x_main]
        self.in_side = [x.to(op) for x in self.x_side]
        self.wpack = self._pack()
        self.dbias = self.bias.float()
        self.dbias_b = self.bias_b.float() if self.bias_b is not None else None
        self.dres = None
        if s["residual"] == "f32":
            self.dres = self.residual.float()
        elif s["residual"] == "h16":
            self.dres = self.residual.to(op)
        self.dcomb = tuple(t.float().contiguous() for t in self.comb) if self.comb else None
        self.dpyr_prev = self.pyr_prev.float() if self.pyr_prev is not None else None

    def _pack(self):
        s, lib = self.s, self.lib
        cm, cs, cout = sum(s["main"]), sum(s["side"]), s["Cout"]
        if s["nin"]:                                         # q/k/v: the fp32 [C][3C] NIN concatenation, ksize -1
            w1, ks = self.w_main[:, :, 0, 0].t().contiguous().float(), -1
        else:
            w1 = self.w_main.float()
            if s["pyr_C"]:                                   # pyramid: weight rows zero-padded to the MMA N of 16
                w1 = torch.cat([w1, torch.zeros(16 - s["pyr_C"], *w1.shape[1:], device=DEV)]).contiguous()
            ks = 3 if s["taps"] == 9 else 1
        w2 = self.w_side.float().contiguous() if cs else None
        nbytes = C.c_int64()
        _check(lib, lib.fdbm_pack_conv_weights(None, cm, ks, None, cs, cout, None, C.byref(nbytes), None))
        wpack = torch.empty(nbytes.value // 2, dtype=_op(), device=DEV)
        _check(lib, lib.fdbm_pack_conv_weights(w1.data_ptr(), cm, ks, _ptr(w2), cs, cout, wpack.data_ptr(), None, _stream()))
        return wpack

    def build_table(self):
        """realistic tier: the table through fdbm_gn_table from fp64 sums of the 16-bit inputs, two sources as plan.cu:488"""
        B = self.B
        sums = [torch.stack([x.sum((1, 2)), x.pow(2).sum((1, 2))], -1).contiguous() for x in self.x_main]
        self.dtable = torch.empty(B, sum(self.s["main"]), 2, device=DEV)
        _check(self.lib, self.lib.fdbm_gn_table(sums[0].data_ptr(), self.s["main"][0], _ptr(sums[1]) if len(sums) > 1 else None,
                                                self.s["main"][1] if len(sums) > 1 else 0, self.gamma.data_ptr(),
                                                self.beta.data_ptr(), 0, B, self.T * self.Fq, self.dtable.data_ptr(), None,
                                                _stream()))

    def desc(self, out_f32, out_h16, sums, pyr_out, scale):
        from fdbm_b200 import _lib
        s = self.s
        d = _lib.ConvDesc(wpack=self.wpack.data_ptr(), bias=self.dbias.data_ptr(), scale=scale, B=self.B, T=self.T, F=self.Fq,
                          Cout=s["Cout"], out_f32=_ptr(out_f32), out_h16=_ptr(out_h16), sums=_ptr(sums),
                          sums_prezeroed=int(s["prezeroed"]))
        n = 0
        c_off = 0
        cm = sum(s["main"])
        for x, c in zip(self.in_main, s["main"]):
            seg = _lib.ConvSeg(in_=x.data_ptr(), C=c, taps=s["taps"])
            if s["norm"]:                                    # tab + C1 for the second source, stride = all normalised channels
                seg.norm_tab, seg.tab_stride = self.dtable.data_ptr() + 8 * c_off, cm
                seg.act = 0 if self.exact else s["act"]     # the exact tier has no SiLU
            d.seg[n] = seg
            n += 1
            c_off += c
        for x, c in zip(self.in_side, s["side"]):
            d.seg[n] = _lib.ConvSeg(in_=x.data_ptr(), C=c, taps=1)
            n += 1
        d.n_seg = n
        if self.dbias_b is not None:
            d.bias_b, d.bias_b_stride = self.dbias_b.data_ptr(), 0 if s["film_uniform"] else s["Cout"]
        if s["residual"] == "f32":
            d.residual = self.dres.data_ptr()
        elif s["residual"] == "h16":
            d.residual_h16 = self.dres.data_ptr()
        if self.dcomb:
            d.comb_pyr, d.comb_w, d.comb_b, d.comb_C = self.dcomb[0].data_ptr(), self.dcomb[1].data_ptr(), self.dcomb[2].data_ptr(), s["comb_C"]
        if s["pyr_C"]:
            d.narrow_n, d.pyr_out, d.pyr_C, d.pyr_prev = 1, pyr_out.data_ptr(), s["pyr_C"], _ptr(self.dpyr_prev)
        return d

    def ref(self, scale):
        """fp64: transform on load -> conv -> epilogue; [B,T,F,n_out] (pyramid: [B,T,F,pyr_C])"""
        s = self.s
        xm = torch.cat(self.x_main, -1)
        if s["norm"]:
            if self.exact:
                xm = xm * self.table[:, None, None, :, 0] + self.table[:, None, None, :, 1]
            else:
                cm = xm.shape[-1]
                xm = _ntfc(F.group_norm(_nchw(xm), min(cm // 4, 32), self.gamma.double(), self.beta.double(), eps=1e-6))
            if s["act"] and not self.exact:
                xm = F.silu(xm)
        k = self.w_main.shape[-1]
        acc = F.conv2d(_nchw(xm), self.w_main, padding=k // 2)
        if self.w_side is not None:
            acc = acc + F.conv2d(_nchw(torch.cat(self.x_side, -1)), self.w_side[:, :, None, None])
        out = _ntfc(acc)
        n_out = out.shape[-1]
        if s["pyr_C"]:
            out = out + self.bias[:n_out]
            if self.pyr_prev is not None:
                import fdbm_oracle as O
                out = out + _ntfc(O.fir_up2(_nchw(self.pyr_prev)))
            return out.contiguous()
        out = out + self.bias
        if self.bias_b is not None:
            out = out + (self.bias_b[:1] if s["film_uniform"] else self.bias_b)[:, None, None, :]
        if self.residual is not None:
            out = out + self.residual
        out = out * scale
        if self.comb:
            pyr, w, b = self.comb
            out = out + b + torch.einsum("btfk,nk->btfn", pyr, w)
        return out.contiguous()

    def run(self, scale, table=None):
        """one launch; returns (fp32 result, 16-bit result, sums, the sums buffer's initial content)"""
        s, B, T, Fq = self.s, self.B, self.T, self.Fq
        if table is not None:
            self.dtable = table
        out = out16 = sums = pyr = None
        sums0 = None
        if s["pyr_C"]:
            pyr = torch.full((B, T, Fq, s["pyr_C"]), float("nan"), device=DEV)
        else:
            out = torch.full((B, T, Fq, s["Cout"]), float("nan"), device=DEV)
            out16 = torch.full((B, T, Fq, s["Cout"]), float("nan"), dtype=_op(), device=DEV)
        if s["sums"]:
            if s["prezeroed"]:                               # statistics are added onto what the buffer holds
                sums0 = _dyadic((B, s["Cout"], 2), -64, 64, 4, torch.Generator().manual_seed(5))
                sums = sums0.clone()
            else:
                sums = torch.full((B, s["Cout"], 2), float("nan"), dtype=torch.float64, device=DEV)
        d = self.desc(out, out16, sums, pyr, scale)
        _check(self.lib, self.lib.fdbm_conv_igemm_ex(C.byref(d), _stream()))
        torch.cuda.synchronize()
        return (pyr if s["pyr_C"] else out), out16, sums, sums0


def _where(diff_mask):
    idx = diff_mask.nonzero()
    return f"{idx.shape[0]} mismatching elements, first (b, t, f, c) = {idx[:4].tolist()}"


def _assert_sums(sums, sums0, ref, rtol=1e-6):
    want = torch.stack([ref.sum((1, 2)), ref.pow(2).sum((1, 2))], -1)
    if sums0 is not None:
        want = want + sums0
    for j, what in ((0, "sum"), (1, "sum of squares")):
        err = (sums[..., j] - want[..., j]).abs()
        tol = rtol * float(want[..., j].abs().max())
        bad = err > tol
        assert not bad.any(), f"channel {what}: {bad.sum().item()} of {bad.numel()} (b, c) off, first {bad.nonzero()[:4].tolist()}, max err {float(err.max()):.3g} (tol {tol:.3g})"


def _exact_check(case, scale):
    ref = case.ref(scale)
    # headroom: every partial sum below 2^12 on a grid >= 2^-8 needs at most 20 of fp32's 24 significand bits
    assert float(ref.abs().max()) < 2 ** 12
    got, got16, sums, sums0 = case.run(scale, table=case.table.float().contiguous() if case.table is not None else None)
    want = ref.float()
    assert torch.equal(got, want), "fp32 output differs from the exact fp64 reference: " + _where(got != want)
    if got16 is not None:
        want16 = want.to(_op())
        assert torch.equal(got16, want16), "16-bit output differs from the rounded reference: " + _where(got16 != want16)
    if sums is not None:
        _assert_sums(sums, sums0, ref)


@pytest.mark.parametrize("config,shape", EXACT_CASES)
def test_conv_config_exact(lib, config, shape):
    s = _spec(config, shape)
    B, T, Fq = SHAPES[shape]
    case = _Case(lib, s, B, T, Fq, exact=True, seed=EXACT_CASES.index((config, shape)))
    _exact_check(case, s["scale_exact"])


# per-element bound of the realistic tier, in units of the operand format's unit round-off u (2^-11 fp16, 2^-8 bf16).
# Each normalised operand element carries up to ~3 roundings of size u * |y| (the 16-bit rounding of y / 2, the packed
# tanh.approx, the 16-bit h + h * tanh(h)); the output error is their sum weighted by the ~1/sqrt(K) weights, so its
# standard deviation is ~u * ref.std() (the rel L2 bound below), and over <= 10^6 outputs the largest is ~5 sigma.
# 32 u leaves a factor ~6 for the tails; one border pixel that reads a wrong table row or a shifted halo is off by
# ~0.1 ref.std(), > 6x the bound in fp16.
PER_ELEMENT_U = 32
REL_L2 = 1e-3


def _real_check(case, scale):
    if case.s["norm"]:
        case.build_table()
    ref = case.ref(scale)
    got, got16, sums, sums0 = case.run(scale)
    assert torch.isfinite(got).all()
    u = _unit()
    rel_bound = REL_L2 * u / 2.0 ** -11
    err = float((got.double() - ref).pow(2).sum().sqrt() / ref.pow(2).sum().sqrt())
    assert err < rel_bound, f"rel L2 {err:.3g} >= {rel_bound:.3g}"
    dev = (got.double() - ref).abs() / ref.std()
    worst = float(dev.max())
    assert worst < PER_ELEMENT_U * u, f"max |got - ref| / ref.std() = {worst:.3g} at (b, t, f, c) {(dev == dev.max()).nonzero()[0].tolist()}"
    if sums is not None:
        _assert_sums(sums, sums0, ref, rtol=2e-3)


@pytest.mark.parametrize("config,shape", REAL_CASES)
def test_conv_config_realistic(lib, config, shape):
    s = _spec(config, shape)
    B, T, Fq = SHAPES[shape]
    case = _Case(lib, s, B, T, Fq, exact=False, seed=1000 + REAL_CASES.index((config, shape)))
    _real_check(case, s["scale_real"])


# ------------------------------------------------------------------------------------------------
# persistent CTAs: more than one item per CTA (second TMEM accumulator stage, ring phases across items, statistics flushed
# when a CTA's next item belongs to another utterance, the next tile's residual prefetch), once per kernel instantiation
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("config", ["conv0_film", "conv1_identity", "conv1_combine"])    # plain, RES16, COMB kernels
def test_conv_persistent_exact(lib, config):
    s = _spec(config, "aligned")
    if config == "conv1_combine":
        s.update(main=[256], side=[256, 128], Cout=256)
    B, T, Fq = 5, 128, 64
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    n_items = _n_items(B, T, Fq, s["Cout"])
    assert n_items >= 2 * n_sms, f"{n_items} items on {n_sms} SMs: not a multi-item launch"
    case = _Case(lib, s, B, T, Fq, exact=True, seed=77 + len(config))
    _exact_check(case, s["scale_exact"])


# ------------------------------------------------------------------------------------------------
# GroupNorm tables
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C1,C2,blk_real", [(256, 128, 0), (128, 128, 0), (256, 0, 96), (256, 128, 96)])
def test_gn_table(lib, C1, C2, blk_real):
    """fdbm_gn_table against fp64: groups straddling the concatenation boundary (256 + 128: 12 channels per group) and the
    nf96 layout (every 128-channel block = 96 real channels + 32 padding, groups over the real channels only)."""
    g = torch.Generator().manual_seed(C1 + C2 + blk_real)
    B, px = 3, 37 * 11
    Ct = C1 + C2
    x_mean = torch.randn(B, Ct, generator=g, dtype=torch.float64) * 0.7 + 0.2
    x_sq = x_mean ** 2 + torch.rand(B, Ct, generator=g, dtype=torch.float64) * 2 + 0.1
    sums = torch.stack([x_mean * px, x_sq * px], -1)        # (sum, sum of squares); padded channels keep non-zero garbage
    gamma = 1 + 0.1 * torch.randn(Ct, generator=g)
    beta = 0.1 * torch.randn(Ct, generator=g)
    real = torch.arange(Ct)
    if blk_real:
        real = real[(real % 128) < blk_real]
    Cr = real.numel()
    G = min(Cr // 4, 32)
    grp_s = sums[:, real, 0].reshape(B, G, -1).sum(-1)
    grp_q = sums[:, real, 1].reshape(B, G, -1).sum(-1)
    cnt = Cr // G * px
    mean = grp_s / cnt
    rstd = 1.0 / torch.sqrt((grp_q / cnt - mean ** 2).clamp_min(0) + 1e-6)
    a = torch.zeros(B, Ct, dtype=torch.float64)
    b = torch.zeros(B, Ct, dtype=torch.float64)
    gi = torch.arange(Cr) // (Cr // G)
    a[:, real] = gamma.double()[real] * rstd[:, gi]
    b[:, real] = beta.double()[real] - mean[:, gi] * a[:, real]
    s1 = sums[:, :C1].contiguous().to(DEV)
    s2 = sums[:, C1:].contiguous().to(DEV) if C2 else None
    table = torch.full((B, Ct, 2), float("nan"), device=DEV)
    stats = torch.full((B, G, 2), float("nan"), device=DEV)
    gd, bd = gamma.to(DEV), beta.to(DEV)
    _check(lib, lib.fdbm_gn_table(s1.data_ptr(), C1, _ptr(s2), C2, gd.data_ptr(), bd.data_ptr(), blk_real, B, px, table.data_ptr(),
                                  stats.data_ptr(), _stream()))
    torch.cuda.synchronize()
    table, stats = table.cpu().double(), stats.cpu().double()
    if blk_real:
        pad = (torch.arange(Ct) % 128) >= blk_real
        assert torch.equal(table[:, pad], torch.zeros_like(table[:, pad])), "padded channels must get exactly (0, 0)"
    # fp32 outputs of fp64 arithmetic: scale to 2 roundings, shift = beta - mean * scale to the rounding of its larger term
    assert ((table[..., 0] - a).abs() <= 3e-7 * a.abs()).all()
    assert ((table[..., 1] - b).abs() <= 3e-7 * (beta.double().abs() + (b - beta.double()).abs()) + 1e-12).all()
    assert ((stats[..., 0] - mean).abs() <= 1e-7 * mean.abs() + 1e-12).all()
    assert ((stats[..., 1] - rstd).abs() <= 1e-7 * rstd).all()


# ------------------------------------------------------------------------------------------------
# conv -> GroupNorm table -> normalise-on-load conv on one stream without host synchronisation: the plans rely on this
# order, with programmatic dependent launch at small batches (B <= 8) and plain stream order above
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [2, 9])
def test_dependent_launch_chain(lib, B):
    from fdbm_b200 import _lib
    g = torch.Generator().manual_seed(B)
    T, Fq, Cc = 32, 16, 128
    op = _op()
    x = _dyadic((B, T, Fq, Cc), -4, 4, 2, g)
    w1 = _dyadic((Cc, Cc, 3, 3), -8, 8, 16, g)
    b1 = _dyadic((Cc,), -32, 32, 16, g)
    w2 = (torch.randn(Cc, Cc, 3, 3, generator=g) / (9 * Cc) ** 0.5).to(op).double().to(DEV)
    b2 = torch.randn(Cc, generator=g).double().to(DEV)
    gamma = (1 + 0.1 * torch.randn(Cc, generator=g)).to(DEV)
    beta = (0.1 * torch.randn(Cc, generator=g)).to(DEV)
    packs = []
    for w in (w1, w2):
        nb = C.c_int64()
        _check(lib, lib.fdbm_pack_conv_weights(None, Cc, 3, None, 0, Cc, None, C.byref(nb), None))
        wp = torch.empty(nb.value // 2, dtype=op, device=DEV)
        wf = w.float().contiguous()
        _check(lib, lib.fdbm_pack_conv_weights(wf.data_ptr(), Cc, 3, None, 0, Cc, wp.data_ptr(), None, _stream()))
        packs.append(wp)
    xin = x.to(op)
    b1d, b2d = b1.float(), b2.float()
    h = torch.full((B, T, Fq, Cc), float("nan"), dtype=op, device=DEV)
    sums = torch.full((B, Cc, 2), float("nan"), dtype=torch.float64, device=DEV)
    table = torch.full((B, Cc, 2), float("nan"), device=DEV)
    out = torch.full((B, T, Fq, Cc), float("nan"), device=DEV)
    torch.cuda.synchronize()
    d1 = _lib.ConvDesc(n_seg=1, wpack=packs[0].data_ptr(), bias=b1d.data_ptr(), B=B, T=T, F=Fq, Cout=Cc, out_h16=h.data_ptr(),
                       sums=sums.data_ptr())
    d1.seg[0] = _lib.ConvSeg(in_=xin.data_ptr(), C=Cc, taps=9)
    d2 = _lib.ConvDesc(n_seg=1, wpack=packs[1].data_ptr(), bias=b2d.data_ptr(), B=B, T=T, F=Fq, Cout=Cc, out_f32=out.data_ptr())
    d2.seg[0] = _lib.ConvSeg(in_=h.data_ptr(), C=Cc, taps=9, norm_tab=table.data_ptr(), tab_stride=Cc, act=1)
    _check(lib, lib.fdbm_conv_igemm_ex(C.byref(d1), _stream()))
    _check(lib, lib.fdbm_gn_table(sums.data_ptr(), Cc, None, 0, gamma.data_ptr(), beta.data_ptr(), 0, B, T * Fq, table.data_ptr(),
                                  None, _stream()))
    _check(lib, lib.fdbm_conv_igemm_ex(C.byref(d2), _stream()))
    torch.cuda.synchronize()
    # reference chain: the first convolution is exact; GroupNorm statistics from its fp32 values, applied to its 16-bit copy
    r1 = _ntfc(F.conv2d(_nchw(x), w1, padding=1)) + b1
    assert torch.equal(h, r1.float().to(op))
    G = 32
    grp = r1.reshape(B, T * Fq, G, Cc // G)
    mean = grp.mean((1, 3))
    var = grp.pow(2).mean((1, 3)) - mean ** 2
    rstd = 1.0 / torch.sqrt(var + 1e-6)
    sc = gamma.double() * rstd.repeat_interleave(Cc // G, 1)
    sh = beta.double() - mean.repeat_interleave(Cc // G, 1) * sc
    a = F.silu(h.double() * sc[:, None, None, :] + sh[:, None, None, :])
    ref = _ntfc(F.conv2d(_nchw(a), w2, padding=1)) + b2
    u = _unit()
    err = float((out.double() - ref).pow(2).sum().sqrt() / ref.pow(2).sum().sqrt())
    assert err < REL_L2 * u / 2.0 ** -11, f"rel L2 {err:.3g}"
    assert float(((out.double() - ref).abs() / ref.std()).max()) < PER_ELEMENT_U * u


# ------------------------------------------------------------------------------------------------
# host-side refusals of launch_conv_igemm (checked before any launch)
# ------------------------------------------------------------------------------------------------
def _refusal_desc(**over):
    from fdbm_b200 import _lib
    B, T, Fq = over.pop("B", 1), over.pop("T", 16), over.pop("F", 8)
    keep = []

    def t(*shape, dtype=torch.float32):
        x = torch.zeros(*shape, dtype=dtype, device=DEV)
        keep.append(x)
        return x.data_ptr()

    segs = over.pop("segs", [(128, 9)])
    cout = over.pop("Cout", 128)
    d = _lib.ConvDesc(n_seg=len(segs), wpack=t(1 << 20, dtype=_op()), bias=t(256), B=B, T=T, F=Fq, Cout=cout,
                      out_f32=t(B, T, Fq, max(cout, 16)))
    for i, (c, taps) in enumerate(segs):
        d.seg[i] = _lib.ConvSeg(in_=t(B, T, Fq, c, dtype=_op()), C=c, taps=taps)
    for k, v in over.items():
        setattr(d, k, t(*v[1], dtype=v[2]) if isinstance(v, tuple) and v[0] == "tensor" else v)
    return d, keep


@pytest.mark.parametrize("what,over,message", [
    ("17 K-blocks", dict(segs=[(512, 9), (512, 1), (64, 1)]), "at most 16 K-blocks"),
    ("Cout not a multiple of the MMA N", dict(Cout=192), "Cout must be a multiple of 128"),
    ("pyramid level with odd T", dict(T=15, Cout=16, narrow_n=1, out_f32=None, pyr_C=4, pyr_out=("tensor", (1, 15, 8, 4), torch.float32),
                                      pyr_prev=("tensor", (1, 7, 4, 4), torch.float32)), "pyramid level with odd size"),
    ("fp32 and 16-bit residual", dict(residual=("tensor", (1, 16, 8, 128), torch.float32),
                                      residual_h16=("tensor", (1, 16, 8, 128), torch.float16)), "bad residual arguments"),
])
def test_conv_refusals(lib, what, over, message):
    d, keep = _refusal_desc(**over)
    rc = lib.fdbm_conv_igemm_ex(C.byref(d), _stream())
    msg = lib.fdbm_last_error().decode()
    assert rc != 0 and message in msg, (what, rc, msg)
    torch.cuda.synchronize()
