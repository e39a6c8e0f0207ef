"""The Python seams of the drop-in boundary, checked against what the REFERENCE's own objects give (CPU, no CUDA call).

tests/golden/dropin.npz holds those values (oracle/make_golden.py `dropin`, seeded inputs): argparse defaults, state_dict layout,
requires_grad flags and init statistics of the backbones, Bridge attributes and path maths, pc / ode_int sampler outputs of a
stand-in model, SpecsDataModule attributes.  With FDBM_REFERENCE naming a checkout of the original project,
test_golden_matches_the_reference also recomputes them from its classes and checks registry / state_dict interchange live.
SURVEY.md section 8(b): (1) BackboneRegistry.register / get_by_name + add_argparse_args + **kwargs tolerance,
(2) Bridge attributes and path maths, (3) SpecsDataModule attributes, state_dict compatibility in both directions."""
import json
import os

import numpy as np
import pytest
import torch

import make_golden as MG
from helpers import load_npz

REF = os.environ.get("FDBM_REFERENCE")


@pytest.fixture(scope="module")
def golden(golden_dir):
    g = load_npz(os.path.join(golden_dir, "dropin.npz"))
    return json.loads(str(g.pop("meta"))), g


def as_json(x):
    return json.loads(json.dumps(x))


def test_our_backbones_register_into_the_reference_registry(golden):
    """`BackboneRegistry.register(name)(cls)` + `get_by_name(name)(**kwargs)` (util/registry.py:17-30, model.py:47-48) with the
    kwargs soup train.py passes (every argparse group's values at once), and the reference's flags, state_dict layout,
    parameter flags and initialisation law."""
    import fdbm_b200
    meta, _ = golden
    R = fdbm_b200.BackboneRegistry
    R.register("ncsnpp_v2_b200")(fdbm_b200.NCSNpp_v2)
    R.register("ncsnpp_v2_predictive_b200")(fdbm_b200.NCSNpp_v2_predictive)
    cls = R.get_by_name("ncsnpp_v2_b200")
    assert cls is fdbm_b200.NCSNpp_v2
    # argparse seam (train.py:92-93): same flags, same defaults
    assert as_json(MG.argparse_defaults(cls)) == meta["ncsnpp_v2_args"]
    # constructor tolerates the reference's full kwargs dictionary (model.py:47-48 passes **kwargs of ALL groups)
    ours = cls(**MG.dropin_soup(meta["ncsnpp_v2_args"]))
    # state_dict compatibility in both directions, strict
    assert {k: list(v.shape) for k, v in ours.state_dict().items()} == meta["ncsnpp_v2_shapes"]
    ours.load_state_dict({k: torch.zeros(s) for k, s in meta["ncsnpp_v2_shapes"].items()}, strict=True)
    # requires_grad flags agree (the Fourier projection is frozen, layerspp.py:37): torch_ema / Adam see the same parameter list
    assert [[n, p.requires_grad] for n, p in ours.named_parameters()] == meta["ncsnpp_v2_requires_grad"]
    # same initialisation law: per-tensor standard deviations of a fresh model agree statistically
    torch.manual_seed(0)
    params = dict(cls().named_parameters())
    stds = meta["ncsnpp_v2_init_std"]
    assert set(stds) == {n for n, p in params.items() if p.numel() > 4096}
    for n, s in stds.items():
        assert abs(float(params[n].detach().std()) - s) < 0.08 * s + 1e-9, n
    # unsupported architecture variants are refused loudly, not silently ignored
    for bad in (dict(dropout=0.1), dict(fir_kernel=[1, 2, 1]), dict(resamp_with_conv=False), dict(progressive="none")):
        with pytest.raises(NotImplementedError):
            cls(**bad)
    pred = R.get_by_name("ncsnpp_v2_predictive_b200")()
    assert {k: list(v.shape) for k, v in pred.state_dict().items()} == meta["ncsnpp_v2_predictive_shapes"]
    pred.load_state_dict({k: torch.zeros(s) for k, s in meta["ncsnpp_v2_predictive_shapes"].items()}, strict=True)


def test_forward_without_cuda_fails_loudly():
    import fdbm_b200
    net = fdbm_b200.NCSNpp_v2()
    x = torch.zeros(1, 1, 257, 64, dtype=torch.complex64)
    with pytest.raises(RuntimeError):
        net(x, x, torch.ones(1))                     # CPU tensors: no fallback


@pytest.mark.parametrize("path,kw", [("sb", dict(noise_schedule="bb")), ("sb", dict(noise_schedule="ve")),
                                     ("sb", dict(noise_schedule="vp", c=0.3)), ("sb", dict(noise_schedule="gmax")), ("fm", dict())])
def test_bridge_host_maths_equal_the_reference(golden, path, kw):
    """Attributes callers read / mutate (infer_single.py:55-56, model.py:451-452) and every scalar function of the paths."""
    import fdbm_b200
    meta, g = golden
    tag = f"{path}_{kw.get('noise_schedule', 'ot')}"
    assert MG.DROPIN_PATHS[tag] == (path, kw)
    m = meta[tag]
    ob = fdbm_b200.Bridge(path, N=7, sampler_type="sde_ei", sampling_eps=1e-3, **kw)
    for attr, want in m["attrs"].items():
        assert as_json(getattr(ob, attr)) == want, attr
    assert ob.path.sampling_direction == m["sampling_direction"] and ob.path.T == m["path_T"]
    ob.N, ob.sampler_type = 3, "ode_ei"                                           # mutable after construction
    assert ob.time_grid().numel() == 4

    def check(name, values, exact=True, rtol=1e-6, atol=1e-7):
        assert f"{tag}_{name}_{len(values)}" not in g, name
        for i, v in enumerate(values):
            got, want = torch.as_tensor(v).numpy(), g[f"{tag}_{name}_{i}"]
            if exact:
                assert got.dtype == want.dtype and np.array_equal(got, want), (name, i)
            else:
                assert got.shape == want.shape and np.allclose(got, want, rtol=rtol, atol=atol), (name, i)

    t = torch.tensor(MG.DROPIN_T)
    s, y, x = MG.dropin_bridge_inputs()
    check("path_param", ob.path.path_param(t))
    check("std", [ob._std(t)])
    check("probability_path", ob.probability_path(s, y, t))
    check("score_fn", [ob.score_fn(t, x, s, y)])
    # ode / sde: the reference's [B]-into-[B,1,F,T] product is only meaningful for B = 1 (its callers); equal there
    t1 = torch.tensor([0.4])
    x1, s1, y1 = x[:1], s[:1], y[:1]
    check("ode", [ob.path.ode(t1, x1, s1, y1)], exact=False)
    if path == "sb":
        check("sde", ob.path.sde(t1, x1, s1, y1), exact=False, atol=1e-8)
        check("auxiliary_param", [torch.as_tensor(v, dtype=torch.float32) for v in ob.path.auxiliary_param(t1)], exact=False,
              rtol=1e-5, atol=1e-8)
        check("sampling_param_ode_ei", ob.path.sampling_param_ode_ei(t1 * 0.5, t1, 1, "cpu"))
        check("sampling_param_sde_ei", ob.path.sampling_param_sde_ei(t1 * 0.5, t1, 1, "cpu"))
    # argparse seam of Bridge and of the path classes
    assert as_json(MG.argparse_defaults(fdbm_b200.Bridge)) == meta["bridge_args"]
    assert as_json(MG.argparse_defaults(type(ob.path))) == m["path_args"]


def test_oracle_pc_and_ode_int_samplers_equal_the_reference(golden):
    """The oracle's restatement of pc_sampler / ode_sampler_int (the GPU tests' yardstick) against the reference's own
    Bridge, with a cheap stand-in model (B = 1, as the reference's broadcasting requires)."""
    import fdbm_oracle as O
    _, g = golden
    y, zs, model = MG.dropin_sampler_inputs()
    for corrector, steps, predictor in MG.DROPIN_PC:
        got = O.Bridge("sb", N=4, sampler_type="pc").pc_sampler(model, y, predictor_name=predictor, corrector_name=corrector,
                                                                 snr=0.3, corrector_steps=steps, z0=zs[0], zs=zs[1:])
        assert torch.allclose(got, torch.from_numpy(g[f"pc_{corrector}_{predictor}"]), rtol=1e-5, atol=1e-6), (corrector, predictor)
    got = O.Bridge("fm", sampler_type="ode_int").ode_sampler_int(model, y, rtol=1e-6, atol=1e-6, z0=zs[0])
    assert torch.allclose(got, torch.from_numpy(g["ode_int_fm"]), rtol=1e-5, atol=1e-6)


def test_data_module_attributes_and_pad_spec(golden):
    import fdbm_b200
    meta, g = golden
    od = fdbm_b200.SpecsDataModule(base_dir="/unused", n_fft=512, hop_length=256, num_frames=256, window="sqrthann", gpu=False)
    for attr, want in meta["data_module"].items():
        assert as_json(getattr(od, attr)) == want, attr
    assert od.window.numpy().dtype == g["data_module_window"].dtype and np.array_equal(od.window.numpy(), g["data_module_window"])
    assert sorted(od.stft_kwargs) == meta["data_module_stft_kwargs"]
    with pytest.raises(NotImplementedError):
        fdbm_b200.pad_spec(torch.zeros(1, 1, 257, 10, dtype=torch.complex64), mode="bogus")


def test_golden_matches_the_reference(golden):
    """tests/golden/dropin.npz recomputed from the original project's classes, and our backbones registered into ITS registry with
    state_dicts interchanged both ways.  Needs a checkout of the original project (FDBM_REFERENCE)."""
    if not REF or not os.path.isdir(os.path.join(REF, "fdbm")):
        pytest.skip("needs a checkout of the original project: set FDBM_REFERENCE")
    import fdbm_b200
    Bridge, R, SpecsDataModule = MG.import_reference()[:3]
    meta, g = golden
    rec = MG.dropin_record(Bridge, R, SpecsDataModule)
    rmeta = json.loads(str(rec.pop("meta")))
    ref_std, want_std = rmeta.pop("ncsnpp_v2_init_std"), meta["ncsnpp_v2_init_std"]
    assert set(ref_std) == set(want_std) and all(abs(ref_std[n] - s) < 0.08 * s + 1e-9 for n, s in want_std.items())
    assert rmeta == {k: v for k, v in meta.items() if k != "ncsnpp_v2_init_std"}
    assert set(rec) == set(g)
    for k, v in rec.items():
        assert v.shape == g[k].shape and np.allclose(v, g[k], rtol=1e-5, atol=1e-6), k
    R.register("ncsnpp_v2_b200")(fdbm_b200.NCSNpp_v2)
    ours, theirs = R.get_by_name("ncsnpp_v2_b200")(), R.get_by_name("ncsnpp_v2")()
    ours.load_state_dict(theirs.state_dict(), strict=True)
    theirs.load_state_dict(ours.state_dict(), strict=True)
    y, _, model = MG.dropin_sampler_inputs()
    with pytest.raises(ValueError):
        Bridge("sb", N=4, sampler_type="pc").sampler(model, y)                 # 'reverse_diffusion' is not registered
