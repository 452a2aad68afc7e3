"""Needs a checkout of the unmodified reference in $TRANSFERATTACK_REFERENCE (skipped without one): the LIVE reference as the judge of
  (1) oracle/torch_ref.py — the eager restatement must reproduce the reference's perturbation bit for bit, and
  (2) the drop-in boundary — the reference's OWN plugin files, loaded on top of this package's Attack/utils through
      transferattack_b200.compat (kernels replaced by the oracle stand-in, so no GPU is needed), must produce exactly what
      they produce on the reference's own base class (SURVEY.md Appendix B.2 regression matrix)."""
import random

import numpy as np
import pytest
import torch

from conftest import bits_equal, n_diff_bits
from helpers import REF_ROOT, TinyNet, import_reference, make_attack, seed_all

pytestmark = pytest.mark.reference


def _net(seed=0, classes=1000):
    torch.manual_seed(seed)
    return TinyNet(classes).eval()


def _data(B=2, S=224):
    g = torch.Generator().manual_seed(1)
    return torch.rand(B, 3, S, S, generator=g), torch.randint(0, 1000, (B,), generator=g)


@pytest.fixture(scope="module")
def ref():
    return import_reference()


@pytest.fixture(scope="module")
def adopted():
    import transferattack_b200.compat as compat
    return compat.adopt_reference_plugins(REF_ROOT, package_name="transferattack_adopted")


@pytest.fixture(autouse=True)
def oracle_backend():
    from transferattack_b200 import ops
    from oracle_backend import OracleBackend
    ops._install_backend_for_tests(OracleBackend())
    yield
    ops._install_backend_for_tests(None)


TORCH_REF_CASES = {
    "fgsm": {}, "ifgsm": {}, "mifgsm": {}, "nifgsm": {}, "dim": {}, "tim": {}, "sim": {"epoch": 3}, "admix": {"epoch": 2},
    "vmifgsm": {"num_neighbor": 3, "epoch": 3}, "vnifgsm": {"num_neighbor": 2, "epoch": 3}, "emifgsm": {"epoch": 3},
}


@pytest.mark.parametrize("name", sorted(TORCH_REF_CASES))
def test_torch_ref_equals_live_reference(ref, name):
    from oracle import torch_ref
    kw = TORCH_REF_CASES[name]
    x, y = _data()
    net = _net()
    seed_all(3)
    d_ref = make_attack(ref, name, net, **kw)(x, y)
    seed_all(3)
    d = torch_ref.REF_ZOO[name](torch_ref.ref_wrap_model(net), **kw)(x, y)
    assert bits_equal(d.numpy(), d_ref.numpy()), n_diff_bits(d.numpy(), d_ref.numpy())


def test_torch_ref_pifgsm_equals_live_reference(ref, monkeypatch):
    """gradient/pifgsm.py hard-codes .cuda() (pifgsm.py:52); with Tensor.cuda shimmed to the identity the UNMODIFIED file runs
    on this GPU-less box and pins the device-agnostic restatement bit for bit (two configurations)."""
    from oracle import torch_ref
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    x, y = _data()
    for kw in ({"epoch": 4}, {"epoch": 3, "decay": 1.0, "kern_size": 5}):
        net = _net()
        d_ref = make_attack(ref, "pifgsm", net, **kw)(x, y)
        d = torch_ref.RefPIFGSM(torch_ref.ref_wrap_model(net), **kw)(x, y)
        assert bits_equal(d.numpy(), d_ref.numpy()), (kw, n_diff_bits(d.numpy(), d_ref.numpy()))


def test_torch_ref_ssm_and_the_matrix_form_equal_live_reference(ref, monkeypatch):
    """SURVEY §8 f4: input_transformation/ssm.py hard-codes .cuda(); with the shim the UNMODIFIED file pins (a) the device-agnostic
    restatement RefSSM bit for bit and (b) the float64 MATRIX form of its transform (oracle.spectrum_transform — what the
    tcgen05 kernel is tested against) to 2e-6."""
    import oracle
    from oracle import torch_ref
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.nn.Module, "cuda", lambda self, *a, **k: self)
    x, y = _data()
    kw = {"num_spectrum": 2, "epoch": 2}
    net = _net()
    seed_all(3); d_ref = make_attack(ref, "ssm", net, **kw)(x, y)
    seed_all(3); d = torch_ref.RefSSM(torch_ref.ref_wrap_model(net), **kw)(x, y)
    assert bits_equal(d.numpy(), d_ref.numpy()), n_diff_bits(d.numpy(), d_ref.numpy())
    live = make_attack(ref, "ssm", net, **kw)
    g = torch.Generator().manual_seed(9)
    img = torch.rand(2, 3, 224, 224, generator=g); mask = torch.rand(2, 3, 224, 224, generator=g) + 0.5
    fft = live.idct_2d(live.dct_2d(img) * mask).numpy()
    assert np.abs(fft - oracle.spectrum_transform(img.numpy(), None, mask.numpy())).max() <= 2e-6
    # the native plugin on this box (transform = the float64 matrix form through the stand-in backend): same draws, same loop
    import transferattack_b200 as tab
    seed_all(3); d_new = make_attack(tab, "ssm", net, **kw)(x, y)
    assert float((d_new == d_ref).float().mean()) >= 0.9


def test_torch_ref_gra_and_adaea_equal_live_reference(ref):
    """SURVEY §8 f4: the restatements of gradient/gra.py and ensemble/adaea.py that the native plugins are tested against"""
    from oracle import torch_ref
    x, y = _data()
    kw = {"num_neighbor": 3, "epoch": 3}
    seed_all(3); d_ref = make_attack(ref, "gra", _net(), **kw)(x, y)
    seed_all(3); d = torch_ref.RefGRA(torch_ref.ref_wrap_model(_net()), **kw)(x, y)
    assert bits_equal(d.numpy(), d_ref.numpy()), n_diff_bits(d.numpy(), d_ref.numpy())
    nets = [_net(0), _net(3), _net(5), _net(7)]
    seed_all(5); d_ref = make_attack(ref, "adaea", nets, epoch=2)(x, y)
    seed_all(5); d = torch_ref.RefAdaEA(torch_ref.RefEnsemble([torch_ref.ref_wrap_model(n) for n in nets]), epoch=2)(x, y)
    assert bits_equal(d.numpy(), d_ref.numpy()), n_diff_bits(d.numpy(), d_ref.numpy())
    # and the native plugins (kernels replaced by the C oracle on this box) against the live reference itself
    import transferattack_b200 as tab
    seed_all(3); d_ref = make_attack(ref, "gra", _net(), **kw)(x, y)
    seed_all(3); d = make_attack(tab, "gra", _net(), **kw)(x, y)
    assert bits_equal(d.numpy(), d_ref.numpy())
    seed_all(5); d_ref = make_attack(ref, "adaea", nets, epoch=2)(x, y)
    seed_all(5); d = make_attack(tab, "adaea", nets, epoch=2)(x, y)
    assert int((d != d_ref).sum()) <= 1e-5 * d.numel()


def test_torch_ref_ens_and_composite(ref):
    from oracle import torch_ref
    x, y = _data()
    nets = [_net(0), _net(3)]
    d_ref = make_attack(ref, "ens", nets, epoch=3)(x, y)
    ens = torch_ref.RefEnsemble([torch_ref.ref_wrap_model(n) for n in nets])
    assert bits_equal(torch_ref.ref_mifgsm(ens, epoch=3)(x, y).numpy(), d_ref.numpy())
    # DI-TI-MI as the survey composes it from the reference's own classes (SURVEY §3.2)
    DIM, TIM = ref.load_attack_class("dim"), ref.load_attack_class("tim")

    class Composite(DIM):
        def __init__(self, **kw):
            super().__init__(**kw)
            self.kernel = TIM.generate_kernel(self, "gaussian", 15)
        get_grad = TIM.get_grad
    net = _net()
    seed_all(4); d_ref = make_attack(ref, Composite, net, epoch=3)(x, y)
    seed_all(4); d = torch_ref.RefDITIMI(torch_ref.ref_wrap_model(net), epoch=3)(x, y)
    assert bits_equal(d.numpy(), d_ref.numpy())
    # … and with SIM's scale copies in front (config 3's "+SIM S=5" variant), again composed from the reference's own hooks
    SIM = ref.load_attack_class("sim")

    class Composite5(Composite):
        num_scale = 5

        def transform(self, x, **kw):
            return DIM.transform(self, SIM.transform(self, x))
        get_loss = SIM.get_loss
    seed_all(4); d_ref = make_attack(ref, Composite5, net, epoch=2)(x, y)
    seed_all(4); d = torch_ref.RefSIDITIMI(torch_ref.ref_wrap_model(net), epoch=2)(x, y)
    assert bits_equal(d.numpy(), d_ref.numpy())


# ---- drop-in matrix: reference plugin files on OUR base class ------------------------------------------------------------
GRADIENT = ["fgsm", "ifgsm", "mifgsm", "nifgsm", "vmifgsm", "vnifgsm", "emifgsm", "aifgtm", "ifgssm", "smifgrm", "vaifgsm",
            "rap", "pcifgsm", "iefgsm", "gra", "gnp", "mig", "dta", "pgn", "mef", "gifgsm", "rgmifgsm", "dual_mifgsm",
            "ens_mifgsm", "fgsra", "gaa", "foolmix", "adamsi_fgm"]
INPUT_T = ["dim", "tim", "sim", "dem", "admix", "maskblock", "sia", "usmm", "decowa", "l2t", "bsr"]
ENSEMBLE = ["ens", "svre", "adaea", "cwa"]
SMALL = {"epoch": 2}


def _try_make(pkg, name, nets, extra):
    kw = dict(extra)
    try:
        return make_attack(pkg, name, nets, **kw)
    except TypeError:
        kw.pop("epoch", None)
        return make_attack(pkg, name, nets, **kw)


# reference plugin files that hard-code `.cuda()` (pifgsm.py:52, ssm.py:50-52, …): runnable on this GPU-less box once
# Tensor.cuda / Module.cuda are shimmed to the identity — the plugin FILES stay unmodified
CUDA_HARDCODED = ["pifgsm", "ssm"]          # (su / lpm / everywhere / stm need a feature-hook model, scikit-opt, a target or checkpoints)


@pytest.mark.parametrize("name", CUDA_HARDCODED)
def test_reference_plugin_with_cuda_shim_runs_unchanged_on_this_base(ref, adopted, name, monkeypatch):
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.nn.Module, "cuda", lambda self, *a, **k: self)
    if name not in ref.attack_zoo:
        pytest.skip("not in the reference registry")
    test_reference_plugin_runs_unchanged_on_this_base(ref, adopted, name)


@pytest.mark.parametrize("name", GRADIENT + INPUT_T + ENSEMBLE)
def test_reference_plugin_runs_unchanged_on_this_base(ref, adopted, name):
    x, y = _data(2, 224)
    nets = [_net(0), _net(3), _net(5), _net(7)] if name in ENSEMBLE else _net(0)
    try:
        a_ref = _try_make(ref, name, nets, SMALL)
    except Exception as e:   # missing optional dependency / checkpoint in this container: not a property of the boundary
        pytest.skip("reference plugin %s does not instantiate here: %s" % (name, str(e)[:80]))
    if hasattr(a_ref, "epoch") and a_ref.epoch > 3:
        a_ref.epoch = 2
    seed_all(11)
    try:
        d_ref = a_ref(x, y)
    except Exception as e:
        pytest.skip("reference plugin %s does not run on CPU here: %s" % (name, str(e)[:80]))
    a_new = _try_make(adopted, name, nets, SMALL)
    if hasattr(a_new, "epoch") and a_new.epoch > 3:
        a_new.epoch = 2
    # it really is the reference's plugin file on top of OUR base class
    import transferattack_b200.attack as our_attack
    assert isinstance(a_new, our_attack.Attack) and type(a_new).__mro__[1].__module__.startswith("transferattack_adopted.")
    seed_all(11)
    d_new = a_new(x, y)
    assert d_new.shape == d_ref.shape
    assert bits_equal(d_new.detach().numpy(), d_ref.detach().numpy()), (name, n_diff_bits(d_new.detach().numpy(), d_ref.detach().numpy()))


def test_reference_plugins_are_never_graph_captured_unless_hook_free(adopted):
    """The reference's dim.py / tim.py define hooks (host coin flip; F.conv2d) and know nothing about CUDA graphs: on this base
    they stay eager. Its mifgsm.py only configures the base loop, whose hooks are ours → capturable."""
    assert make_attack(adopted, "mifgsm", _net())._graph_ok()
    assert make_attack(adopted, "ifgsm", _net())._graph_ok()
    for name in ("dim", "tim", "sim", "nifgsm", "admix"):
        assert not make_attack(adopted, name, _net())._graph_ok(), name
