"""oracle/torch_ref.py — the eager restatement every GPU end-to-end test is judged against — pinned without a reference checkout.

tests/test_reference_live.py compares the restatement bit for bit with the live, unmodified reference on the configurations
below (same surrogate, inputs, seeds and arguments). That needs a checkout of the reference; this module needs none. It keeps
each of those perturbations as the SHA-256 of its float32 bytes plus a fixed sample of its values
(tests/golden/torch_ref_cases.npz), so a change to RefDITIMI, RefSIDITIMI, RefSSM, RefGRA, RefAdaEA, RefPIFGSM, RefEnsemble or
the base loop is caught on every run. It also keeps the live tests' other checks that need only those perturbations: the
native GRA / AdaEA / SSM plugins against them, and the float64 matrix form of SSM's transform against its FFT formulation.

The digests were recorded from oracle/torch_ref.py while it was held bit-identical to the reference by the live tests:

    python tests/test_torch_ref_golden.py        # rewrites tests/golden/torch_ref_cases.npz
"""
import hashlib
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

from conftest import GOLDEN, load_golden  # noqa: E402
from helpers import TinyNet, make_attack, seed_all  # noqa: E402

N_SAMPLE = 512

# test_reference_live.TORCH_REF_CASES
ZOO_CASES = {
    "fgsm": {}, "ifgsm": {}, "mifgsm": {}, "nifgsm": {}, "dim": {}, "tim": {}, "sim": {"epoch": 3}, "admix": {"epoch": 2},
    "vmifgsm": {"num_neighbor": 3, "epoch": 3}, "vnifgsm": {"num_neighbor": 2, "epoch": 3}, "emifgsm": {"epoch": 3},
}
PIFGSM_CASES = [{"epoch": 4}, {"epoch": 3, "decay": 1.0, "kern_size": 5}]
SSM_KW = {"num_spectrum": 2, "epoch": 2}
GRA_KW = {"num_neighbor": 3, "epoch": 3}
ADAEA_SEEDS = [0, 3, 5, 7]


def _net(seed=0, classes=1000):
    torch.manual_seed(seed)
    return TinyNet(classes).eval()


def _data(B=2, S=224):
    g = torch.Generator().manual_seed(1)
    return torch.rand(B, 3, S, S, generator=g), torch.randint(0, 1000, (B,), generator=g)


def _spectrum_inputs():
    g = torch.Generator().manual_seed(9)
    img = torch.rand(2, 3, 224, 224, generator=g)
    return img, torch.rand(2, 3, 224, 224, generator=g) + 0.5


def _case(key):
    """The restatement's output for one configuration of tests/test_reference_live.py, computed as that test computes it."""
    from oracle import torch_ref as R
    wrap = R.ref_wrap_model
    x, y = _data()
    if key.startswith("zoo_"):
        name = key[4:]
        net = _net()
        seed_all(3)
        return R.REF_ZOO[name](wrap(net), **ZOO_CASES[name])(x, y)
    if key.startswith("pifgsm_"):
        return R.RefPIFGSM(wrap(_net()), **PIFGSM_CASES[int(key[7:])])(x, y)
    if key == "ssm":
        net = _net()
        seed_all(3)
        return R.RefSSM(wrap(net), **SSM_KW)(x, y)
    if key == "ssm_fft":
        img, mask = _spectrum_inputs()
        r = R.RefSSM.__new__(R.RefSSM)
        return r.idct_2d(r.dct_2d(img) * mask)
    if key == "gra":
        seed_all(3)
        return R.RefGRA(wrap(_net()), **GRA_KW)(x, y)
    if key == "adaea":
        nets = [_net(s) for s in ADAEA_SEEDS]
        seed_all(5)
        return R.RefAdaEA(R.RefEnsemble([wrap(n) for n in nets]), epoch=2)(x, y)
    if key == "ens":
        nets = [_net(0), _net(3)]
        return R.ref_mifgsm(R.RefEnsemble([wrap(n) for n in nets]), epoch=3)(x, y)
    if key == "ditimi":
        net = _net()
        seed_all(4)
        return R.RefDITIMI(wrap(net), epoch=3)(x, y)
    if key == "siditimi":
        net = _net()
        seed_all(4)
        return R.RefSIDITIMI(wrap(net), epoch=2)(x, y)
    raise KeyError(key)


KEYS = (["zoo_" + n for n in sorted(ZOO_CASES)] + ["pifgsm_%d" % i for i in range(len(PIFGSM_CASES))]
        + ["ssm", "ssm_fft", "gra", "adaea", "ens", "ditimi", "siditimi"])


def _f32(t):
    return np.ascontiguousarray(t.detach().cpu().numpy(), dtype=np.float32)


def _digest(a):
    return np.frombuffer(hashlib.sha256(a.tobytes()).digest(), np.uint8)


def _sample_index(n):
    return np.sort(np.random.default_rng(0).choice(n, min(n, N_SAMPLE), replace=False))


@pytest.fixture(scope="module")
def G():
    return load_golden("torch_ref_cases")


@pytest.fixture
def oracle_backend():
    from transferattack_b200 import ops
    from oracle_backend import OracleBackend
    ops._install_backend_for_tests(OracleBackend())
    yield
    ops._install_backend_for_tests(None)


def _check(G, key, d):
    a = _f32(d)
    assert list(a.shape) == list(G[key + "_shape"]), (key, a.shape)
    sample = a.reshape(-1)[_sample_index(a.size)]
    assert np.array_equal(_digest(a), G[key + "_sha256"]), (
        key, "%d of %d sampled values differ" % (int((sample.view(np.uint32) != G[key + "_sample"].view(np.uint32)).sum()), sample.size))


@pytest.mark.parametrize("key", KEYS)
def test_torch_ref_matches_recorded_output(G, key):
    _check(G, key, _case(key))


def test_spectrum_matrix_form_matches_fft_formulation(G):
    """SSM's transform as the float64 matrix product the tcgen05 kernel is tested against (oracle.spectrum_transform) and as the
    reference's FFT chain (input_transformation/ssm.py:41-55, restated in RefSSM) agree to 2e-6."""
    import oracle
    img, mask = _spectrum_inputs()
    fft = _case("ssm_fft")
    _check(G, "ssm_fft", fft)
    assert np.abs(fft.numpy() - oracle.spectrum_transform(img.numpy(), None, mask.numpy())).max() <= 2e-6


def test_native_plugins_track_recorded_outputs(G, oracle_backend):
    """The native GRA, AdaEA and SSM plugins (kernels replaced by the C oracle's stand-in) against the recorded perturbations,
    with the bounds of tests/test_reference_live.py: GRA bit for bit, AdaEA within 1e-5 of the elements, SSM >= 90 % equal."""
    import transferattack_b200 as tab
    x, y = _data()
    ref = {k: _case(k) for k in ("gra", "adaea", "ssm")}
    for k, d in ref.items():
        _check(G, k, d)
    seed_all(3)
    d = make_attack(tab, "gra", _net(), **GRA_KW)(x, y)
    assert torch.equal(d, ref["gra"])
    nets = [_net(s) for s in ADAEA_SEEDS]          # built before seeding: _net() reseeds torch
    seed_all(5)
    d = make_attack(tab, "adaea", nets, epoch=2)(x, y)
    assert int((d != ref["adaea"]).sum()) <= 1e-5 * d.numel()
    net = _net()
    seed_all(3)
    d = make_attack(tab, "ssm", net, **SSM_KW)(x, y)
    assert float((d == ref["ssm"]).float().mean()) >= 0.9


if __name__ == "__main__":
    out = {}
    for key in KEYS:
        a = _f32(_case(key))
        out[key + "_sha256"] = _digest(a)
        out[key + "_shape"] = np.array(a.shape, np.int64)
        out[key + "_sample"] = a.reshape(-1)[_sample_index(a.size)]
    np.savez_compressed(os.path.join(GOLDEN, "torch_ref_cases.npz"), **out)
    print(len(KEYS), "cases,", os.path.getsize(os.path.join(GOLDEN, "torch_ref_cases.npz")), "bytes")
