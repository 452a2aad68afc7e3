"""DIM over its whole draw space: every (rnd, top, left) the plugin can draw, on every launch path, eager and graph-replayed.

DIM (input_transformation/dim.py) draws rnd in [min(S, R), max(S, R)) and top, left in [0, R - rnd) with R = int(S * rate). The
kernels derive tap / inverse tables, band row maxima, shared-memory sizes and path eligibility from each draw on the host, so a
draw that sizes something wrong fails quietly. This module checks every draw against two references:

  * forward: bit-identical to torch CUDA's own F.interpolate -> F.pad -> F.interpolate chain (default blend);
  * adjoint: within a rounding bar of an fp64 restatement of the same operator. DIM is separable, y = M_top X M_left^T with
    M_off = A_{R->S}[:, off:off+rnd] A_{S->rnd} (S x S), A the dense bilinear matrix whose weights are built in fp32 exactly as
    ATen and host_taps build them and then held in fp64. The adjoint reference is Gin64 = M_top^T G M_left, and the bar is
        |gin - Gin64| <= 16 u (M_top^T |G| M_left)   elementwise, u = 2^-24 (exactly 0 where the right side is 0).
    The C oracle meets it within ~2 u and the adjoint of the neighbouring draw misses it (the CPU tests below pin both).

The CPU tests (no marker) pin the reference and the draw enumeration; the GPU tests sweep the static path
(ta_dim_*_ws), the graph path (ta_dim_*_dyn), whole batches and the dispatcher's size limits. TA_B200_TEST_DIM_ALL=1 makes the
sampled sweeps of the non-default kernel settings exhaustive."""
import ctypes
import os
import types

import numpy as np
import pytest
import torch

import oracle

U = 2.0 ** -24
BAR = 16.0                 # adjoint bar in units of u (see the module docstring)
CHUNK = 512                # records per pack upload / draws per host synchronisation

CASES = [(224, 1.1), (299, 1.1), (64, 1.5), (32, 2.0)]
COUNTS = {(224, 1.1): 3795, (299, 1.1): 8555, (64, 1.5): 11440, (32, 2.0): 11440}

# (dim.impl, dim.bwd, dim.fwdtab, dim.sepconst): the settings of test_kernels_gpu.py's dim_impl fixture
DEFAULT = (2, 0, 0, 1)
SETTINGS = {"default": (2, 0, 0, 1), "walk": (4, 0, 0, 1), "walk-wstab-rtpitch": (4, 0, 1, 0), "sep": (3, 0, 0, 1),
            "sep-wstab-rtpitch": (3, 0, 1, 0), "direct": (1, 0, 0, 1), "direct-gather-wstab": (1, 1, 1, 1), "fourpass": (0, 0, 0, 1)}
EXHAUSTIVE = os.environ.get("TA_B200_TEST_DIM_ALL", "") == "1"


# ---------------------------------------------------------------------------------------------------------- draw space
def draw_space(S, rate):
    """The plugin's draw domain (DIM.draw): rnd in [min(S, R), max(S, R)), top and left in [0, R - rnd)."""
    R = int(S * rate)
    for rnd in range(min(S, R), max(S, R)):
        rem = R - rnd
        for top in range(rem):
            for left in range(rem):
                yield rnd, top, left


def corner_draws(S, rate):
    """every rnd with (top, left) in {0, rem - 1}^2"""
    R = int(S * rate)
    out = []
    for rnd in range(min(S, R), max(S, R)):
        ends = sorted({0, R - rnd - 1})
        out += [(rnd, t, l) for t in ends for l in ends]
    return out


def sampled_draws(S, rate, frac=0.1, seed=0):
    """corners plus a fixed-seed sample of `frac` of the space (everything with TA_B200_TEST_DIM_ALL=1), in space order"""
    space = list(draw_space(S, rate))
    if EXHAUSTIVE:
        return space
    keep = set(corner_draws(S, rate))
    rng = np.random.default_rng(seed + S)
    keep.update(space[i] for i in rng.choice(len(space), int(round(frac * len(space))), replace=False))
    return [d for d in space if d in keep]


# ---------------------------------------------------------------------------------------------------------- fp64 reference
def interp_matrix(n_in, n_out):
    """Dense [n_out, n_in] bilinear resize (align_corners=False) with the weights of ATen / host_taps, computed in fp32:
    scale = (float)in/out, src = max(0, fmaf(scale, d + 0.5f, -0.5f)), l1 = src - i0, l0 = 1 - l1, i1 = i0 + (i0 < in - 1);
    then held in fp64. (fmaf: the product and the sum are exact in fp64, so one rounding to fp32 is the fused result.)"""
    scale = np.float32(n_in) / np.float32(n_out)
    d = np.arange(n_out, dtype=np.float64)
    src = (np.float64(scale) * (d + 0.5) - 0.5).astype(np.float32)
    src = np.maximum(src, np.float32(0.0))
    i0 = src.astype(np.int64)
    l1 = (src - i0.astype(np.float32)).astype(np.float32)
    l0 = (np.float32(1.0) - l1).astype(np.float32)
    i1 = i0 + (i0 < n_in - 1)
    A = np.zeros((n_out, n_in), np.float64)
    np.add.at(A, (np.arange(n_out), i0), l0.astype(np.float64))
    np.add.at(A, (np.arange(n_out), i1), l1.astype(np.float64))
    return A


class Reference:
    """M_off matrices of one (S, R) in fp64 on `device`, cached per (rnd, off)."""

    def __init__(self, S, R, device):
        self.S, self.R, self.device = S, R, device
        self.A2 = torch.from_numpy(interp_matrix(R, S)).to(device)      # [S, R]
        self.A1 = {}
        self.M = {}

    def m(self, rnd, off):
        key = (rnd, off)
        if key not in self.M:
            if rnd not in self.A1:
                self.A1[rnd] = torch.from_numpy(interp_matrix(self.S, rnd)).to(self.device)   # [rnd, S]
            self.M[key] = self.A2[:, off:off + rnd] @ self.A1[rnd]
        return self.M[key]

    def forward(self, x64, rnd, top, left):
        return self.m(rnd, top) @ x64 @ self.m(rnd, left).T

    def adjoint(self, g2, rnd, top, left):
        """g2 = stack([G, |G|]) in fp64 -> stack([Gin64, M_top^T |G| M_left])"""
        return self.m(rnd, top).T @ g2 @ self.m(rnd, left)


def stack_abs(g):
    g = g.double()
    return torch.stack([g, g.abs()])


def ratio_u(out, ref2):
    """elementwise |out - ref| / (u * bound) with ref2 = stack([ref, bound]); 0 where both are 0, huge where only the error is
    not, NaN for a NaN output"""
    err = (out.double() - ref2[0]).abs()
    return err / (U * ref2[1] + 1e-300)


def first_bad(mask):
    idx = torch.nonzero(mask.reshape(-1))
    return int(mask.sum()), (int(idx[0, 0]) if len(idx) else None)


# ---------------------------------------------------------------------------------------------------------- CPU: pins
def _scaled_planes(rng, S, scales):
    g = rng.standard_normal((len(scales) + 1, S, S))
    g[:len(scales)] *= np.asarray(scales)[:, None, None]
    g[-1] = 0.0                                                        # one all-zero plane
    return g.astype(np.float32)


def _oracle_sample():
    rng = np.random.default_rng(28)
    space = list(draw_space(224, 1.1))
    pick = [space[i] for i in rng.choice(len(space), 24, replace=False)]
    return [(224, 0, 0), (224, 21, 21), (245, 0, 0), (235, 5, 6)] + pick


ORACLE_SCALES = [1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1, 1.0, 10.0]


def test_draw_space_counts():
    for (S, rate), n in COUNTS.items():
        assert sum(1 for _ in draw_space(S, rate)) == n, (S, rate)
    assert len(set(draw_space(224, 1.1))) == 3795


@pytest.mark.parametrize("S,rate", CASES)
def test_plugin_draws_stay_in_the_draw_space(S, rate):
    from transferattack_b200.input_transformation.dim import DIM
    space = set(draw_space(S, rate))
    plugin = types.SimpleNamespace(resize_rate=rate, diversity_prob=0.5)
    state = torch.get_rng_state()
    try:
        for seed in range(4):
            torch.manual_seed(seed)
            for _ in range(500):
                p = DIM.draw(plugin, S)
                if p is None:
                    continue
                rnd, R, top, left = p
                assert R == int(S * rate) and (rnd, top, left) in space, (S, rate, seed, p)
    finally:
        torch.set_rng_state(state)


def test_reference_matches_the_oracle():
    """orc_dim_bwd / orc_dim_fwd (fp64 scatter, fp32 chain) against the matrix restatement, within the bar"""
    S, R = 224, 246
    ref = Reference(S, R, "cpu")
    rng = np.random.default_rng(5)
    g = _scaled_planes(rng, S, ORACLE_SCALES)
    x = rng.random((3, S, S), dtype=np.float32)
    g2, x2 = stack_abs(torch.from_numpy(g)), stack_abs(torch.from_numpy(x))
    worst_b = worst_f = 0.0
    for rnd, top, left in _oracle_sample():
        rb = ratio_u(torch.from_numpy(oracle.dim_bwd(g, rnd, R, top, left)), ref.adjoint(g2, rnd, top, left))
        rf = ratio_u(torch.from_numpy(oracle.dim_fwd(x, rnd, R, top, left, blend=1)), ref.forward(x2, rnd, top, left))
        worst_b, worst_f = max(worst_b, float(rb.max())), max(worst_f, float(rf.max()))
        assert float(rb.max()) <= BAR and float(rf.max()) <= BAR, (rnd, top, left, float(rb.max()), float(rf.max()))
    print("oracle vs fp64 reference: adjoint %.2f u, forward %.2f u" % (worst_b, worst_f))


def test_reference_rejects_the_neighbouring_draw():
    """the bar has power: the adjoint of (rnd, top, left +- 1) or (rnd, top +- 1, left) misses it on every sampled draw"""
    S, R = 224, 246
    ref = Reference(S, R, "cpu")
    g = _scaled_planes(np.random.default_rng(6), S, ORACLE_SCALES)
    g2 = stack_abs(torch.from_numpy(g))
    for rnd, top, left in _oracle_sample():
        want = ref.adjoint(g2, rnd, top, left)
        nl = left + 1 if left + 1 <= R - rnd else left - 1
        nt = top + 1 if top + 1 <= R - rnd else top - 1
        for t, l in ((top, nl), (nt, left)):
            r = float(ratio_u(torch.from_numpy(oracle.dim_bwd(g, rnd, R, t, l)), want).max())
            assert r > BAR, (rnd, top, left, "neighbour", t, l, r)


# ---------------------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def be():
    from transferattack_b200 import ops
    ops._install_backend_for_tests(None)
    return ops.backend()


class tuned:
    """set (dim.impl, dim.bwd, dim.fwdtab, dim.sepconst) and dim.tma; restore the defaults on exit"""

    def __init__(self, setting, tma=1):
        self.setting, self.tma = setting, tma

    def __enter__(self):
        from transferattack_b200 import _lib
        impl, bwd, fwdtab, sepconst = self.setting
        for k, v in (("dim.impl", impl), ("dim.bwd", bwd), ("dim.fwdtab", fwdtab), ("dim.sepconst", sepconst), ("dim.tma", self.tma)):
            _lib.tune_set(k, v)
        return self

    def __exit__(self, *a):
        from transferattack_b200 import _lib
        for k, v in (("dim.impl", 2), ("dim.bwd", 0), ("dim.fwdtab", 0), ("dim.sepconst", 1), ("dim.tma", 1)):
            _lib.tune_set(k, v)


def torch_chain(x, rnd, R, top, left):
    import torch.nn.functional as F
    S = x.shape[-1]
    y = F.interpolate(x, size=[rnd, rnd], mode="bilinear", align_corners=False)
    y = F.pad(y, [left, R - rnd - left, top, R - rnd - top], value=0)
    return F.interpolate(y, size=[S, S], mode="bilinear", align_corners=False)


def grad_planes(gen, shape):
    """N(0, 1) planes scaled by 10^k, k cycling through [-8, 3] over the planes, plus one all-zero plane at the end"""
    g = torch.randn(shape, generator=gen, device="cuda")
    flat = g.view(-1, shape[-2], shape[-1])
    k = torch.arange(flat.shape[0], device="cuda") % 12 - 8
    flat *= torch.pow(10.0, k.float())[:, None, None]
    flat[-1] = 0
    return g


class Checker:
    """Per-draw references of one (S, rate) with fixed inputs x [1, 3, S, S] and g [1, 13, S, S] (scales 1e-8 .. 1e3 and a zero
    plane). check() returns device scalars (forward differing elements, worst adjoint ratio in u); explain() recomputes one
    draw on the host side of the failure with counts and first indices."""

    def __init__(self, be, S, rate, seed=0, x=None, g=None):
        self.be, self.S, self.R = be, S, int(S * rate)
        gen = torch.Generator(device="cuda").manual_seed(seed)
        self.x = torch.rand((1, 3, S, S), generator=gen, device="cuda") if x is None else x
        self.g = grad_planes(gen, (1, 13, S, S)) if g is None else g
        self.g2 = stack_abs(self.g)
        self.ref = Reference(S, self.R, "cuda")
        self.cache = {}

    def refs(self, d):
        if d not in self.cache:
            rnd, top, left = d
            self.cache = {d: (torch_chain(self.x, rnd, self.R, top, left), self.ref.adjoint(self.g2, rnd, top, left))}
        return self.cache[d]

    def check(self, d):
        rnd, top, left = d
        yf, gref = self.refs(d)
        out = self.be.dim(self.x, rnd, self.R, top, left, True)
        gin = self.be.dim(self.g, rnd, self.R, top, left, False)
        return (out.view(torch.int32) != yf.view(torch.int32)).sum(), ratio_u(gin, gref).amax()

    def explain(self, d, what):
        rnd, top, left = d
        yf, gref = self.refs(d)
        out = self.be.dim(self.x, rnd, self.R, top, left, True)
        gin = self.be.dim(self.g, rnd, self.R, top, left, False)
        n, i = first_bad(out.view(torch.int32) != yf.view(torch.int32))
        r = ratio_u(gin, gref)
        m, j = first_bad(~(r <= BAR))
        return ("S=%d R=%d rnd=%d top=%d left=%d %s: forward %d differing elements (first flat index %s); adjoint %d elements over "
                "%g u (first flat index %s, worst %.3g u)" % (self.S, self.R, rnd, top, left, what, n, i, m, BAR, j, float(r.max())))


def sweep(checker, draws, runs, label):
    """runs: [(name, setting, tma)]; every draw under every run. Returns {name: worst ratio}."""
    worst = {name: torch.zeros((), dtype=torch.float64, device="cuda") for name, _, _ in runs}
    for c0 in range(0, len(draws), CHUNK):
        chunk = draws[c0:c0 + CHUNK]
        res = {name: [] for name, _, _ in runs}
        for d in chunk:
            for name, setting, tma in runs:
                with tuned(setting, tma):
                    res[name].append(checker.check(d))
        for name, setting, tma in runs:
            f = torch.stack([a for a, _ in res[name]]).cpu()
            b = torch.stack([b for _, b in res[name]])
            worst[name] = torch.maximum(worst[name], b.amax())
            b = b.cpu()
            bad = [k for k in range(len(chunk)) if int(f[k]) != 0 or not float(b[k]) <= BAR]
            if bad:
                with tuned(setting, tma):
                    msg = checker.explain(chunk[bad[0]], "%s %s tma=%d static" % (label, name, tma))
                pytest.fail("%d of %d draws fail; first: %s" % (len(bad), len(chunk), msg))
    return {name: float(w) for name, w in worst.items()}


# ---------------------------------------------------------------------------------------------------------- GPU: static path
@pytest.mark.gpu
@pytest.mark.parametrize("S,rate", CASES)
def test_static_every_draw_default(be, S, rate):
    """ta_dim_fwd_ws / ta_dim_bwd_ws (default settings) on every draw of the space"""
    draws = list(draw_space(S, rate))
    w = sweep(Checker(be, S, rate), draws, [("default", DEFAULT, 1)], "static")
    print("DIM static S=%d R=%d default: %d draws, worst adjoint %.3f u" % (S, int(S * rate), len(draws), w["default"]))


@pytest.mark.gpu
@pytest.mark.parametrize("S,rate", CASES)
def test_static_other_settings(be, S, rate):
    """every other kernel setting, and every setting with TMA off: corners of every rnd plus a fixed 10 % sample"""
    draws = sampled_draws(S, rate)
    runs = [(name, s, 1) for name, s in SETTINGS.items() if name != "default"] + [(name + "-notma", s, 0) for name, s in SETTINGS.items()]
    w = sweep(Checker(be, S, rate, seed=1), draws, runs, "static")
    for name, r in w.items():
        print("DIM static S=%d R=%d %s: %d draws, worst adjoint %.3f u" % (S, int(S * rate), name, len(draws), r))


# ---------------------------------------------------------------------------------------------------------- GPU: graph path
def _call(fn, *args):
    from transferattack_b200 import _lib
    _lib.check(fn(*args), fn.__name__)


@pytest.mark.gpu
@pytest.mark.parametrize("tma", [1, 0])
@pytest.mark.parametrize("name", list(SETTINGS))
@pytest.mark.parametrize("S,rate", CASES[:3])
def test_dyn_every_draw_equals_static(be, S, rate, name, tma):
    """ta_dim_fwd_dyn / ta_dim_bwd_dyn stepped by the device counter through packs of the whole draw space plus the identity
    record: bit-identical to ta_dim_*_ws with the same draw and the same kernel family. The graph path has no four-pass variant
    and no gather adjoint: for those settings the comparator is the direct kernels (dim.impl 1, dim.bwd 0)."""
    from transferattack_b200 import _lib
    lib = be.lib
    R = int(S * rate)
    impl, _, _, sepconst = SETTINGS[name]
    static_setting = (impl if impl else 1, 0, 0, sepconst)
    records = list(draw_space(S, rate)) + [None]
    gen = torch.Generator(device="cuda").manual_seed(7)
    P = 2
    x = torch.rand((1, P, S, S), generator=gen, device="cuda")
    g = torch.randn((1, P, S, S), generator=gen, device="cuda") * torch.tensor([1e-3, 1.0], device="cuda")[None, :, None, None]
    n = P * S * S
    stride = (n + 63) // 64 * 64                      # every output slot 256-byte aligned
    bufs = torch.empty((4, CHUNK, stride), device="cuda")
    ws = torch.empty(int(lib.ta_dim_ws_bytes()), dtype=torch.uint8, device="cuda")
    it = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    nb = 4 * stride
    checked = 0
    for c0 in range(0, len(records), CHUNK):
        chunk = records[c0:c0 + CHUNK]
        packs = be.dim_packs(chunk, S, R).cuda()
        be.counter_add(it, set_to=0)
        base = [bufs[k].data_ptr() for k in range(4)]
        with tuned(SETTINGS[name], tma):
            for i in range(len(chunk)):
                o = [ctypes.c_void_p(b + i * nb) for b in base]
                _call(lib.ta_dim_fwd_dyn, ptr(x), o[0], P, S, R, ptr(packs), len(chunk), ptr(it), ctypes.c_void_p(stream))
                _call(lib.ta_dim_bwd_dyn, ptr(g), o[1], P, S, R, ptr(packs), len(chunk), ptr(it), ctypes.c_void_p(stream))
                be.counter_add(it, delta=1)
        with tuned(static_setting, tma):
            for i, d in enumerate(chunk):
                o = [ctypes.c_void_p(b + i * nb) for b in base]
                if d is None:                                   # identity record: both directions copy
                    bufs[2, i, :n].copy_(x.reshape(-1)); bufs[3, i, :n].copy_(g.reshape(-1))
                    continue
                _call(lib.ta_dim_fwd_ws, ptr(x), o[2], P, S, d[0], R, d[1], d[2], ptr(ws), ctypes.c_void_p(stream))
                _call(lib.ta_dim_bwd_ws, ptr(g), o[3], P, S, d[0], R, d[1], d[2], ptr(ws), ctypes.c_void_p(stream))
        k = len(chunk)
        iv = bufs[:, :k, :n].view(torch.int32)
        diff = torch.stack([(iv[0] != iv[2]).sum(1), (iv[1] != iv[3]).sum(1)]).cpu()
        assert int(it.item()) == k
        for direction in (0, 1):
            bad = torch.nonzero(diff[direction]).flatten().tolist()
            if bad:
                i = bad[0]
                cnt, first = first_bad(iv[direction, i] != iv[direction + 2, i])
                pytest.fail("S=%d R=%d draw=%s %s tma=%d dyn vs static %s: %d differing elements (first flat index %s); %d of %d "
                            "records differ" % (S, R, chunk[i], name, tma, ("forward", "adjoint")[direction], cnt, first, len(bad), k))
        checked += k
    print("DIM dyn S=%d R=%d %s tma=%d: %d records (incl. identity) bit-identical to static" % (S, R, name, tma, checked))


# ---------------------------------------------------------------------------------------------------------- GPU: batches
@pytest.mark.gpu
def test_whole_batches(be):
    """corner draws and 3 random draws at 224 -> 246 over whole batches: every plane distinct, forward bit-identical to torch,
    adjoint within the bar everywhere (a skipped, duplicated or swapped plane fails)"""
    S, rate = 224, 1.1
    R = int(S * rate)
    rng = np.random.default_rng(11)
    space = list(draw_space(S, rate))
    draws = corner_draws(S, rate) + [space[i] for i in rng.choice(len(space), 3, replace=False)]
    ref = Reference(S, R, "cuda")
    gen = torch.Generator(device="cuda").manual_seed(12)
    worst = 0.0
    for B, C in [(1, 3), (3, 3), (64, 3), (341, 3), (64, 1), (64, 4)]:
        x = torch.rand((B, C, S, S), generator=gen, device="cuda")
        g = grad_planes(gen, (B, C, S, S))
        g2 = stack_abs(g)
        for rnd, top, left in draws:
            what = "S=%d R=%d rnd=%d top=%d left=%d default static B=%d C=%d" % (S, R, rnd, top, left, B, C)
            out = be.dim(x, rnd, R, top, left, True)
            n, i = first_bad(out.view(torch.int32) != torch_chain(x, rnd, R, top, left).view(torch.int32))
            assert n == 0, "%s forward: %d differing elements (first flat index %s)" % (what, n, i)
            r = ratio_u(be.dim(g, rnd, R, top, left, False), ref.adjoint(g2, rnd, top, left))
            m, j = first_bad(~(r <= BAR))
            assert m == 0, "%s adjoint: %d elements over %g u (first flat index %s, worst %.3g u)" % (what, m, BAR, j, float(r.max()))
            worst = max(worst, float(r.max()))
        del g2
    print("DIM batches: %d draws x 6 shapes, worst adjoint %.3f u" % (len(draws), worst))


# ---------------------------------------------------------------------------------------------------------- GPU: dispatcher
def _few_draws(S, rate):
    R = int(S * rate)
    mid = (S + R) // 2
    return [(S, 0, 0), (S, R - S - 1, 0), (S, 0, R - S - 1), (R - 1, 0, 0), (mid, 1, R - mid - 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("S,rate,names", [(512, 1.1, list(SETTINGS)),       # kDimMaxS: direct kernels, R = 563
                                          (512, 1.2, ["default"]),          # R = 614 > kDimMaxR: the four-pass kernels of dim.cu
                                          (513, 1.1, ["default"])])         # S > kDimMaxS: dim.cu
def test_dispatcher_sizes(be, S, rate, names):
    ch = Checker(be, S, rate, seed=3)
    for name in names:
        for tma in (1, 0):
            with tuned(SETTINGS[name], tma):
                for d in _few_draws(S, rate):
                    f, b = ch.check(d)
                    assert int(f) == 0 and float(b) <= BAR, ch.explain(d, "%s tma=%d static" % (name, tma))


@pytest.mark.gpu
def test_dispatcher_dyn_at_the_table_limit(be):
    """S = 512 (R = 563): graph path equal to the static path; beyond the tables (R = 614, S = 513) a clean refusal naming them"""
    from transferattack_b200 import _lib
    S, R = 512, 563
    draws = _few_draws(S, 1.1)
    x = torch.rand((1, 2, S, S), device="cuda"); g = torch.randn((1, 2, S, S), device="cuda")
    packs = be.dim_packs(draws, S, R).cuda()
    it = torch.zeros(1, dtype=torch.int32, device="cuda")
    for d in draws:
        assert torch.equal(be.dim_dyn(x, R, packs, len(draws), it, True), be.dim(x, d[0], R, d[1], d[2], True)), d
        assert torch.equal(be.dim_dyn(g, R, packs, len(draws), it, False), be.dim(g, d[0], R, d[1], d[2], False)), d
        be.counter_add(it, delta=1)
    for S2, R2 in ((512, 614), (513, 564)):
        with pytest.raises(RuntimeError, match=r"\(S <= 512, R <= 576\)"):
            be.dim_packs([(S2, 0, 0)], S2, R2)
        x2 = torch.zeros((1, 1, S2, S2), device="cuda")
        for fwd in (True, False):
            with pytest.raises(RuntimeError, match=r"\(S <= 512, R <= 576\)"):
                be.dim_dyn(x2, R2, packs, len(draws), it, fwd)
    assert "S <= 512" in _lib.last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SETTINGS))
def test_dispatcher_unaligned_view(be, name):
    """a contiguous view 4 bytes into its storage: TMA switches off and the bits are those of an aligned run with dim.tma = 0"""
    S, rate = 224, 1.1
    R = int(S * rate)
    ch = Checker(be, S, rate, seed=4)
    n = ch.x.numel()
    xs = torch.empty(n + 1, device="cuda"); xs[1:] = ch.x.reshape(-1)
    gs = torch.empty(ch.g.numel() + 1, device="cuda"); gs[1:] = ch.g.reshape(-1)
    xu, gu = xs[1:].view(ch.x.shape), gs[1:].view(ch.g.shape)
    assert xu.is_contiguous() and xu.data_ptr() % 16 == 4
    for d in _few_draws(S, rate):
        rnd, top, left = d
        with tuned(SETTINGS[name], 0):
            f0, b0 = be.dim(ch.x, rnd, R, top, left, True), be.dim(ch.g, rnd, R, top, left, False)
        with tuned(SETTINGS[name], 1):
            fu, bu = be.dim(xu, rnd, R, top, left, True), be.dim(gu, rnd, R, top, left, False)
            f, b = ch.check(d)
            assert int(f) == 0 and float(b) <= BAR, ch.explain(d, "%s aligned" % name)
        for direction, (a, c) in enumerate(((fu, f0), (bu, b0))):
            cnt, first = first_bad(a.view(torch.int32) != c.view(torch.int32))
            assert cnt == 0, "S=%d R=%d draw=%s %s unaligned %s: %d differing elements (first flat index %s)" % (
                S, R, d, name, ("forward", "adjoint")[direction], cnt, first)


@pytest.mark.gpu
def test_dispatcher_plane_limit(be):
    """planes <= 65535 (the grid's y extent): 65535 runs and matches torch; 65536 is refused on the host with TA_EINVAL and a
    message naming the limit, before any launch, on the static and the graph path"""
    from transferattack_b200 import _lib
    lib = be.lib
    S, R, d = 2, 3, (2, 0, 1)
    x = torch.rand((65535, 1, S, S), device="cuda")
    assert torch.equal(be.dim(x, d[0], R, d[1], d[2], True), torch_chain(x, d[0], R, d[1], d[2]))
    big = torch.rand((65536, 1, S, S), device="cuda"); out = torch.empty_like(big)
    ws = torch.empty(int(lib.ta_dim_ws_bytes()), dtype=torch.uint8, device="cuda")
    packs = be.dim_packs([d], S, R).cuda()
    it = torch.zeros(1, dtype=torch.int32, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    torch.cuda.synchronize()
    before = _lib.launch_count()
    for fn in (lib.ta_dim_fwd_ws, lib.ta_dim_bwd_ws):
        assert fn(p(big), p(out), 65536, S, d[0], R, d[1], d[2], p(ws), None) == _lib.TA_EINVAL
        assert "65535" in _lib.last_error(), _lib.last_error()
    for fn in (lib.ta_dim_fwd_dyn, lib.ta_dim_bwd_dyn):
        assert fn(p(big), p(out), 65536, S, R, p(packs), 1, p(it), None) == _lib.TA_EINVAL
        assert "65535" in _lib.last_error(), _lib.last_error()
    assert _lib.launch_count() == before
    with pytest.raises(RuntimeError, match="65535"):
        be.dim(big, d[0], R, d[1], d[2], True)


@pytest.mark.gpu
def test_dispatcher_shared_memory_limit(be):
    """an image whose bands do not fit a CTA's shared memory is refused with a message naming the limit"""
    S = 4096
    R = int(S * 1.1)
    x = torch.zeros((1, 1, S, S), device="cuda")
    for fwd in (True, False):
        with pytest.raises(RuntimeError, match="204800 B limit"):
            be.dim(x, S, R, 0, 0, fwd)
