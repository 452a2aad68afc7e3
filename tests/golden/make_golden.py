"""Generate tests/golden/*.npz by running the UNMODIFIED reference (a checkout of Trustworthy-AI-Group/TransferAttack) on CPU:

    TRANSFERATTACK_REFERENCE=<checkout> python tests/golden/make_golden.py

Shims (SURVEY.md §8c; no reference source is edited or copied):
  * `timm` is absent → a stub module with `list_models()` is inserted before import;
  * `Attack.load_model` (a documented override point, attack.py:40-65) is overridden to return
    `wrap_model(<seeded random-weight net>)` because there is no network for pretrained weights.

Every array stored here is either an input we drew from a seeded generator or an output produced by the
reference's own code path (its classes' hooks / transforms / forward).
"""
import os
import sys
import tempfile
import types
import zlib

import numpy as np
import torch
import torch.nn as nn
import torchvision

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("TRANSFERATTACK_REFERENCE", "")


def import_reference():
    if not os.path.isdir(os.path.join(REF, "transferattack")):
        sys.exit("set TRANSFERATTACK_REFERENCE to a checkout of the unmodified reference")
    if "timm" not in sys.modules:
        try:
            import timm  # noqa: F401
        except ModuleNotFoundError:
            t = types.ModuleType("timm")
            t.list_models = lambda *a, **k: []
            sys.modules["timm"] = t
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import transferattack  # noqa: E402
    return transferattack


class TinyNet(nn.Module):
    """Small deterministic CNN used for the end-to-end goldens (seeded init, eval mode)."""

    def __init__(self, classes=10):
        super().__init__()
        self.c1 = nn.Conv2d(3, 8, 3, stride=2, padding=1)
        self.c2 = nn.Conv2d(8, 16, 3, stride=2, padding=1)
        self.fc = nn.Linear(16, classes)

    def forward(self, x):
        x = torch.relu(self.c1(x))
        x = torch.relu(self.c2(x))
        return self.fc(x.mean(dim=(2, 3)))


def tiny_net(seed=0):
    torch.manual_seed(seed)
    return TinyNet().eval()


def make(ta, name, net_or_list, **kw):
    from transferattack.utils import wrap_model, EnsembleModel
    cls = ta.load_attack_class(name)

    def load_model(self, _n):
        if isinstance(net_or_list, (list, tuple)):
            return EnsembleModel([wrap_model(m) for m in net_or_list])
        return wrap_model(net_or_list)

    P = type("P_" + name, (cls,), {"load_model": load_model})
    return P(model_name="tiny", **kw)


def f32(t):
    return t.detach().cpu().numpy().astype(np.float32)


def gen_hooks(ta):
    torch.manual_seed(11)
    B, C, H, W = 3, 3, 20, 20
    atk = make(ta, "mifgsm", tiny_net())
    g = torch.randn(B, C, H, W) * 1e-3
    g[0, 0, 0, :5] = 0.0                      # exact zeros: sign(0) = 0
    m = torch.randn(B, C, H, W)
    data = torch.rand(B, C, H, W)
    delta = (torch.rand(B, C, H, W) * 2 - 1) * atk.epsilon
    out = {"g": f32(g), "m": f32(m), "data": f32(data), "delta": f32(delta),
           "eps": np.float32(atk.epsilon), "alpha": np.float32(atk.alpha)}
    out["scale"] = f32(g.abs().mean(dim=(1, 2, 3)))
    atk.decay = 1.0
    out["mom_first"] = f32(atk.get_momentum(g, 0))
    out["mom_d1"] = f32(atk.get_momentum(g, m))
    atk.decay = 0.7
    out["mom_d07"] = f32(atk.get_momentum(g, m))
    atk.decay = 0
    out["mom_d0"] = f32(atk.get_momentum(g, m))
    atk.decay = 1.0
    mom = atk.get_momentum(g, m)
    out["upd_linf"] = f32(atk.update_delta(delta, data, mom, atk.alpha))
    out["upd_linf_neg"] = f32(atk.update_delta(delta, data, mom, -atk.alpha))
    alpha_t = torch.rand(B, C, H, W) * atk.alpha
    out["alpha_t"] = f32(alpha_t)
    out["upd_linf_tensor"] = f32(atk.update_delta(delta, data, mom, alpha_t))
    # all-zero gradient sample → NaN momentum → sign(NaN)=0 → delta only box-clamped
    gz = g.clone(); gz[1] = 0
    mz = atk.get_momentum(gz, m)
    out["gz"] = f32(gz); out["mom_nan"] = f32(mz)
    out["upd_nan"] = f32(atk.update_delta(delta, data, mz, atk.alpha))
    # L2
    atk.norm = "l2"
    big = torch.randn(B, C, H, W)
    out["g_l2"] = f32(big)
    out["upd_l2_small"] = f32(atk.update_delta(delta * 0.01, data, big, 0.01))      # stays inside the ball
    out["upd_l2_big"] = f32(atk.update_delta(delta, data, big, 2.0))                # renorm branch
    atk.norm = "linfty"
    # init_delta with random start: replay the draws to expose the pre-clamp noise
    atk.random_start = True
    torch.manual_seed(5)
    d0 = atk.init_delta(data)
    torch.manual_seed(5)
    noise = torch.zeros_like(data).uniform_(-atk.epsilon, atk.epsilon)
    out["init_noise"] = f32(noise); out["init_linf"] = f32(d0)
    atk.norm = "l2"
    torch.manual_seed(6)
    d1 = atk.init_delta(data)
    torch.manual_seed(6)
    nrm = torch.zeros_like(data).normal_(-atk.epsilon, atk.epsilon)
    r = torch.zeros_like(data).uniform_(0, 1)
    out["init_l2_normal"] = f32(nrm); out["init_l2_r"] = f32(r); out["init_l2"] = f32(d1)
    atk.norm = "linfty"; atk.random_start = False
    # NI look-ahead (nifgsm.py:39)
    ni = make(ta, "nifgsm", tiny_net())
    out["ni_x"] = f32(ni.transform(data + delta, momentum=m))
    out["ni_coef"] = np.float32(ni.alpha * ni.decay)
    out["x_adv"] = f32(data + delta)
    np.savez_compressed(os.path.join(HERE, "hooks.npz"), **out)


def gen_dim(ta):
    out = {}
    cases = [("s32", 2, 3, 32), ("s64", 1, 3, 64), ("s224", 1, 1, 224), ("s30", 1, 2, 30)]
    atk = make(ta, "dim", tiny_net())
    atk.diversity_prob = 1.0   # always transform (torch.rand(1) > 1.0 is never true)
    for seed, (tag, B, C, S) in enumerate(cases):
        for rep in range(1 if S == 224 else 2):
            key = "%s_%d" % (tag, rep)
            torch.manual_seed(100 + 7 * seed + rep)
            x = torch.rand(B, C, S, S, requires_grad=True)
            gout = torch.randn(B, C, S, S)
            rs = 300 + 13 * seed + rep
            torch.manual_seed(rs)
            y = atk.transform(x)
            (gin,) = torch.autograd.grad(y, x, gout)
            # replay the CPU-generator draws (dim.py:47,54,60,62): coin, rnd, top, left
            torch.manual_seed(rs)
            torch.rand(1)
            R = int(S * atk.resize_rate)
            rnd = torch.randint(low=min(S, R), high=max(S, R), size=(1,), dtype=torch.int32)
            rem = R - rnd
            top = torch.randint(low=0, high=rem.item(), size=(1,), dtype=torch.int32)
            left = torch.randint(low=0, high=rem.item(), size=(1,), dtype=torch.int32)
            out[key + "_x"] = f32(x); out[key + "_y"] = f32(y)
            out[key + "_gout"] = f32(gout); out[key + "_gin"] = f32(gin)
            out[key + "_params"] = np.array([int(rnd), R, int(top), int(left), rs], np.int32)
    np.savez_compressed(os.path.join(HERE, "dim.npz"), **out)


def gen_tim(ta):
    out = {}
    for kt, ks in [("gaussian", 15), ("uniform", 15), ("linear", 15), ("gaussian", 5), ("gaussian", 7), ("gaussian", 3)]:
        atk = make(ta, "tim", tiny_net(), kernel_type=kt, kernel_size=ks)
        key = "%s%d" % (kt, ks)
        out[key + "_kernel"] = f32(atk.kernel)
        for tag, (B, H, W) in {"a": (2, 32, 32), "b": (1, 224, 224), "c": (1, 17, 45)}.items():
            if tag == "b" and key != "gaussian15":
                continue
            torch.manual_seed(zlib.crc32((key + tag).encode()) % 1000)
            w = torch.randn(B, 3, H, W)
            delta = torch.zeros(B, 3, H, W, requires_grad=True)
            loss = (delta * w).sum()
            g = atk.get_grad(loss, delta)       # conv2d(w, K, padding='same', groups=3)
            out["%s_%s_in" % (key, tag)] = f32(w)
            out["%s_%s_out" % (key, tag)] = f32(g)
    np.savez_compressed(os.path.join(HERE, "tim.npz"), **out)


def gen_sim_admix_emi(ta):
    out = {}
    torch.manual_seed(21)
    B, C, H, W = 3, 3, 16, 16
    x = torch.rand(B, C, H, W, requires_grad=True)
    sim = make(ta, "sim", tiny_net())
    y = sim.transform(x)
    gout = torch.randn_like(y)
    (gin,) = torch.autograd.grad(y, x, gout)
    out.update(sim_x=f32(x), sim_y=f32(y), sim_gout=f32(gout), sim_gin=f32(gin), sim_S=np.int32(sim.num_scale))
    lab = torch.tensor([1, 2, 3])
    out["sim_labels"] = lab.repeat(sim.num_scale).numpy()

    adm = make(ta, "admix", tiny_net())
    torch.manual_seed(22)
    y = adm.transform(x)
    torch.manual_seed(22)
    perms = np.stack([torch.randperm(B).numpy() for _ in range(adm.num_admix)]).astype(np.int32)
    gout = torch.randn_like(y)
    (gin,) = torch.autograd.grad(y, x, gout)
    out.update(admix_y=f32(y), admix_perm=perms, admix_gout=f32(gout), admix_gin=f32(gin),
               admix_S=np.int32(adm.num_scale), admix_A=np.int32(adm.num_admix),
               admix_strength=np.float32(adm.admix_strength))

    emi = make(ta, "emifgsm", tiny_net())
    gbar = torch.randn(B, C, H, W)
    y = emi.transform(x, grad=gbar)
    gout = torch.randn_like(y)
    (gin,) = torch.autograd.grad(y, x, gout)
    factors = np.linspace(-emi.radius, emi.radius, num=emi.num_sample)
    out.update(emi_gbar=f32(gbar), emi_y=f32(y), emi_gout=f32(gout), emi_gin=f32(gin),
               emi_coef=np.array([np.float32(f * emi.alpha) for f in factors], np.float32),
               emi_y0=f32(emi.transform(x, grad=0)))
    np.savez_compressed(os.path.join(HERE, "sim_admix_emi.npz"), **out)


def gen_vmi(ta):
    """Drive the reference's get_variance (vmifgsm.py:42-58) with scripted gradients / noise so its own
    accumulate (`grad += ...`) and finalize (`grad / N - cur_grad`) lines produce the golden."""
    out = {}
    torch.manual_seed(31)
    B, C, H, W = 2, 3, 12, 12
    N = 4
    data = torch.rand(B, C, H, W)
    delta = ((torch.rand(B, C, H, W) * 2 - 1) * (16 / 255)).requires_grad_(True)
    grads = [torch.randn(B, C, H, W) * 1e-3 for _ in range(N)]
    cur = torch.randn(B, C, H, W) * 1e-3
    seen = []
    base = ta.load_attack_class("vmifgsm")

    class P(base):
        def load_model(self, _n):
            from transferattack.utils import wrap_model
            return wrap_model(tiny_net())

        def get_logits(self, x, **kw):
            seen.append(x.detach().clone())
            return x

        def get_loss(self, logits, label):
            return logits.sum()

        def get_grad(self, loss, delta, **kw):
            return grads[len(seen) - 1]

    atk = P(model_name="tiny", num_neighbor=N)
    torch.manual_seed(32)
    v = atk.get_variance(data, delta, None, cur, 0)
    torch.manual_seed(32)
    noises = [torch.zeros_like(delta).uniform_(-atk.radius, atk.radius) for _ in range(N)]
    out.update(data=f32(data), delta=f32(delta), cur=f32(cur), variance=f32(v), N=np.int32(N),
               grads=np.stack([f32(g) for g in grads]), noises=np.stack([f32(n) for n in noises]),
               x_near=np.stack([f32(s) for s in seen]), radius=np.float32(atk.radius))
    # vmifgsm.py:87 grad + variance
    out["g_plus_v"] = f32(cur + v)
    np.savez_compressed(os.path.join(HERE, "vmi.npz"), **out)


def gen_misc(ta):
    from transferattack.utils import wrap_model, save_images
    from PIL import Image
    out = {}
    torch.manual_seed(41)
    x = torch.rand(2, 3, 24, 24, requires_grad=True)
    pre = wrap_model(nn.Identity())[0]    # PreprocessingModel(224, ImageNet mean/std); Resize(224) of 24x24 upsamples
    # exercise Normalize only (Resize is a no-op at 224; here we call .normalize directly)
    y = pre.normalize(x)
    gout = torch.randn_like(y)
    (gin,) = torch.autograd.grad(y, x, gout)
    out.update(norm_x=f32(x), norm_y=f32(y), norm_gout=f32(gout), norm_gin=f32(gin),
               norm_mean=np.array(pre.normalize.mean, np.float32), norm_std=np.array(pre.normalize.std, np.float32))
    # save_images quantisation (utils.py:63-66) incl. the edge values from SURVEY Appendix B
    data = torch.rand(2, 3, 8, 8)
    delta = (torch.rand(2, 3, 8, 8) * 2 - 1) * (16 / 255)
    delta = torch.min(torch.max(delta, 0 - data), 1.0 - data)
    data[0, 0, 0, :4] = torch.tensor([0.9999999, 0.5, 254.9999 / 255, 1.0]); delta[0, 0, 0, :4] = 0
    with tempfile.TemporaryDirectory() as d:
        save_images(d, data + delta, ["a.png", "b.png"])
        u8 = np.stack([np.array(Image.open(os.path.join(d, f))) for f in ["a.png", "b.png"]])
    out.update(q_data=f32(data), q_delta=f32(delta), q_u8=u8)
    np.savez_compressed(os.path.join(HERE, "misc.npz"), **out)


def gen_e2e(ta):
    """Full reference runs on CPU with TinyNet(s). Machine-stable only as far as the CPU conv kernels
    are; `logits0` is stored as a fingerprint so the consumer can detect a host whose kernels differ."""
    B, S = 2, 32
    torch.manual_seed(1)
    x = torch.rand(B, 3, S, S)
    y = torch.randint(0, 10, (B,))
    runs = {
        "ifgsm": {}, "mifgsm": {}, "nifgsm": {}, "fgsm": {}, "tim": {}, "dim": {}, "sim": {}, "admix": {},
        "vmifgsm": {"num_neighbor": 3}, "vnifgsm": {"num_neighbor": 3}, "emifgsm": {},
        "mifgsm_rs": {"random_start": True}, "mifgsm_l2": {"norm": "l2", "epsilon": 1.0, "alpha": 0.2},
        "mifgsm_targeted": {"targeted": True},
    }
    out = {"x": f32(x), "y": y.numpy()}
    net = tiny_net(0)
    from transferattack.utils import wrap_model
    out["logits0"] = f32(wrap_model(net)(x))
    for key, kw in runs.items():
        name = key.split("_")[0]
        atk = make(ta, name, net, **kw)
        lab = torch.stack([y, (y + 1) % 10]) if kw.get("targeted") else y
        torch.manual_seed(2)
        np.random.seed(2)
        out["delta_" + key] = f32(atk(x, lab))
    ens = make(ta, "ens", [tiny_net(0), tiny_net(3)])
    torch.manual_seed(2)
    out["delta_ens"] = f32(ens(x, y))
    # per-iteration trace of MI-FGSM: inputs and outputs of get_momentum/update_delta as the reference ran them
    base = ta.load_attack_class("mifgsm")
    trace = []

    class T(base):
        def load_model(self, _n):
            return wrap_model(net)

        def get_momentum(self, grad, momentum, **kw):
            r = super().get_momentum(grad, momentum, **kw)
            trace.append(["g", f32(grad), "m_in", None if isinstance(momentum, (int, float)) else f32(momentum),
                          "scale", f32(grad.abs().mean(dim=(1, 2, 3))), "m_out", f32(r)])
            return r

        def update_delta(self, delta, data, grad, alpha, **kw):
            r = super().update_delta(delta, data, grad, alpha, **kw)
            trace[-1] += ["d_in", f32(delta), "d_out", f32(r)]
            return r

    T(model_name="tiny", epoch=4)(x, y)
    for i, rec in enumerate(trace):
        d = dict(zip(rec[0::2], rec[1::2]))
        for k, v in d.items():
            if v is not None:
                out["trace%d_%s" % (i, k)] = v
    out["trace_len"] = np.int32(len(trace))
    np.savez_compressed(os.path.join(HERE, "e2e.npz"), **out)


def main():
    torch.set_num_threads(1)   # run-to-run and host-to-host reproducible reduction order
    ta = import_reference()
    gen_hooks(ta)
    gen_dim(ta)
    gen_tim(ta)
    gen_sim_admix_emi(ta)
    gen_vmi(ta)
    gen_misc(ta)
    gen_e2e(ta)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
