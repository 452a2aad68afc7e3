import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

from conftest import REF_ROOT  # noqa: F401  (a checkout of the unmodified reference, or "")


class TinyNet(nn.Module):
    """Same small CNN as tests/golden/make_golden.py (seeded init, eval mode)."""

    def __init__(self, classes=10):
        super().__init__()
        self.c1 = nn.Conv2d(3, 8, 3, stride=2, padding=1)
        self.c2 = nn.Conv2d(8, 16, 3, stride=2, padding=1)
        self.fc = nn.Linear(16, classes)

    def forward(self, x):
        x = torch.relu(self.c1(x))
        x = torch.relu(self.c2(x))
        return self.fc(x.mean(dim=(2, 3)))


def tiny_net(seed=0, device="cpu"):
    torch.manual_seed(seed)
    return TinyNet().eval().to(device)


def make_attack(pkg, name, net_or_list, wrap=None, ens=None, **kw):
    """Instantiate `pkg.load_attack_class(name)` with load_model overridden (the reference's documented override
    point, attack.py:40-65) to return the given seeded net(s) wrapped by the package's own wrap_model."""
    cls = pkg.load_attack_class(name) if isinstance(name, str) else name
    wrap = wrap or pkg.utils.wrap_model
    ens = ens or pkg.utils.EnsembleModel

    def load_model(self, _n):
        if isinstance(net_or_list, (list, tuple)):
            return ens([wrap(m) for m in net_or_list])
        return wrap(net_or_list)

    # graph_safe: this loader returns plain seeded torchvision / tiny nets (no host randomness in their forward), so the class
    # that supplies the surrogate opts in to CUDA-graph capture itself (attack.py: _GRAPH_HOOKS includes load_model)
    P = type("P_" + cls.__name__, (cls,), {"load_model": load_model, "graph_safe": True})
    return P(model_name="tiny", **kw)


def import_reference():
    """The unmodified reference package (from $TRANSFERATTACK_REFERENCE)."""
    if "timm" not in sys.modules:
        try:
            import timm  # noqa: F401
        except ModuleNotFoundError:
            t = types.ModuleType("timm")
            t.list_models = lambda *a, **k: []
            sys.modules["timm"] = t
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import transferattack
    return transferattack


def seed_all(s):
    torch.manual_seed(s)
    np.random.seed(s)
    import random
    random.seed(s)
