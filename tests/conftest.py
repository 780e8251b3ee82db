"""pytest plumbing: `gpu` marker, repo root on sys.path, golden-fixture loader."""
import hashlib
import json
import math
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def rebuild_weight(shape, init_state, perturb_state, std):
    """A golden weight stored as its recipe instead of its values: nn.Conv2d's default init (kaiming_uniform_, a=sqrt(5))
    drawn from the CPU generator state `init_state`, plus make_golden.perturb()'s N(0, std^2) step drawn from
    `perturb_state`.  This replays the draws that made the weight the reference ran with, bit for bit."""
    gen = torch.Generator()
    gen.set_state(init_state)
    w = torch.empty(shape)
    torch.nn.init.kaiming_uniform_(w, a=math.sqrt(5), generator=gen)
    gen.set_state(perturb_state)
    return w.add_(torch.randn(shape, generator=gen) * std)


def sha256(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


class Golden(dict):
    """arrays as torch tensors; `.meta` dict; `.sd` = state-dict sub-mapping ('sd/' keys, plus the weights listed in
    meta['rebuilt'], which are stored as 'rng_init/' and 'rng_perturb/' generator states and rebuilt here)."""

    def __init__(self, name):
        super().__init__()
        with np.load(os.path.join(GOLDEN, name + ".npz")) as f:
            self.meta = json.loads(bytes(f["meta"]).decode())
            self.sd = {}
            for k in f.files:
                if k == "meta" or k.startswith("rng_"):
                    continue
                t = torch.from_numpy(np.array(f[k]))
                if k.startswith("sd/"):
                    self.sd[k[3:]] = t
                else:
                    self[k] = t
            for k, r in self.meta.get("rebuilt", {}).items():
                w = rebuild_weight(r["shape"], torch.from_numpy(f["rng_init/" + k]), torch.from_numpy(f["rng_perturb/" + k]),
                                   r["std"])
                assert sha256(w) == r["sha256"], "%s: %s does not rebuild bit-exactly with this torch" % (name, k)
                self.sd[k] = w


@pytest.fixture
def allow_library():
    """Tests on nets narrower than the kernels take (hidden width 8 / 16: attention head dim < 8, Linear K < 32) opt in
    to the library layers explicitly; everything else must run on flowk kernels only (`no_library`)."""
    from flowk import _lib
    old = _lib.ALLOW_LIBRARY
    _lib.ALLOW_LIBRARY = True
    yield _lib
    _lib.ALLOW_LIBRARY = old


@pytest.fixture
def no_library():
    """Asserts that the test body never routed a CUDA tensor to cuDNN / cuBLAS / ATen conditioner layers."""
    from flowk import _lib
    old, before = _lib.ALLOW_LIBRARY, _lib.LIBRARY_FALLBACKS
    _lib.ALLOW_LIBRARY = False
    yield _lib
    _lib.ALLOW_LIBRARY = old
    assert _lib.LIBRARY_FALLBACKS == before


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def load(name):
        if name not in cache:
            cache[name] = Golden(name)
        return cache[name]
    return load
