"""The host front-end ``ViT`` and ``SimpleViT`` share (vit_flax_b200/runtime.py), without a GPU: the public surface of
both classes, and the engine cache driven through a recording fake ``Engine``."""
import inspect

import numpy as np
import pytest

from vit_flax_b200 import SimpleViT, ViT, flatten_params, runtime, simple_vit
from _util import TINY

SIMPLE = dict(image_size=32, patch_size=8, num_classes=10, dim=64, depth=2, heads=2, mlp_dim=128)

# str(inspect.signature(...)) of every public method, and the public names of each class
SURFACE = {
    ViT: {
        "apply": "(self, variables: 'Any', x: 'Any', rngs: 'Any' = None, *, precision: 'Optional[str]' = None, "
                 "device: 'Optional[int]' = None, max_batch: 'Optional[int]' = None, reload: 'bool' = False)",
        "apply_stream": "(self, variables: 'Any', batches, *, precision: 'Optional[str]' = None, "
                        "device: 'Optional[int]' = None, max_batch: 'int' = 256)",
        "attention_maps": "(self, variables: 'Any', x: 'Any', rngs: 'Any' = None, *, layers=None, "
                          "precision: 'Optional[str]' = None, device: 'Optional[int]' = None, "
                          "max_batch: 'Optional[int]' = None, reload: 'bool' = False)",
        "init": "(self, rngs: 'Any', x: 'Any') -> 'Dict[str, Dict]'",
        "num_params": "(self, channels: 'int' = 3) -> 'int'",
        "trainer": "(self, variables: 'Any', tx, *, precision: 'Optional[str]' = None, device: 'Optional[int]' = None, "
                   "max_batch: 'Optional[int]' = None)",
        "vjp": "(self, variables: 'Any', x: 'Any', rngs: 'Any' = None, *, wrt: 'str' = 'params', "
               "precision: 'Optional[str]' = None, device: 'Optional[int]' = None, max_batch: 'Optional[int]' = None)",
    },
    SimpleViT: {
        "apply": "(self, variables: 'Any', img: 'Any', rngs: 'Any' = None, *, precision: 'Optional[str]' = None, "
                 "device: 'Optional[int]' = None, max_batch: 'Optional[int]' = None, reload: 'bool' = False)",
        "attention_maps": "(self, variables: 'Any', img: 'Any', rngs: 'Any' = None, *, layers=None, "
                          "precision: 'Optional[str]' = None, device: 'Optional[int]' = None, "
                          "max_batch: 'Optional[int]' = None)",
        "init": "(self, rngs: 'Any', x: 'Any') -> 'Dict[str, Dict]'",
        "trainer": "(self, variables: 'Any', tx, *, precision: 'Optional[str]' = None, device: 'Optional[int]' = None, "
                   "max_batch: 'Optional[int]' = None)",
        "vjp": "(self, variables: 'Any', img: 'Any', *, wrt: 'str' = 'params', precision: 'Optional[str]' = None, "
               "device: 'Optional[int]' = None, max_batch: 'Optional[int]' = None)",
    },
}
PUBLIC_NAMES = {ViT: {"apply", "apply_stream", "attention_maps", "dim_head", "dropout", "emb_dropout", "init",
                      "num_params", "pool", "trainer", "vjp"},
                SimpleViT: {"apply", "attention_maps", "channels", "dim_head", "init", "trainer", "vjp"}}


@pytest.mark.parametrize("cls", [ViT, SimpleViT], ids=lambda c: c.__name__)
def test_public_surface_is_unchanged(cls):
    assert {n for n in dir(cls) if not n.startswith("_")} == PUBLIC_NAMES[cls]
    for name, sig in SURFACE[cls].items():
        assert str(inspect.signature(getattr(cls, name))) == sig, name


class FakeEngine:
    """Records what the cache does to it; ``forward_host`` returns zeros."""
    made = []

    def __init__(self, **kw):
        self.kw, self.loads, self.closed = kw, [], False
        self.max_batch = kw["max_batch"]
        FakeEngine.made.append(self)

    def load_params(self, tree):
        self.loads.append(flatten_params(tree))

    def set_dropout_key(self, key):
        pass

    def forward_host(self, images):
        return np.zeros((images.shape[0], self.kw["num_classes"]), np.float32)

    def close(self):
        self.closed = True


@pytest.fixture
def fake(monkeypatch):
    runtime.clear_cache()
    FakeEngine.made = []
    monkeypatch.setattr(runtime, "Engine", FakeEngine)
    yield FakeEngine
    runtime.clear_cache()


def test_same_variables_load_once_and_an_inplace_edit_reloads(fake):
    v = ViT(**TINY)
    img = np.zeros((2, 32, 32, 3), np.float32)
    variables = v.init(0, img)
    v.apply(variables, img, device=0)
    v.apply({"params": variables["params"]}, img, device=0)     # a new container around the same leaves
    assert len(fake.made) == 1 and len(fake.made[0].loads) == 1
    variables["params"]["Dense_0"]["kernel"] *= 0.5
    v.apply(variables, img, device=0)
    assert len(fake.made) == 1 and len(fake.made[0].loads) == 2
    kw = fake.made[0].kw
    assert (kw["pool"], kw["channels"], kw["precision"], kw["device"], kw["max_batch"]) == \
        ("cls", 3, runtime._DEFAULT_PRECISION, 0, 2)


def test_simple_vit_engine_config_and_leaves(fake):
    v = SimpleViT(**SIMPLE)
    img = np.zeros((2, 3, 32, 32), np.float32)
    variables = v.init(0, img)
    assert v.apply(variables, img, device=0).shape == (2, 10)
    v.apply(variables, img, device=0)
    (eng,) = fake.made
    assert {k: eng.kw[k] for k in ("pool", "nchw", "cls_token", "ln_eps", "channels")} == \
        dict(pool="mean", nchw=True, cls_token=False, ln_eps=1e-5, channels=3)
    assert len(eng.loads) == 1
    want = flatten_params(v._engine_tree(variables))
    assert sorted(eng.loads[0]) == sorted(want) and all(np.array_equal(eng.loads[0][k], want[k]) for k in want)


def test_larger_batch_replaces_the_engine_and_clear_cache_closes_both_models(fake):
    v, s = ViT(**TINY), SimpleViT(**SIMPLE)
    img, simg = np.zeros((1, 32, 32, 3), np.float32), np.zeros((1, 3, 32, 32), np.float32)
    variables, svariables = v.init(0, img), s.init(0, simg)
    v.apply(variables, img, device=0)
    v.apply(variables, np.zeros((4, 32, 32, 3), np.float32), device=0)
    first, second = fake.made
    assert first.closed and not second.closed and second.max_batch == 4 and len(second.loads) == 1
    v.apply(variables, img, device=0)                          # a smaller batch keeps the larger engine
    s.apply(svariables, simg, device=0)
    assert len(fake.made) == 3 and not any(e.closed for e in fake.made[1:])
    runtime.clear_cache()
    assert all(e.closed for e in fake.made)
    assert simple_vit.clear_cache is runtime.clear_cache      # the name SimpleViT callers used clears the same cache
