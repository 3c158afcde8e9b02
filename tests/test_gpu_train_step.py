"""The on-device training step on a real B200: the cross-entropy kernel and the AdamW step against the float64
references of tests/_adamw_oracle.py, the skip on non-finite gradients, the exactness of the in-place weight refresh,
whole training runs against float64 torch through the oracle's forward, SimpleViT, and the errors."""
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import vit_torch
from vit_flax_b200 import SimpleViT, ViT, _lib, adamw, init_params, load_params, perturb_params, save_params
from vit_flax_b200._lib import VitB200Error
from vit_flax_b200.engine import Engine
from vit_flax_b200.params import flatten_params
from vit_flax_b200.runtime import clear_cache
from vit_flax_b200.simple_vit import clear_cache as clear_simple_cache, posemb_sincos_2d
from vit_flax_b200.train import _fold_in
from _adamw_oracle import adamw_ref, xent_ref
from _util import C2, TINY, images_for

pytestmark = pytest.mark.gpu

TINY_MEAN2 = dict(image_size=(16, 32), patch_size=(8, 16), num_classes=16, dim=128, depth=1, heads=2, mlp_dim=64)
SIMPLE = dict(image_size=32, patch_size=8, num_classes=10, dim=64, depth=2, heads=2, mlp_dim=128)
TOL = {"fp16": 2e-2, "bf16": 8e-2}
HP = dict(lr=1e-2, b1=0.9, b2=0.99, eps=1e-8, weight_decay=0.05)


@pytest.fixture(scope="module")
def lib(lib_built):
    assert lib_built.vitb200_device_count() >= 1, "no sm_100 device"
    return lib_built


@pytest.fixture(autouse=True)
def _fresh_cache():
    yield
    clear_cache()
    clear_simple_cache()
    torch.cuda.empty_cache()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def rel_err(got, want):
    want = np.asarray(want, dtype=np.float64)
    return float(np.abs(np.asarray(got, dtype=np.float64) - want).max() / max(np.abs(want).max(), 1e-30))


def split(eng, flat):
    return {p: flat[off: off + int(np.prod(s))].reshape(s) for p, (off, s) in eng.leaf_offsets().items()}


def params_of(eng):
    return {p: eng.get_param(p) for p in eng.param_table()}


def moments_of(eng):
    mu, nu, cnt = eng.optim_state()
    return split(eng, mu.cpu().numpy()), split(eng, nu.cpu().numpy()), int(cnt.cpu()[0])


def tiny_engine(precision="fp16", cfg=TINY, batch=8, **kw):
    variables = perturb_params(init_params(seed=3, **cfg), seed=4)
    eng = Engine(precision=precision, max_batch=batch, **kw, **cfg)
    eng.load_params(variables)
    return eng, variables


def forward_backward(eng, cfg, batch, seed, bad=False):
    x = torch.as_tensor(images_for(cfg, batch, seed=seed), device="cuda")
    eng.train_forward(x)
    dl = torch.as_tensor(np.random.default_rng(seed).standard_normal((batch, cfg["num_classes"])).astype(np.float32),
                         device="cuda")
    if bad:
        dl[0, 1] = float("inf")
    eng.backward(dl)


# ---------------------------------------------------------------- 1. cross-entropy kernel
@pytest.mark.parametrize("eps", [0.0, 0.1])
@pytest.mark.parametrize("B", [1, 7, 256])
@pytest.mark.parametrize("Cn", [10, 1000, 37])
def test_xent_kernel_matches_float64(lib, Cn, B, eps):
    rng = np.random.default_rng(Cn + B)
    z = (rng.standard_normal((B, Cn)) * 3).astype(np.float32)
    z[0, :2] = [1e4, -1e4]                      # stability: logits of magnitude 1e4
    if B > 1:
        z[-1] *= 3000.0
    y = rng.integers(0, Cn, B).astype(np.int32)
    zt, yt = torch.as_tensor(z, device="cuda"), torch.as_tensor(y, device="cuda")
    loss = torch.empty((), device="cuda")
    dl = torch.empty_like(zt)
    _lib.check(lib.vitb200_softmax_xent(stream(), zt.data_ptr(), yt.data_ptr(), B, Cn, eps, 8.0, loss.data_ptr(), dl.data_ptr()))
    want_loss, want_dl = xent_ref(z, y, eps, dscale=8.0)
    assert abs(float(loss) - want_loss) <= 2e-6 * abs(want_loss)
    assert rel_err(dl.cpu().numpy(), want_dl) < 2e-6


def test_xent_out_of_range_label_is_nan(lib):
    z = torch.randn((4, 10), device="cuda")
    loss = torch.empty((), device="cuda")
    dl = torch.empty_like(z)
    for bad in (10, -1):
        y = torch.tensor([0, bad, 3, 4], dtype=torch.int32, device="cuda")
        _lib.check(lib.vitb200_softmax_xent(stream(), z.data_ptr(), y.data_ptr(), 4, 10, 0.0, 1.0, loss.data_ptr(), dl.data_ptr()))
        assert math.isnan(float(loss))
        d = dl.cpu().numpy()
        assert np.isnan(d[1]).all() and np.isfinite(d[[0, 2, 3]]).all()


# ---------------------------------------------------------------- 2. the update against the reference
@pytest.mark.parametrize("clip", [0.0, 0.05])
def test_update_matches_reference_on_the_same_gradients(lib, clip):
    eng, _ = tiny_engine()
    table = eng.param_table()
    frozen = {"pos_embedding", "Transformer_0/PreNorm_1/LayerNorm_0/bias", "Dense_1/bias"}
    decay = {p: p.endswith("kernel") for p in table}
    trainable = {p: p not in frozen for p in table}
    eng.set_leaf_flags({p: (_lib.LEAF_TRAINABLE if trainable[p] else 0) | (_lib.LEAF_DECAY if decay[p] else 0) for p in table})
    p0 = params_of(eng)
    params = {k: v.astype(np.float64) for k, v in p0.items()}
    mu = {k: np.zeros(s) for k, s in table.items()}
    nu = {k: np.zeros(s) for k, s in table.items()}
    count = 0
    for step in range(3):
        forward_backward(eng, TINY, 8, seed=10 + step)
        grads = split(eng, eng.grads_flat().cpu().numpy())
        eng.adamw_step(**HP, max_grad_norm=clip, grad_scale=0.5)
        params, mu, nu, count, _, norm = adamw_ref(params, grads, mu, nu, count, decay=decay, trainable=trainable,
                                                   max_grad_norm=clip, grad_scale=0.5, **HP)
        got_c, skipped, got_norm = eng.optim_status()
        assert (got_c, skipped) == (step + 1, 0) and got_norm == pytest.approx(norm, rel=1e-5)
        got_p = params_of(eng)
        got_mu, got_nu, _ = moments_of(eng)
        for k in table:
            if not trainable[k]:
                assert np.array_equal(got_p[k], p0[k]) and not got_mu[k].any() and not got_nu[k].any(), k
                continue
            assert rel_err(got_p[k], params[k]) < 2e-6, (step, k)
            assert rel_err(got_mu[k], mu[k]) < 2e-6, (step, k)
            assert rel_err(got_nu[k], nu[k]) < 2e-6, (step, k)
    if clip:
        assert norm > clip      # the clipping branch was taken


def test_update_is_deterministic(lib):
    """Two models with the same weights, moments and gradient buffer step to bit-identical weights and moments."""
    a, _ = tiny_engine()
    b, _ = tiny_engine()
    for step in range(2):
        forward_backward(a, TINY, 8, seed=20 + step)
        forward_backward(b, TINY, 8, seed=20 + step)
        b.grads_flat().copy_(a.grads_flat())
        a.adamw_step(**HP, max_grad_norm=0.1)
        b.adamw_step(**HP, max_grad_norm=0.1)
    pa, pb = params_of(a), params_of(b)
    assert all(np.array_equal(pa[k], pb[k]) for k in pa)
    ma, mb = a.optim_state(), b.optim_state()
    assert all(torch.equal(x, y) for x, y in zip(ma, mb))


# ---------------------------------------------------------------- 3. skip on non-finite gradients
def test_non_finite_gradients_skip_the_step(lib):
    eng, _ = tiny_engine()
    forward_backward(eng, TINY, 8, seed=30)
    eng.adamw_step(**HP)
    p1 = params_of(eng)
    mu1, nu1, c1 = moments_of(eng)
    forward_backward(eng, TINY, 8, seed=31, bad=True)
    eng.adamw_step(**HP)
    count, skipped, norm = eng.optim_status()
    assert (count, skipped) == (1, 1) and math.isnan(norm)
    p2 = params_of(eng)
    mu2, nu2, c2 = moments_of(eng)
    assert c2 == c1 == 1
    assert all(np.array_equal(p1[k], p2[k]) and np.array_equal(mu1[k], mu2[k]) and np.array_equal(nu1[k], nu2[k]) for k in p1)
    forward_backward(eng, TINY, 8, seed=32)
    grads = split(eng, eng.grads_flat().cpu().numpy())
    eng.adamw_step(**HP)
    want, _, _, t, _, _ = adamw_ref({k: v.astype(np.float64) for k, v in p1.items()}, grads, mu1, nu1, 1, **HP)
    assert t == 2 and eng.optim_status()[:2] == (2, 0)
    got = params_of(eng)
    assert max(rel_err(got[k], want[k]) for k in got) < 2e-6


# ---------------------------------------------------------------- 4. the refresh is exact
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_refreshed_weights_equal_a_fresh_load(lib, precision):
    variables = perturb_params(init_params(seed=5, **TINY), seed=6)
    tr = ViT(**TINY).trainer(variables, adamw(1e-2), precision=precision, max_batch=64)
    x64 = torch.as_tensor(images_for(TINY, 64, seed=7), device="cuda")
    x1 = x64[:1].clone()
    # small-batch forwards run as graphs keyed by the (images, logits) pointers: with fixed buffers, the calls after the
    # steps replay the graphs captured here, before any step
    outs = {64: torch.empty((64, 8), device="cuda"), 1: torch.empty((1, 8), device="cuda")}
    before = {b: tr._eng.forward(x, out=outs[b]).clone() for b, x in ((64, x64), (1, x1))}
    labels = torch.as_tensor(np.random.default_rng(8).integers(0, 8, 64), device="cuda")
    for _ in range(3):
        tr.step(x64, labels)
    trained = tr.params()
    fresh = Engine(precision=precision, max_batch=64, **TINY)
    fresh.load_params(trained)
    for b, x in ((64, x64), (1, x1)):
        got = tr._eng.forward(x, out=outs[b])
        assert got.data_ptr() == outs[b].data_ptr() and not torch.equal(got, before[b])
        assert torch.equal(got, fresh.forward(x))
        assert torch.equal(got, tr.apply(x))
        assert torch.equal(got, ViT(**TINY).apply(trained, x, precision=precision))
    assert torch.equal(tr._eng.train_forward(x64), fresh.train_forward(x64))
    assert not torch.equal(tr.apply(x64), ViT(**TINY).apply(variables, x64, precision=precision))


# ---------------------------------------------------------------- 5. training follows the float64 oracle
def _oracle_run(variables, img, labels, steps, lr, wd, **cfg):
    tree = flatten_params(variables)
    leaves = {k: torch.as_tensor(np.asarray(v)).to(torch.float64).clone().requires_grad_(True) for k, v in tree.items()}
    from vit_flax_b200.checkpoint import _unflatten
    opt = torch.optim.AdamW(list(leaves.values()), lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=wd)
    y = torch.as_tensor(labels, dtype=torch.int64)
    losses = []
    for _ in range(steps):
        opt.zero_grad()
        logits = vit_torch._vit_forward({"params": _unflatten(leaves)}, torch.as_tensor(img, dtype=torch.float64), **cfg)
        loss = torch.nn.functional.cross_entropy(logits, y)
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    return losses


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("cfg,pool", [(TINY, "cls"), (TINY_MEAN2, "mean")])
def test_training_follows_the_float64_oracle(lib, cfg, pool, precision):
    variables = perturb_params(init_params(seed=9, **cfg), seed=10)
    img = images_for(cfg, 16, seed=11)
    labels = np.random.default_rng(12).integers(0, cfg["num_classes"], 16)
    want = _oracle_run(variables, img, labels, 5, 1e-3, 1e-4, pool=pool, **cfg)
    tr = ViT(**cfg, pool=pool).trainer(variables, adamw(1e-3), precision=precision, max_batch=16)
    x = torch.as_tensor(img, device="cuda")
    got = [float(tr.step(x, labels)) for _ in range(5)]
    for k, (g, w) in enumerate(zip(got, want)):
        assert abs(g - w) <= TOL[precision] * abs(w), (k, got, want)
    assert tr.last_step()[:2] == (5, 0)


def test_overfits_a_small_batch(lib):
    variables = perturb_params(init_params(seed=13, **TINY), seed=14)
    x = torch.as_tensor(images_for(TINY, 32, seed=15), device="cuda")
    labels = torch.as_tensor(np.random.default_rng(16).integers(0, 8, 32), device="cuda")
    tr = ViT(**TINY).trainer(variables, adamw(3e-3, weight_decay=0.0), max_batch=32)
    losses = [tr.step(x, labels) for _ in range(150)]
    first, last = float(losses[0]), float(losses[-1])
    assert abs(first - math.log(8)) < 1.0 and last < 0.1, (first, last)


# ---------------------------------------------------------------- 6. other models
def test_dropout_training_draws_new_masks_and_learns(lib):
    cfg = dict(TINY, dropout=0.1, emb_dropout=0.1)
    variables = perturb_params(init_params(seed=17, **TINY), seed=18)
    x = torch.as_tensor(images_for(TINY, 16, seed=19), device="cuda")
    labels = torch.as_tensor(np.random.default_rng(20).integers(0, 8, 16), device="cuda")
    tr = ViT(**cfg).trainer(variables, adamw(3e-3, weight_decay=0.0), max_batch=16)
    with pytest.raises(ValueError, match="dropout"):
        tr.step(x, labels)
    assert len({_fold_in(7, k) for k in range(100)}) == 100
    eng = tr._eng                            # on the device: the key of step k gives its own masks, the same key the same
    logits = {}
    for name, k in (("k0", 0), ("k0 again", 0), ("k1", 1)):
        eng.set_dropout_key(_fold_in(7, k))
        logits[name] = eng.train_forward(x).clone()
    assert torch.equal(logits["k0"], logits["k0 again"]) and not torch.equal(logits["k0"], logits["k1"])
    losses = [float(tr.step(x, labels, rngs={"dropout": 7})) for _ in range(100)]
    assert np.mean(losses[-5:]) < 0.6 * np.mean(losses[:5]), losses


def test_simple_vit_freezes_what_it_lacks_and_round_trips(lib, tmp_path):
    m = SimpleViT(**SIMPLE)
    img = np.random.default_rng(21).standard_normal((8, 3, 32, 32)).astype(np.float32)
    variables = m.init({"params": 22}, img)
    tr = m.trainer(variables, adamw(1e-2), max_batch=8)
    labels = np.random.default_rng(23).integers(0, 10, 8)
    for _ in range(3):
        tr.step(img, labels)
    eng = tr._eng
    assert np.array_equal(eng.get_param("pos_embedding")[0], posemb_sincos_2d(4, 4, 64))
    for p in ("cls", "LayerNorm_0/bias", "Transformer_0/PreNorm_0/LayerNorm_0/bias",
              "Transformer_0/PreNorm_1/LayerNorm_0/bias", "Transformer_0/Attention_1/Dense_1/bias"):
        assert not eng.get_param(p).any(), p
    trained = tr.params()
    assert sorted(flatten_params(trained)) == sorted(flatten_params(variables))
    assert not np.array_equal(flatten_params(trained)["Dense_1/kernel"], flatten_params(variables)["Dense_1/kernel"])
    save_params(trained, tmp_path / "p.msgpack")
    back = load_params(tmp_path / "p.msgpack")
    np.testing.assert_array_equal(m.apply(back, img), tr.apply(img))


# ---------------------------------------------------------------- 7. isolation and errors
def test_training_does_not_touch_the_apply_cache(lib):
    variables = perturb_params(init_params(seed=24, **TINY), seed=25)
    img = images_for(TINY, 4, seed=26)
    before = ViT(**TINY).apply(variables, img)
    tr = ViT(**TINY).trainer(variables, adamw(1e-2), max_batch=4)
    for _ in range(2):
        tr.step(img, np.arange(4))
    np.testing.assert_array_equal(ViT(**TINY).apply(variables, img), before)
    assert not np.array_equal(tr.apply(img), before)


def test_update_and_backward_order_is_enforced(lib):
    eng, _ = tiny_engine()
    with pytest.raises(VitB200Error, match="backward"):
        eng.adamw_step(**HP)                                   # before any backward
    x = torch.as_tensor(images_for(TINY, 8, seed=27), device="cuda")
    dl = torch.randn((8, 8), device="cuda")
    eng.train_forward(x)
    eng.backward(dl, wrt="input")
    with pytest.raises(VitB200Error, match="backward"):
        eng.adamw_step(**HP)                                   # after an image-only backward
    eng.train_forward(x)
    eng.backward(dl)
    eng.adamw_step(**HP)
    with pytest.raises(VitB200Error, match="backward"):
        eng.adamw_step(**HP)                                   # twice on one backward
    eng.train_forward(x)
    eng.backward(dl)
    eng.adamw_step(**HP)
    with pytest.raises(VitB200Error, match="optimiser step"):
        eng.backward(dl)                                       # its forward ran on the old weights
    eng.train_forward(x)
    eng.backward(dl)
    with pytest.raises(VitB200Error):
        eng.adamw_step(**dict(HP, b1=1.5))
    assert eng.optim_status()[0] == 2


def test_softmax_xent_checks_its_inputs(lib):
    eng, _ = tiny_engine()
    z = torch.randn((4, 8), device="cuda")
    y = torch.tensor([0, 1, 2, 3], dtype=torch.int32, device="cuda")
    loss, _ = eng.softmax_xent(z, y)
    assert math.isfinite(float(loss))
    for bad_z, bad_y in ((z.double(), y), (z.t(), y), (z[:, :1].expand(4, 8), y), (z.cpu(), y), (z, y.long()), (z, y[:3]),
                         (z, y.cpu()), (z, y.view(4, 1))):
        with pytest.raises(ValueError):
            eng.softmax_xent(bad_z, bad_y)
    with pytest.raises(ValueError):
        eng.softmax_xent(z, y, dlogits=torch.empty((4, 7), device="cuda"))
    with pytest.raises(VitB200Error, match="device memory"):      # the C entry point checks where the buffers live
        lib_loss = torch.empty((), device="cuda")
        _lib.check(lib.vitb200_softmax_xent(stream(), z.data_ptr(), y.cpu().data_ptr(), 4, 8, 0.0, 1.0,
                                            lib_loss.data_ptr(), torch.empty_like(z).data_ptr()))


def test_fp32_training_is_refused(lib):
    variables = perturb_params(init_params(seed=28, **TINY), seed=29)
    with pytest.raises(ValueError, match="fp16 or bf16"):
        ViT(**TINY).trainer(variables, adamw(1e-3), precision="fp32")
    eng = Engine(precision="fp32", max_batch=2, **TINY)
    eng.load_params(variables)
    with pytest.raises(VitB200Error) as e:
        eng.adamw_step(**HP)
    assert e.value.code == -4


def test_state_dict_round_trip(lib):
    variables = perturb_params(init_params(seed=30, **TINY), seed=31)
    img = images_for(TINY, 8, seed=32)
    labels = np.random.default_rng(33).integers(0, 8, 8)
    a = ViT(**TINY).trainer(variables, adamw(1e-2), max_batch=8)
    for _ in range(3):
        a.step(img, labels)
    sd = a.state_dict()
    b = ViT(**TINY).trainer(perturb_params(init_params(seed=34, **TINY), seed=35), adamw(1e-2), max_batch=8)
    b.load_state_dict(sd)
    sd2 = b.state_dict()
    assert (sd2["count"], sd2["step"]) == (3, 3)
    for key in ("params", "mu", "nu"):
        fa, fb = flatten_params(sd[key]), flatten_params(sd2[key])
        assert sorted(fa) == sorted(fb) and all(np.array_equal(fa[k], fb[k]) for k in fa), key
    assert any(flatten_params(sd["mu"])[k].any() for k in flatten_params(sd["mu"]))
    np.testing.assert_array_equal(a.apply(img), b.apply(img))


# ---------------------------------------------------------------- 8. full size
def test_vit_b16_batch_256_steps_without_synchronising(lib):
    variables = perturb_params(init_params(seed=36, **C2), seed=37)
    tr = ViT(**C2).trainer(variables, adamw(1e-4, max_grad_norm=1.0), max_batch=256)
    x = torch.randn((256, 224, 224, 3), device="cuda")
    y = torch.randint(0, 1000, (256,), device="cuda")
    losses = [tr.step(x, y)]
    torch.cuda.synchronize()
    losses.append(tr.step(x, y))
    ev = torch.cuda.Event()
    ev.record()
    assert not ev.query(), "step waited for the GPU"
    losses.append(tr.step(x, y))
    count, skipped, norm = tr.last_step()
    assert count == 3 and skipped == 0 and math.isfinite(norm)
    assert all(math.isfinite(float(l)) for l in losses)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_trainer_on_a_second_device_while_the_first_is_current(lib):
    """Every launch of the step, the cross-entropy included, goes to the trainer's device, not the current one."""
    torch.cuda.set_device(0)
    variables = perturb_params(init_params(seed=44, **TINY), seed=45)
    img = images_for(TINY, 8, seed=46)
    labels = np.random.default_rng(47).integers(0, 8, 8)
    tr = ViT(**TINY).trainer(variables, adamw(1e-2), device=1, max_batch=8)
    losses = [tr.step(img, labels) for _ in range(3)]
    assert torch.cuda.current_device() == 0
    assert all(l.device == torch.device("cuda", 1) and math.isfinite(float(l)) for l in losses)
    assert tr.last_step()[:2] == (3, 0)
    ref = ViT(**TINY).trainer(variables, adamw(1e-2), device=0, max_batch=8)
    ref_losses = [float(ref.step(img, labels)) for _ in range(3)]
    np.testing.assert_allclose([float(l) for l in losses], ref_losses, rtol=1e-3)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        variables = perturb_params(init_params(seed=40, **TINY), seed=41)
        img = images_for(TINY, 8 * world, seed=42)[8 * rank: 8 * (rank + 1)]
        labels = np.random.default_rng(43).integers(0, 8, 8 * world)[8 * rank: 8 * (rank + 1)]
        tr = ViT(**TINY).trainer(variables, adamw(1e-2), device=rank, max_batch=8)
        for _ in range(2):
            tr.step(img, labels)
        flat = flatten_params(tr.params())
        digest = torch.as_tensor(np.concatenate([flat[k].ravel() for k in sorted(flat)]), device=f"cuda:{rank}")
        others = [torch.empty_like(digest) for _ in range(world)]
        dist.all_gather(others, digest)
        q.put((rank, all(torch.equal(o, digest) for o in others), tr.last_step()[0]))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_replicas_stay_identical():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = sorted(q.get(timeout=300) for _ in procs)
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    assert res == [(0, True, 2), (1, True, 2)]
