"""Classifier-free guidance (UbConfig.class_dropout, ub_trainer_set_guidance) on the GPU.  The oracle needs no change:
a guided model with K classes is oracle/unet_oracle.py's model with num_classes = K + 1, the null class being label K.

Training: the label drops (rate, independence, reproducibility, explicit -1), one forward + backward against the
oracle run on the effective labels, a 10-step captured loss trace against an eager replay.  Sampling: the guided
respaced sampler against the oracle's eps_u + s (eps_c - eps_u), identities (s = 1, s = 0, checkpoints), the training
state after sampling, and the calls the library refuses."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

import learn_sigma_oracle as LS
import spaced_oracle as SO
from test_trainer_gpu import check_grads

pytestmark = pytest.mark.gpu

K = 10                # classes of the guided model; the null class is label K
TOL_PARITY = 3e-2     # max-abs over max|ref|, the bound of test_sampler_spaced_gpu.py
TOL_RUNS = 2e-2       # two device runs (GroupNorm-statistics atomics), the bound of test_sampler_spaced_gpu.py
TOL_FULL_L2 = 3e-2    # relative L2 of a full run and of the learned range, as in test_sampler_spaced_gpu.py
SMALL = dict(H=32, W=32, channel_mult=(1, 2), att_start_level=1)


def _oracle_model(O, okw=None, v_scale=0.0):
    """Oracle config with K + 1 classes and perturb_zero_params weights; v_scale > 0 (six-output head) adds
    N(0, v_scale^2) to the head's v rows, so that the learned variance varies between pixels."""
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.UNetConfig(num_classes=K + 1, **(okw or {}))
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    if v_scale:
        off = 0
        for name, shape in O.param_spec(cfg):
            n = int(np.prod(shape))
            if name == "out.2.weight":
                w = flat[off:off + n].reshape(shape).clone()
                w[3:] += v_scale * torch.randn(w[3:].shape, generator=torch.Generator().manual_seed(7))
                flat = flat.clone()
                flat[off:off + n] = w.reshape(-1)
            off += n
    return cfg, flat


def _label_rows(O, cfg, g):
    off = sum(int(np.prod(s)) for _, s in O.param_spec(cfg)[:4])
    return g[off:off + (K + 1) * 4 * cfg.model_channels].reshape(K + 1, -1)


# ------------------------------------------------------------------------------------------------------------ training
def _drops(ub, tr, labels, steps):
    """Effective labels of `steps` captured or eager training steps (zero batch, lr = 0)."""
    tr.set_labels(np.asarray(labels, np.int32))
    x0 = np.zeros((tr.cfg.B, 3, tr.cfg.H, tr.cfg.W), np.float32)
    out = []
    for _ in range(steps):
        tr.train_step(x0, lr=0.0, want_loss=False)
        out.append(tr.get_effective_labels())
    return np.array(out)


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_drop_decisions(ub, p):
    B, steps = 32, 60
    labels = np.arange(B) % K
    tr = ub.Trainer(B=B, num_classes=K, class_dropout=p, **SMALL)
    eff = _drops(ub, tr, labels, steps)
    dropped = eff == -1
    assert ((eff == labels) | dropped).all()  # a kept label is the caller's
    n = dropped.size
    rate = dropped.mean()
    bound = 4.5 * math.sqrt(p * (1 - p) / n)
    print(f"p = {p}: drop rate {rate:.4f} over {n} coins (binomial bound +-{bound:.4f})")
    assert abs(rate - p) <= bound
    # independence: pairs of neighbouring images and the same image on consecutive steps are dropped together at p^2
    m = dropped.size - dropped.shape[0]
    pb = 4.5 * math.sqrt(p * p * (1 - p * p) / m)
    for both in ((dropped[:, 1:] & dropped[:, :-1]).mean(), (dropped[1:] & dropped[:-1]).mean()):
        assert abs(both - p * p) <= pb, (both, p * p, pb)
    assert dropped.sum(axis=1).max() < B  # not one coin per step
    tr.close()


def test_drops_reproducible_eager_and_captured(ub):
    B, steps, p = 16, 12, 0.5
    labels = np.arange(B) % K
    labels[[2, 9]] = -1
    kw = dict(B=B, num_classes=K, class_dropout=p, **SMALL)
    trs = [ub.Trainer(**kw), ub.Trainer(**kw, use_cuda_graph=0), ub.Trainer(**kw, seed=0x5eed + 1)]
    a, b, c = (_drops(ub, tr, labels, steps) for tr in trs)
    for tr in trs:
        tr.close()
    assert np.array_equal(a, b)           # the same seed: the same decisions, eager or captured
    assert not np.array_equal(a, c)       # another seed: other decisions
    assert (a[:, [2, 9]] == -1).all() and (c[:, [2, 9]] == -1).all()  # -1 stays null
    assert not np.array_equal(a[0], a[1])  # the step counter reaches the coins


CASES = [("default", {}, {}, 4),
         ("learn_sigma scale-shift", dict(learn_sigma=1, use_scale_shift_norm=1),
          dict(out_channels=6, use_scale_shift_norm=True), 2)]


@pytest.mark.parametrize("what,kw,okw,B", CASES, ids=[c[0] for c in CASES])
def test_forward_backward_matches_oracle(ub, oracle, what, kw, okw, B):
    """The oracle runs on the effective labels (-1 -> K).  Bounds of test_class_conditional_matches_oracle."""
    O = oracle
    cfg, flat = _oracle_model(O, okw, v_scale=0.05 if kw.get("learn_sigma") else 0.0)
    x0, t, noise = O.synthetic_batch(cfg, B)
    tr = ub.Trainer(B=B, num_classes=K, class_dropout=0.3, **kw)
    assert tr.nparams == flat.numel()
    tr.set_params(flat.numpy())
    tr.set_labels(np.array([3, -1, 7, 3][:B], np.int32))
    loss = tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    eff = tr.get_effective_labels()
    assert eff[1] == -1
    y = torch.from_numpy(np.where(eff < 0, K, eff)).long()
    out, g = tr.get_output(), tr.get_grads()
    if kw.get("learn_sigma"):
        loss_ref, _, _, out_ref, g_ref = LS.train_step_grads(O, cfg, flat, x0, t, noise, y)
    else:
        loss_ref, out_ref, g_ref = O.train_step_grads(cfg, flat, x0, t, noise, y)
    g_ref = g_ref.numpy()
    print(f"[cfg {what}] effective labels {eff}, loss {loss:.6g} (ref {float(loss_ref):.6g})")
    assert abs(loss - float(loss_ref)) <= 2e-3 * float(loss_ref)
    assert np.abs(out - out_ref.numpy()).max() <= 3e-2 * np.abs(out_ref.numpy()).max()
    rows = {name: rel for rel, name, _, _ in check_grads(O, cfg, g, g_ref, "cfg " + what)}
    assert rows["label_emb.weight"] <= 2e-2, rows["label_emb.weight"]
    ge = _label_rows(O, cfg, g)
    used = set(y.tolist())
    assert np.abs(ge[K]).max() > 0                                   # the null row learns
    assert np.abs(ge[[k for k in range(K + 1) if k not in used]]).max() == 0.0
    # the null row's gradient is non-zero exactly when the step dropped a label (no -1 among the labels now)
    tr.set_labels(np.array([3, 5, 7, 3][:B], np.int32))
    seen = set()
    for _ in range(20):
        tr.update(lr=0.0)  # (advances the step counter, leaves the parameters)
        tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
        any_drop = bool((tr.get_effective_labels() == -1).any())
        assert (np.abs(_label_rows(O, cfg, tr.get_grads())[K]).max() > 0) == any_drop
        seen.add(any_drop)
    assert seen == {True, False}
    tr.close()


def test_ten_step_captured_trace_matches_eager(ub, oracle):
    O = oracle
    cfg, flat = _oracle_model(O)
    B = 4
    kw = dict(B=B, num_classes=K, class_dropout=0.3)
    trs = [ub.Trainer(**kw), ub.Trainer(**kw, use_cuda_graph=0)]
    g = torch.Generator().manual_seed(5)
    batches = [(torch.rand(B, 3, 64, 64, generator=g) * 2 - 1, torch.randint(0, 1000, (B, 1), generator=g).float(),
                torch.randn(B, 3, 64, 64, generator=g)) for _ in range(10)]
    traces = []
    for tr in trs:
        tr.set_params(flat.numpy())
        tr.set_labels(np.array([1, 4, -1, 9], np.int32))
        losses, effs = [], []
        for x0, t, noise in batches:
            losses.append(tr.train_step(x0.numpy(), t.numpy(), noise.numpy(), lr=1e-4))
            effs.append(tr.get_effective_labels())
        traces.append((np.array(losses), np.array(effs)))
        tr.close()
    (la, ea), (lb, eb) = traces
    print("captured", la, "\neager   ", lb, "\ndrops", (ea == -1).astype(int).tolist())
    assert np.isfinite(la).all()
    assert np.array_equal(ea, eb)
    assert 10 < (ea == -1).sum() < 40  # column 2 always, the others at p
    assert np.abs(la - lb).max() <= 1e-3 * np.abs(lb).max()


# ------------------------------------------------------------------------------------------------------------ sampling
B_S, SHAPE = 2, (2, 3, 64, 64)
Y = np.array([3, 7], np.int32)


@pytest.fixture(scope="module")
def guided(ub, oracle):
    O = oracle
    cfg, flat = _oracle_model(O)
    P = O.unflatten_params(cfg, flat)
    tr = ub.Trainer(B=B_S, num_classes=K, class_dropout=0.1)
    tr.set_params(flat.numpy())
    tr.set_labels(Y)
    yield O, cfg, flat, P, tr
    tr.close()


def _guided_fn(O, cfg, P, s, learned=False):
    """The oracle's guided model: eps_u + s (eps_c - eps_u) from two unet_forward calls; a learned-variance model's v
    comes from the conditional pass."""
    yc, yu = torch.from_numpy(Y).long(), torch.full((B_S,), K, dtype=torch.long)

    def fn(x, t):
        tt = torch.full((x.shape[0], 1), float(t))
        oc, ou = O.unet_forward(cfg, P, x, tt, yc), O.unet_forward(cfg, P, x, tt, yu)
        eps = ou[:, :3] + s * (oc[:, :3] - ou[:, :3])
        return torch.cat([eps, oc[:, 3:]], 1) if learned else eps
    return fn


def _draws(n, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*SHAPE, generator=g) * scale
    return x, [torch.randn(*SHAPE, generator=g) for _ in range(n)]


def _launches(ub, fn):
    L = ub.lib()
    n0 = L.ub_launch_count()
    r = fn()
    return r, L.ub_launch_count() - n0


@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("sampler,eta,spec", [("ddim", 0.0, "ddim10"), ("ddim", 1.0, "ddim10"),
                                              ("ancestral", 0.0, "250")])
def test_three_iterations_match_oracle(ub, guided, sampler, eta, spec, clip):
    O, cfg, _, P, tr = guided
    ts = ub.space_timesteps(1000, spec)[:3]
    x, noises = _draws(3, 31, scale=3.0)
    tr.set_guidance(3.0)
    ref = SO.spaced_sample(_guided_fn(O, cfg, P, 3.0), x, ts, sampler, eta, clip, noises).numpy()
    out = tr.sample_spaced(x.numpy(), ts, sampler, eta, clip, torch.stack(noises).numpy())
    tr.set_guidance(1.0)
    err = np.abs(out - ref).max() / np.abs(ref).max()
    print(f"guided s = 3, {sampler} eta {eta} clip {clip}: max-abs / max|ref| {err:.3e}")
    assert err <= TOL_PARITY


def test_full_ddim10_matches_oracle(ub, guided):
    O, cfg, _, P, tr = guided
    ts = ub.space_timesteps(1000, "ddim10")
    x, noises = _draws(10, 32)
    tr.set_guidance(3.0)
    ref = SO.spaced_sample(_guided_fn(O, cfg, P, 3.0), x, ts, "ddim", 0.0, True, noises).numpy()
    out = tr.sample_spaced(x.numpy(), ts, "ddim", 0.0, True, torch.stack(noises).numpy())
    tr.set_guidance(1.0)
    rel = float(np.linalg.norm(out - ref) / np.linalg.norm(ref))
    print(f"guided s = 3 ddim10 full run: relative L2 {rel:.3e}, max-abs/max|ref| "
          f"{np.abs(out - ref).max() / np.abs(ref).max():.3e}")
    assert rel <= TOL_FULL_L2


def test_scale_changes_without_recapture(ub, guided):
    O, cfg, _, P, tr = guided
    ts = ub.space_timesteps(1000, "ddim10")[:3]
    x, noises = _draws(3, 33, scale=3.0)
    counts, outs, errs = [], [], []
    for s in (3.0, 1.5, 2.0):
        tr.set_guidance(s)
        out, n = _launches(ub, lambda: tr.sample_spaced(x.numpy(), ts, "ddim", 1.0, True, torch.stack(noises).numpy()))
        ref = SO.spaced_sample(_guided_fn(O, cfg, P, s), x, ts, "ddim", 1.0, True, noises).numpy()
        err = np.abs(out - ref).max() / np.abs(ref).max()
        print(f"s = {s}: max-abs / max|ref| {err:.3e}, {n} launches")
        assert err <= TOL_PARITY, (s, err)
        counts.append(n), outs.append(out), errs.append(err * np.abs(ref).max())
    tr.set_guidance(1.0)
    assert counts[0] == counts[1] == counts[2]
    assert np.abs(outs[0] - outs[1]).max() > 3 * max(errs)  # the scale reaches the graph
    cond, n1 = _launches(ub, lambda: tr.sample_spaced(x.numpy(), ts, "ddim", 1.0, True, torch.stack(noises).numpy()))
    assert np.abs(cond - outs[0]).max() > 3 * max(errs)
    # per iteration the guided graph adds one forward tape and one label launch to the unguided one, whose other three
    # launches are the timestep fill and the sampler step (with its counter increment)
    assert counts[0] - n1 == n1 - 3 * 3


def test_learned_range_ancestral_matches_oracle(ub, oracle):
    O = oracle
    cfg, flat = _oracle_model(O, dict(out_channels=6), v_scale=0.1)
    P = O.unflatten_params(cfg, flat)
    tr = ub.Trainer(B=B_S, num_classes=K, class_dropout=0.1, learn_sigma=1)
    tr.set_params(flat.numpy())
    tr.set_labels(Y)
    tr.set_guidance(3.0)
    ts = ub.space_timesteps(1000, "250")[:3]
    x, noises = _draws(3, 34, scale=3.0)
    ref = LS.p_sample_loop(_guided_fn(O, cfg, P, 3.0, learned=True), x, ts, True, noises).numpy()
    out = tr.sample_spaced(x.numpy(), ts, "ancestral", 0.0, True, torch.stack(noises).numpy())
    rel = float(np.linalg.norm(out - ref) / np.linalg.norm(ref))
    print(f"guided learned-range ancestral: relative L2 {rel:.3e}, max-abs/max|ref| "
          f"{np.abs(out - ref).max() / np.abs(ref).max():.3e}")
    assert rel <= TOL_FULL_L2
    tr.close()


# ---------------------------------------------------------------------------------------------------------- identities
def test_scale_one_is_the_unguided_call(ub, oracle):
    O = oracle
    _, flat = _oracle_model(O)
    ts = ub.space_timesteps(1000, "ddim10")[:3]
    x, noises = _draws(3, 35, scale=3.0)
    trs = [ub.Trainer(B=B_S, num_classes=K, class_dropout=0.1) for _ in range(2)]
    res = []
    for i, tr in enumerate(trs):
        tr.set_params(flat.numpy())
        tr.set_labels(Y)
        if i:
            tr.set_guidance(3.0)
            tr.sample_spaced(x.numpy(), ts, "ddim", 0.0, True, torch.stack(noises).numpy())
            tr.set_guidance(1.0)
        res.append(_launches(ub, lambda: tr.sample_spaced(x.numpy(), ts, "ddim", 0.0, True,
                                                          torch.stack(noises).numpy())))
    (a, na), (b, nb) = res
    assert na == nb
    assert np.abs(a - b).max() < TOL_RUNS
    for tr in trs:
        tr.close()


def test_scale_zero_is_unconditional(ub, guided):
    _, _, _, _, tr = guided
    ts = ub.space_timesteps(1000, "ddim10")[:3]
    x, noises = _draws(3, 36)
    run = lambda: tr.sample_spaced(x.numpy(), ts, "ddim", 1.0, True, torch.stack(noises).numpy())
    tr.set_guidance(0.0)
    a = run()
    tr.set_guidance(1.0)
    tr.set_labels([-1, -1])
    b = run()
    tr.set_labels(Y)
    c = run()
    print(f"s = 0 against labels -1: max-abs {np.abs(a - b).max():.3e}; against the labels: {np.abs(a - c).max():.3e}")
    assert np.abs(a - b).max() < TOL_RUNS
    assert np.abs(a - c).max() > 3 * np.abs(a - b).max()


def test_checkpoint_is_a_plain_k_plus_one_class_model(ub, oracle, tmp_path):
    O = oracle
    cfg, flat = _oracle_model(O)
    tr = ub.Trainer(B=B_S, num_classes=K, class_dropout=0.1)
    tr.set_params(flat.numpy())
    path = str(tmp_path / "cfg.bin")
    tr.save(path, with_adamw=True)
    plain = ub.Trainer(B=B_S, num_classes=K + 1)
    plain.load(path)
    np.testing.assert_array_equal(plain.get_params(), flat.numpy())
    x0, t, noise = O.synthetic_batch(cfg, B_S)
    xt = O.q_sample(x0, t, noise).numpy()
    tr.set_labels([-1, 4])
    plain.set_labels([K, 4])
    a, b = tr.predict(xt, t.numpy()), plain.predict(xt, t.numpy())
    assert np.abs(a - b).max() <= TOL_RUNS * np.abs(b).max()
    with torch.no_grad():
        ref = O.unet_forward(cfg, O.unflatten_params(cfg, flat), torch.from_numpy(xt), t, torch.tensor([K, 4])).numpy()
    assert np.abs(a - ref).max() <= 3e-2 * np.abs(ref).max()
    # predict stays unguided whatever the scale
    tr.set_guidance(4.0)
    c = tr.predict(xt, t.numpy())
    assert np.abs(a - c).max() <= TOL_RUNS * np.abs(a).max()
    tr.close(), plain.close()


# --------------------------------------------------------------------------------------------------------------- state
def test_guided_sampling_leaves_training_state_untouched(ub, oracle, tmp_path):
    O = oracle
    cfg, flat = _oracle_model(O)
    x0, t, noise = (a.numpy() for a in O.synthetic_batch(cfg, B_S))
    trs = [ub.Trainer(B=B_S, num_classes=K, class_dropout=0.5, ema_rate=0.999) for _ in range(2)]
    for tr in trs:
        tr.set_params(flat.numpy())
        tr.set_labels(Y)
        tr.train_step(x0, t, noise, lr=1e-4)
    tr, ref = trs
    tr.save(str(tmp_path / "before.bin"), with_adamw=True)
    ema = tr.get_ema()
    eff = tr.get_effective_labels()
    x, noises = _draws(3, 37)
    tr.set_guidance(3.0)
    tr.sample_spaced(x.numpy(), ub.space_timesteps(1000, "ddim10"), "ddim", 1.0, True, None, seed=4)
    tr.sample_spaced(x.numpy(), ub.space_timesteps(1000, "250")[:3], "ancestral", 0.0, False,
                     torch.stack(noises).numpy())
    tr.set_guidance(1.0)
    tr.save(str(tmp_path / "after.bin"), with_adamw=True)
    assert (tmp_path / "before.bin").read_bytes() == (tmp_path / "after.bin").read_bytes()
    assert np.array_equal(tr.get_ema(), ema)
    assert np.array_equal(tr.get_effective_labels(), eff)  # sampling leaves the last training step's labels
    la = tr.train_step(x0, t, noise, lr=1e-4)
    lb = ref.train_step(x0, t, noise, lr=1e-4)
    assert np.array_equal(tr.get_effective_labels(), ref.get_effective_labels())
    assert abs(la - lb) <= 1e-3 * abs(lb), (la, lb)
    for tr in trs:
        tr.close()


# ---------------------------------------------------------------------------------------------------------- rejections
def test_rejections(ub, guided):
    L = ub.lib()
    _, _, _, _, tr = guided
    STATE, SHAPE_ = -4, -1
    plain = ub.Trainer(B=B_S, num_classes=K)
    assert L.ub_trainer_set_guidance(plain._h, 2.0) == STATE
    assert b"class_dropout" in L.ub_last_error()
    assert L.ub_trainer_set_guidance(plain._h, 1.0) == STATE
    out = np.zeros(B_S, np.int32)
    assert L.ub_trainer_get_effective_labels(plain._h, out.ctypes.data_as(C.c_void_p), B_S) == STATE
    for bad in ([-1, 3], [0, K]):  # a plain class-conditional trainer refuses -1 as before
        with pytest.raises(ub.UbError, match=rf"outside \[0, {K}\)"):
            plain.set_labels(bad)
    plain.close()
    for s in (float("nan"), float("inf"), -float("inf"), -0.5):
        assert L.ub_trainer_set_guidance(tr._h, s) == SHAPE_, s
        assert b"guidance scale" in L.ub_last_error()
    for bad in ([-2, 3], [0, K], [K + 5, 1]):
        with pytest.raises(ub.UbError, match=rf"outside \[-1, {K}\)"):
            tr.set_labels(bad)
    assert L.ub_trainer_get_effective_labels(tr._h, out.ctypes.data_as(C.c_void_p), B_S + 1) == SHAPE_
    img = np.zeros(SHAPE, np.float32)
    tr.set_guidance(2.0)
    assert L.ub_trainer_sample(tr._h, ub._ptr(img), 40, 38, None, 0, ub._ptr(img)) == STATE
    assert b"guidance" in L.ub_last_error()
    tr.set_guidance(1.0)
    assert L.ub_trainer_sample(tr._h, ub._ptr(img), 40, 38, None, 0, ub._ptr(img)) == 0
    tr.set_labels(Y)
