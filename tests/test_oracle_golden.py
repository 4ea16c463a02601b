"""CPU: both oracle restatements against the golden vectors generated from the unmodified reference."""
import pytest
import torch

from conftest import ALL_CASES, BIG_CASES, TINY_CASES, load_golden, grad_tolerance
from oracle import maml_oracle as O
from oracle.gen_golden import THREADS as GOLDEN_THREADS


@pytest.fixture(autouse=True)
def _golden_thread_count():
    """Run the oracle with the intra-op thread count the fixtures were generated with.  fp32 CPU convolutions split
    their reductions by thread; on the chaotic full-size cases (Mini-ImageNet at inner LR 0.1, Omniglot 20-way) another
    split moves the fp32 result by more than the tolerances below (measured: 4 or 16 threads fail, 8 pass)."""
    saved = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(saved)


def _check(res, g, suffix, loss_rtol):
    ref_loss = g.scalar("loss" + suffix)
    assert abs(float(res["loss"]) - ref_loss) <= loss_rtol * abs(ref_loss)
    ref = g.grads(0, suffix)
    assert list(res["grads"].keys()) == list(ref.keys())
    g32, g64 = g.grads(0, ""), g.grads(0, "64")
    for n, val in res["grads"].items():
        if suffix == "64":
            tol = 1e-9 * float(ref[n].abs().max()) + 1e-12 if ref[n].dtype == torch.float64 else \
                2e-7 * float(ref[n].abs().max()) + 1e-9          # big cases store fp64 grads cast to fp32
            if "conv.bias" in n or "conv-bias" in n:
                tol = max(tol, 1e-9)
        else:
            tol = grad_tolerance(n, g32[n], g64[n], big=g.case in BIG_CASES)
            ref = g64
        err = float((val.double() - ref[n].double()).abs().max())
        assert err <= tol, (g.case, n, err, tol)


@pytest.mark.parametrize("case", TINY_CASES)
@pytest.mark.parametrize("impl", ["autograd", "manual"])
def test_tiny_fp64_exact(case, impl):
    g = load_golden(case)
    fn = O.autograd_train_iter if impl == "autograd" else O.manual_train_iter
    res = fn(g.state(torch.float64), g.args, g.batch(0), g.iters[0][0])
    _check(res, g, "64", 1e-12)


@pytest.mark.parametrize("case", ALL_CASES)
def test_manual_fp32_within_policy(case):
    g = load_golden(case)
    res = O.manual_train_iter(g.state(torch.float32), g.args, g.batch(0), g.iters[0][0])
    # loss: fp32 rounding, or (chaotic full-size cases: Mini-ImageNet at inner LR 0.1) 3x the reference's own fp32-vs-fp64 distance
    _check(res, g, "", max(2e-6, 3.0 * abs(g.scalar("loss") - g.scalar("loss64")) / abs(g.scalar("loss64")) if g.case in BIG_CASES else 0.0))
    assert abs(res["accuracy"] - g.scalar("accuracy")) < (0.051 if g.case in BIG_CASES else 1e-9)
    ref_logits = torch.from_numpy(g.array("logits"))
    ltol = max(1e-3, 30.0 * abs(g.scalar("loss") - g.scalar("loss64")) / abs(g.scalar("loss64"))) if g.case in BIG_CASES else 1e-4
    assert float((res["logits"] - ref_logits).abs().max()) <= ltol * float(ref_logits.abs().max())
    post = g.post(0)
    chaotic = g.case in BIG_CASES and abs(g.scalar("loss") - g.scalar("loss64")) > 1e-3 * abs(g.scalar("loss64"))
    for k, v in res["running"].items():
        a, b = (v[:1], post[k][:1]) if (chaotic and v.dim() == 2) else (v, post[k])   # diverging inner loop: first step only
        assert torch.allclose(a, b, rtol=1e-3 if g.case in BIG_CASES else 5e-5, atol=1e-4 if g.case in BIG_CASES else 5e-6), k


@pytest.mark.parametrize("case", ALL_CASES)
def test_validation_leg_matches_reference(case):
    """Oracle evaluation pass vs the reference's run_validation_iter (val/ fixtures): loss, logits, accuracy and the
    running statistics the reference leaves behind (its backup/restore is an alias, so they ARE mutated)."""
    g = load_golden(case)
    big = g.case in BIG_CASES
    res = O.autograd_train_iter(g.state(), g.args, g.batch(0), g.iters[0][0], training_phase=False,
                                current_epoch=g.iters[0][0])
    ref_loss = float(g.val("loss"))
    assert abs(float(res["loss"]) - ref_loss) <= 2e-6 * abs(ref_loss)
    ref_logits = torch.from_numpy(g.val("logits"))
    assert float((res["logits"] - ref_logits).abs().max()) <= 1e-5 * float(ref_logits.abs().max())
    assert abs(res["accuracy"] - float(g.val("accuracy"))) < 1e-9
    post = g.val_post()
    assert set(post.keys()) == set(res["running"].keys())
    changed = False
    for k, v in res["running"].items():
        assert torch.allclose(v, post[k], rtol=1e-3 if big else 5e-5, atol=1e-4 if big else 5e-6), k
        changed = changed or not torch.equal(post[k], g.state()[k])
    assert changed == bool(g.args.per_step_bn_statistics)


@pytest.mark.parametrize("case", ["omniglot_mamlpp_5w1s"])
def test_autograd_fp64_big(case):
    g = load_golden(case)
    res = O.autograd_train_iter(g.state(torch.float64), g.args, g.batch(0), g.iters[0][0])
    _check(res, g, "64", 1e-9)


@pytest.mark.parametrize("case", ["tiny_pp", "tiny_maml"])
def test_adam_and_second_iteration(case):
    """Adam restatement reproduces the reference's post-step parameters, and a second iteration
    (fresh batch, Adam state carried) reproduces it1."""
    g = load_golden(case)
    state = g.state()
    names = O.trainable_names(g.args)
    m = {n: torch.zeros_like(state[n]) for n in names}
    v = {n: torch.zeros_like(state[n]) for n in names}
    step = 0
    for it, (epoch, _) in enumerate(g.iters):
        res = O.autograd_train_iter(state, g.args, g.batch(it), epoch)
        clamp = [n for n in names if n.startswith("classifier.")] if "imagenet" in g.args.dataset_name else None
        newp, m, v, step = O.adam_step({n: state[n] for n in names}, res["grads"], m, v, step,
                                       O.cosine_lr(g.args, epoch), clamp=clamp)
        state.update(newp)
        state.update(res["running"])
        post = g.post(it)
        for k in post:
            if "conv.bias" in k or "conv-bias" in k:
                continue      # noise-driven in the reference (dead parameter, true gradient 0)
            assert torch.allclose(state[k], post[k], rtol=2e-4, atol=2e-6), (it, k, float((state[k] - post[k]).abs().max()))
        # keep marching from the reference's own parameters so the 2nd iteration is compared like for like
        state = {k: post[k].clone() for k in post}
