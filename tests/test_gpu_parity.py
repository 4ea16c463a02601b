"""GPU parity tests proper: the CUDA path (through the public API and the C ABI) against
  (1) the committed golden vectors of the unmodified reference (fp32 and fp64),
  (2) the CPU oracle on the same seeded inputs, stage by stage (so a mismatch is localised),
  (3) size-independent properties at BASELINE.json's full sizes.
Tolerances: conftest.grad_tolerance (policy text there).  Stage-level checks: 1e-5 relative."""
import os

import numpy as np
import pytest
import torch

from conftest import ALL_CASES, BERNOULLI_CASES, BIG_CASES, GOLDEN_DIR, TINY_CASES, load_golden, grad_tolerance
from engine_layout import geometry, grid_to_nchw, flat_to_nchw, theta_to_ref, rel_err
from oracle import maml_oracle as O

pytestmark = pytest.mark.gpu


def _model(g, device):
    from howtotrainyourmamlpytorch_b200 import MAMLFewShotClassifier
    a = g.args
    m = MAMLFewShotClassifier(im_shape=(2, a.image_channels, a.image_height, a.image_width), device=device, args=a)
    m.load_state_dict(g.state())
    return m


def _report(tag, rows):
    print("\n[%s]" % tag)
    for r in rows:
        print("   " + r)


def _count_exact_ties(fwd_blocks):
    """(#pooling windows, #windows whose maximum is attained by >= 2 elements) over the blocks of one oracle pass."""
    import torch.nn.functional as Fnn
    nwin, nties = 0, 0
    for blk in fwd_blocks:
        y = blk["y"]
        act = torch.where(y > 0, y, 0.01 * y)
        n_, c_, hh, ww = act.shape
        win = Fnn.unfold(act.reshape(n_ * c_, 1, hh, ww), kernel_size=2, stride=2)      # [n*c, 4, windows]
        mx = win.max(dim=1, keepdim=True).values
        nwin += win.shape[0] * win.shape[2]
        nties += int(((win == mx).sum(dim=1) >= 2).sum())
    return nwin, nties


@pytest.mark.parametrize("case", ["tiny_pp", "tiny_maml", "tiny_odd", "tiny_bern"])
def test_stagewise_against_oracle(case, cuda_device):
    """Every materialised intermediate of task 0 against the autograd-free oracle, evaluated in fp64.  ``tiny_bern``
    runs Bernoulli(0.93) binary images (the distribution bench.py uses): thousands of pooling windows with EXACT ties,
    which F.max_pool2d resolves first-max-wins -- a tie resolved differently routes the gradient to another pixel and
    shows up as an O(1) error in dz / dp of that block.  The oracle runs in fp64: on ``tiny_bern`` its fp32
    evaluation is itself farther from exact than these tolerances (up to 4e-5 of max-norm on the inner-loop weights,
    varying with the host's CPU thread count, and one near-tie resolved the other way, which moves a final gradient by
    4e-3 of max-norm), while the engine sits within 0.3x of these tolerances of the fp64 values on every case
    (measured on a B200)."""
    g = load_golden(case)
    a = g.args
    m = _model(g, cuda_device)
    batch = g.batch(0)
    epoch = g.iters[0][0]
    losses, preds, grads = m.meta_gradient(batch, epoch)
    eng = m._engine
    ref = O.manual_train_iter(g.state(torch.float64), a, batch, epoch, keep_intermediates=True)
    inter = [x for x in ref["intermediates"] if "theta" in x and x["task"] == 0][0]
    tang = {x["step"]: x for x in ref["intermediates"] if "Hu" in x and x["task"] == 0}
    geo, (ph, pw) = geometry(a)
    F = int(a.cnn_num_filters)
    n_s = int(a.num_classes_per_set) * int(a.num_samples_per_class)
    S = int(a.number_of_training_steps_per_iter)
    L = len(geo)
    rows, worst = [], 0.0

    def chk(name, got, want, tol=1e-5, absolute=None):
        nonlocal worst
        e = rel_err(got, want) if absolute is None else float((got.double() - want.double()).abs().max())
        rows.append("%-34s %.2e%s" % (name, e, "" if (e <= (tol if absolute is None else absolute)) else "   <-- FAIL"))
        if absolute is None:
            worst = max(worst, e / tol)
        else:
            worst = max(worst, e / absolute)

    for s in range(S):
        th = theta_to_ref(eng.debug_read("theta", 0, s, 0), a)
        for n, v in inter["theta"][s].items():
            if "conv.bias" in n:
                chk("theta[%d] %s" % (s, n[-22:]), th[n], v, absolute=1e-5)
            else:
                chk("theta[%d] %s" % (s, n[-22:]), th[n], v)
        fwd = inter["sup_f"][s]
        for l in range(L):
            gl = geo[l]
            zh = grid_to_nchw(eng.debug_read("sup_zh", 0, s, l), n_s, gl["h"], gl["w"], F)
            chk("sup zh   s%d l%d" % (s, l), zh, fwd["blocks"][l]["zh"], tol=2e-5)
            if l + 1 < L:
                p = grid_to_nchw(eng.debug_read("sup_ain", 0, s, l + 1), n_s, gl["h"] // 2, gl["w"] // 2, F)
            else:
                p = flat_to_nchw(eng.debug_read("sup_ain", 0, s, L), n_s, ph, pw, F)
            chk("sup pool s%d l%d" % (s, l), p, fwd["blocks"][l]["p"], tol=2e-5)
        bwd = inter["sup_b"][s]
        for l in reversed(range(L)):
            gl = geo[l]
            if l + 1 < L:
                dp = grid_to_nchw(eng.debug_read("sup_dp", 0, s, l), n_s, gl["h"] // 2, gl["w"] // 2, F)
            else:
                dp = flat_to_nchw(eng.debug_read("sup_dp", 0, s, l), n_s, ph, pw, F)
            chk("sup dp   s%d l%d" % (s, l), dp, bwd["blocks"][l]["dp"], tol=5e-5)
            dz = grid_to_nchw(eng.debug_read("sup_dz", 0, s, l), n_s, gl["h"], gl["w"], F)
            chk("sup dz   s%d l%d" % (s, l), dz, bwd["blocks"][l]["dz"], tol=5e-5)
        gg = theta_to_ref(eng.debug_read("g", 0, s, 0), a)
        for n, v in inter["sup_g"][s].items():
            if "conv.bias" in n:
                chk("g[%d] %s" % (s, n[-22:]), gg[n], v, absolute=1e-5)
            elif "linear.bias" in n:
                # sum_rows (softmax - onehot): cancels to ~1e-2 of its terms, so fp32 rounding shows up larger
                chk("g[%d] %s" % (s, n[-22:]), gg[n], v, tol=2e-4)
            else:
                chk("g[%d] %s" % (s, n[-22:]), gg[n], v, tol=5e-5)
    if case in BERNOULLI_CASES:
        nwin, nties = 0, 0
        for s in range(S):
            w_, t_ = _count_exact_ties(inter["sup_f"][s]["blocks"])
            nwin += w_; nties += t_
        rows.append("pooling windows with an exact tie (oracle, task 0 support passes): %d of %d -- resolved like "
                    "F.max_pool2d iff the dz / dp rows above agree" % (nties, nwin))
        assert nties > 100, "the Bernoulli case is supposed to exercise exact pooling ties"
    _report(case + " stagewise", rows)
    # final outputs
    assert abs(float(losses["loss"]) - float(ref["loss"])) <= 2e-5 * abs(float(ref["loss"]))
    for n, v in ref["grads"].items():
        e = float((grads[n].cpu().double() - v.double()).abs().max())
        tol = 1e-5 if ("conv.bias" in n or "conv-bias" in n) else 2e-4 * float(v.abs().max()) + 1e-7
        assert e <= tol, ("final grad", n, e, tol)
    assert worst <= 1.0, "stage mismatch (see report above): worst = %.2f x tolerance" % worst


@pytest.mark.parametrize("case", ALL_CASES)
def test_golden_reference_parity(case, cuda_device):
    """Loss, logits, accuracy and every outer gradient vs the unmodified reference (golden fixtures)."""
    g = load_golden(case)
    m = _model(g, cuda_device)
    losses, preds, grads = m.meta_gradient(g.batch(0), g.iters[0][0])
    # Full-size cases: tie-breaking chaos (conftest.grad_tolerance) makes the direct comparison loose by nature; the
    # tight statement for them is test_decision_forced_parity.  Tiny cases stay on the tight fp32 bounds so that a
    # regression in the un-pinned path is visible.
    big = case in BIG_CASES
    # tiny_odd carries one pooling near-tie (margin below an fp32 ulp of the pre-activation): which element wins depends
    # on the summation order of the kernels in use, and a flip moves every gradient by ~1e-4 of its max-norm -- seen with
    # the tensor-core convs in round 1 and again with the tensor-core weight gradient.  Flip-level bound for that case.
    flip_rel = 5e-4 if case == "tiny_odd" else None
    ref_loss32, ref_loss64 = g.scalar("loss"), g.scalar("loss64")
    ltol = max(3 * abs(ref_loss32 - ref_loss64), (5e-3 if big else 2e-5) * abs(ref_loss64))
    assert abs(float(losses["loss"]) - ref_loss64) <= ltol, (float(losses["loss"]), ref_loss32, ref_loss64)
    ref_logits = torch.from_numpy(g.array("logits"))
    got_logits = torch.from_numpy(np.stack(preds))
    assert got_logits.shape == ref_logits.shape
    assert float((got_logits - ref_logits).abs().max()) <= (0.25 if big else 1e-3) * float(ref_logits.abs().max())
    g32, g64 = g.grads(0, ""), g.grads(0, "64")
    if case in BERNOULLI_CASES and not big:
        # Binary images: a third of the pooling windows hold EXACT ties (resolved first-max-wins; the stage-wise test
        # checks that against the oracle) and many more hold near-ties, which fp64 / another summation order resolve
        # differently: the reference's own fp32-vs-fp64 distance is ~1e-3 of max-norm here.  The engine has to sit as
        # close to the fp32 reference as the fp64 reference does (3x), not closer.
        for n in g32:
            if "conv.bias" in n or "conv-bias" in n:
                continue
            e32 = float((grads[n].cpu().double() - g32[n].double()).abs().max())
            own = float((g32[n].double() - g64[n].double()).abs().max())
            assert e32 <= max(3.0 * own, 2e-5 * float(g32[n].abs().max())) + 1e-7, ("fp32-anchored (near-ties)", n, e32, own)
    rows, bad = [], []
    for n in g64:
        got = grads[n].cpu().double()
        err = float((got - g64[n].double()).abs().max())
        tol = grad_tolerance(n, g32[n], g64[n], big=big)
        scale = max(float(g64[n].abs().max()), 1e-30)
        if flip_rel is not None and not ("conv.bias" in n or "conv-bias" in n):
            tol = max(tol, flip_rel * scale)
        rows.append("%-78s err %.2e (%.1e of max)  tol %.2e  ref32-vs-64 %.2e" %
                    (n, err, err / scale, tol, float((g32[n].double() - g64[n].double()).abs().max())))
        if err > tol:
            bad.append(n)
    _report(case + " golden parity (loss %.7f, ref32 %.7f, ref64 %.7f)" % (float(losses["loss"]), ref_loss32, ref_loss64), rows)
    assert not bad, bad
    assert abs(losses["accuracy"] - g.scalar("accuracy")) <= (0.051 if case in BIG_CASES else 1e-6)
    w = g.array("msl")
    for i in range(len(w)):
        assert abs(float(losses["loss_importance_vector_%d" % i]) - w[i]) < 1e-7


@pytest.mark.parametrize("case", TINY_CASES)
def test_train_iterations_post_state(case, cuda_device):
    """run_train_iter (H2D, fwd/bwd, clamp + Adam, running-stat EMA) over the recorded iterations: the
    post-step state_dict must match the reference's."""
    g = load_golden(case)
    m = _model(g, cuda_device)
    for it, (epoch, _) in enumerate(g.iters):
        losses, preds = m.run_train_iter(g.batch(it), epoch)
        # later iterations start from OUR post-Adam weights: Adam's first steps move every weight by ~lr whatever the
        # gradient's size, so noise-level gradient elements move differently (see below) -- on the binary-image case,
        # whose near-ties amplify that, the next loss agrees to ~1e-3 only
        ltol = 1e-4 if (it == 0 or case not in BERNOULLI_CASES) else 2e-3
        assert abs(float(losses["loss"]) - g.scalar("loss", it)) <= ltol * abs(g.scalar("loss", it))
        assert abs(float(losses["learning_rate"]) - g.scalar("learning_rate", it)) <= 1e-9
        if it >= 1 and case in BERNOULLI_CASES:
            continue          # binary images: the chaos of iteration 0's near-ties has gone through Adam; the loss check above is the statement
        post = g.post(it)
        sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
        assert list(sd.keys()) == list(post.keys())
        for k in post:
            if "conv.bias" in k or "conv-bias" in k:
                continue   # dead parameter: the reference's update is pure rounding noise through Adam
            if "running" in k:
                assert torch.allclose(sd[k], post[k], rtol=1e-4, atol=1e-5), (it, k, float((sd[k] - post[k]).abs().max()))
            else:
                # Adam's first steps move every weight by ~lr * g/(|g|+1e-8): an element whose gradient is
                # ~1e-8 (noise level) may legitimately move differently; everything else must agree.
                diff = (sd[k] - post[k]).abs()
                frac_bad = float((diff > 2e-5).float().mean())
                assert frac_bad <= 2e-3 and float(diff.max()) <= 2.5e-3, (it, k, frac_bad, float(diff.max()))
        # The conv biases are dead parameters (BatchNorm removes them; true gradient 0): Adam turns the
        # reference's rounding noise into +-lr steps.  They do shift the batch MEAN that the running
        # statistics record, so adopt the reference's values before the next iteration.
        with torch.no_grad():
            for k, p in m.named_parameters():
                if "conv.bias" in k:
                    p.copy_(post[k].to(p.device))


@pytest.mark.parametrize("case", ["tiny_pp", "tiny_maml", "tiny_bern", "omniglot_mamlpp_5w1s", "omniglot_mamlpp_5w1s_bernoulli"])
def test_validation_iter(case, cuda_device):
    """run_validation_iter against the reference's own run_validation_iter (golden val/ entries): loss, accuracy,
    last-step logits, AND the state afterwards -- parameters untouched, running statistics mutated exactly like the
    reference's (its evaluation backup is an alias, meta_neural_network_architectures.py:240-255)."""
    g = load_golden(case)
    m = _model(g, cuda_device)
    m.current_epoch = g.iters[0][0]
    before = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    losses, preds = m.run_validation_iter(g.batch(0))
    big = case in BIG_CASES
    tol = 1e-3 if big else 2e-5
    ref_loss = float(g.val("loss"))
    assert abs(float(losses["loss"]) - ref_loss) <= tol * abs(ref_loss), (float(losses["loss"]), ref_loss)
    ref_logits = torch.from_numpy(g.val("logits"))
    got = torch.from_numpy(np.stack(preds))
    assert got.shape == ref_logits.shape
    assert float((got - ref_logits).abs().max()) <= 10 * tol * float(ref_logits.abs().max())
    assert abs(float(losses["accuracy"]) - float(g.val("accuracy"))) <= (0.051 if big else 1e-6)
    after = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    post = g.val_post()
    for k in before:
        if "running" in k:
            # step 0 statistics depend on the meta-parameters only: tight.  Later steps see the ADAPTED weights; on the
            # full-size cases (binary images above all) those carry tie-breaking chaos of ~1e-3 relative.
            a0, p0 = (after[k][:1], post[k][:1]) if (big and after[k].dim() == 2) else (after[k], post[k])
            assert torch.allclose(a0, p0, rtol=1e-4, atol=1e-5), (k, float((a0 - p0).abs().max()))
            if big:
                assert torch.allclose(after[k], post[k], rtol=2e-2, atol=5e-3), (k, float((after[k] - post[k]).abs().max()))
        else:
            assert torch.equal(before[k], after[k]), "validation must not change %s" % k
    if g.args.per_step_bn_statistics:
        assert any(not torch.equal(before[k], post[k]) for k in post), "reference fixture should show the mutation"


def _result_vector(m, batch, epoch, shard=None):
    """Raw result vector of one engine call (meta-gradient | loss | n_correct | running-stat partial sums)."""
    if shard is not None:
        m._shard_override = shard
    try:
        m.meta_gradient(batch, epoch)
    finally:
        m._shard_override = None
    return m._result.detach().double().cpu().clone()


@pytest.mark.parametrize("case,G", [("tiny_pp", 3), ("tiny_odd", 2), ("omniglot_mamlpp_5w1s_bernoulli", 2)])
def test_engine_as_rank_r_of_G_sums_to_single_call(case, G, cuda_device):
    """The N>1 data path of the ENGINE (task_offset > 0, tasks_global > n_tasks: 1/B_global scaling and the
    position-weighted running-statistics partial sums of export_kernel): run the engine as rank r of G, one rank after
    the other on one GPU, sum the G result vectors (= what the all-reduce does) and require the single-call vector."""
    g = load_golden(case)
    batch, epoch = g.batch(0), g.iters[0][0]
    B = batch[0].shape[0]
    assert B % G == 0
    Bl = B // G
    m = _model(g, cuda_device)
    full = _result_vector(m, batch, epoch)
    acc = torch.zeros_like(full)
    for r in range(G):
        mr = _model(g, cuda_device)
        # same workspace capacity as the single-call engine: split-K / wgrad chunk plans are made for the handle's
        # max_tasks, so a task's arithmetic is then bit-identical in both runs and only the export scaling differs
        mr._ensure_engine(B)
        shard = tuple(t[r * Bl:(r + 1) * Bl].contiguous() for t in batch)
        acc += _result_vector(mr, shard, epoch, shard=(r, G))
    ms = m._engine.meta_size
    segs = m._engine.segments
    for (off, size), name in zip(segs, m._order):
        a, b = acc[off:off + size], full[off:off + size]
        if "conv.bias" in name or "conv-bias" in name:
            assert float((a - b).abs().max()) <= 1e-5, name
        else:
            assert float((a - b).abs().max()) <= 2e-6 * float(b.abs().max()) + 1e-9, (name, float((a - b).abs().max()), float(b.abs().max()))
    assert abs(float(acc[ms] - full[ms])) <= 1e-6 * abs(float(full[ms]))          # loss
    assert float(acc[ms + 1]) == float(full[ms + 1])                              # number of correct predictions
    tail_a, tail_b = acc[ms + 2:], full[ms + 2:]
    if tail_b.numel():
        assert float((tail_a - tail_b).abs().max()) <= 1e-6 * float(tail_b.abs().max()) + 1e-9   # running-stat partial sums


def _two_rank_worker(rank, world, port, case, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    g = load_golden(case)
    m = _model(g, dev)
    B = g.batch(0)[0].shape[0]
    Bl = B // world
    first = None
    for it, (epoch, _) in enumerate(g.iters):
        shard = tuple(t[rank * Bl:(rank + 1) * Bl].contiguous() for t in g.batch(it))
        losses, preds = m.run_train_iter(shard, epoch)
        if first is None:
            first = {"sd": {k: v.detach().cpu().clone() for k, v in m.state_dict().items()},
                     "loss": float(losses["loss"]), "acc": float(losses["accuracy"])}
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    torch.save({"sd": sd, "first": first, "mode": m.collective_desc()["kind"]}, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("case", ["tiny_odd", "tiny_bern"])
def test_two_gpus_equal_one_gpu(case, cuda_device, tmp_path):
    """Two ranks (tasks sharded, ONE all-reduce per iteration: the engine's peer-memory kernel) against one GPU holding
    the whole meta-batch: after the first iteration same loss / accuracy / post-Adam state_dict (Adam's first step moves
    every weight by ~lr whatever the gradient's size, so noise-level gradient elements may move differently -- same
    criterion as test_train_iterations_post_state); after ALL iterations the two replicas are bit-identical."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s_ = socket.socket(); s_.bind(("127.0.0.1", 0)); port = s_.getsockname()[1]; s_.close()
    mp.spawn(_two_rank_worker, args=(2, port, case, str(tmp_path)), nprocs=2, join=True)
    r0 = torch.load(os.path.join(str(tmp_path), "rank0.pt"))
    r1 = torch.load(os.path.join(str(tmp_path), "rank1.pt"))
    g = load_golden(case)
    m = _model(g, cuda_device)
    losses, _ = m.run_train_iter(g.batch(0), g.iters[0][0])
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    print("\n[two ranks] collective:", r0["mode"])
    f0 = r0["first"]
    assert abs(f0["loss"] - float(losses["loss"])) <= 1e-5 * abs(float(losses["loss"]))
    assert abs(f0["acc"] - float(losses["accuracy"])) <= 1e-9
    for k in sd:
        assert torch.equal(r0["sd"][k], r1["sd"][k]), ("replicas diverged", k)
        if "conv.bias" in k or "conv-bias" in k:
            continue
        diff = (f0["sd"][k] - sd[k]).abs()
        if "running" in k:
            assert torch.allclose(f0["sd"][k], sd[k], rtol=1e-4, atol=1e-5), (k, float(diff.max()))
        else:
            frac_bad = float((diff > 2e-5).float().mean())
            assert frac_bad <= 2e-3 and float(diff.max()) <= 2.5e-3, (k, frac_bad, float(diff.max()))


def test_properties_full_size(cuda_device):
    """BASELINE configs[1] at full size (Omniglot MAML++ 5w1s, B=8): size-independent properties.
    (a) run-to-run reproducible; (b) the batch result is the mean of the single-task results (tasks are
    independent and the meta-gradient is linear in them); (c) task order does not matter."""
    from howtotrainyourmamlpytorch_b200 import MAMLFewShotClassifier, make_args, synthetic_batch
    a = make_args("omniglot_mamlpp_5w1s")
    m = MAMLFewShotClassifier(im_shape=(2, 1, 28, 28), device=cuda_device, args=a)
    batch = synthetic_batch(a, iteration=3, kind="normal")
    l1, p1, g1 = m.meta_gradient(batch, 0)
    l2, p2, g2 = m.meta_gradient(batch, 0)
    for n in g1:
        assert rel_err(g2[n], g1[n]) <= 1e-6, ("reproducibility", n)
    acc = {n: torch.zeros_like(v) for n, v in g1.items()}
    loss = 0.0
    B = batch[0].shape[0]
    for b in range(B):
        one = tuple(t[b:b + 1].contiguous() for t in batch)
        lb, pb, gb = m.meta_gradient(one, 0)
        loss += float(lb["loss"]) / B
        for n in acc:
            acc[n] += gb[n] / B
        assert np.allclose(pb[0], p1[b], rtol=1e-4, atol=1e-5)
    assert abs(loss - float(l1["loss"])) <= 1e-5 * abs(loss)
    for n in acc:
        if "conv.bias" in n or "conv-bias" in n:
            continue
        assert rel_err(g1[n], acc[n]) <= 1e-5, ("linearity in tasks", n, rel_err(g1[n], acc[n]))
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0))
    lp, pp, gp = m.meta_gradient(tuple(t[perm].contiguous() for t in batch), 0)
    for n in g1:
        if "conv.bias" in n or "conv-bias" in n:
            continue
        assert rel_err(gp[n], g1[n]) <= 1e-5, ("task permutation", n)
    assert np.isfinite(float(l1["loss"]))


def _gpu_decisions(m, g, batch, epoch):
    """The discrete decisions the GPU actually took (leaky-ReLU branch per element, arg-max per pooling
    window), reconstructed bit-exactly from the engine's normalised activations zh:
    y = fmaf(gamma, zh, beta) (exact product + one rounding == fp64 evaluation rounded to fp32),
    a = y > 0 ? y : 0.01f * y (fp32), first-max-wins in window order (what F.max_pool2d does on CPU)."""
    import torch.nn.functional as Fnn
    a = g.args
    eng = m._engine
    geo, _ = geometry(a)
    F = int(a.cnn_num_filters)
    N, K, T = int(a.num_classes_per_set), int(a.num_samples_per_class), int(a.num_target_samples)
    S = int(a.number_of_training_steps_per_iter)
    B = batch[0].shape[0]
    sched = O.target_pass_schedule(a, epoch, True, S)
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    dec = {}
    for b in range(B):
        for s in range(S):
            for kind, n in (("sup", N * K), ("tgt", N * T)):
                if kind == "tgt" and sched[s] is None:
                    continue
                per_layer = []
                for l, gl in enumerate(geo):
                    zh = grid_to_nchw(eng.debug_read(kind + "_zh", b, s, l), n, gl["h"], gl["w"], F)
                    _, _, gn, btn, _, _ = O.conv_names(l)
                    gam, bet = (sd[gn][s], sd[btn][s]) if a.per_step_bn_statistics else (sd[gn], sd[btn])
                    y = (gam.double()[None, :, None, None] * zh.double() + bet.double()[None, :, None, None]).float()
                    slope = torch.where(y > 0, torch.ones_like(y), torch.full_like(y, 0.01))
                    act = torch.where(y > 0, y, torch.tensor(0.01, dtype=torch.float32) * y)
                    _, idx = Fnn.max_pool2d(act, 2, 2, return_indices=True)
                    per_layer.append((slope, idx))
                dec[(b, kind, s)] = per_layer
    return dec


@pytest.mark.parametrize("case", ALL_CASES)
def test_decision_forced_parity(case, cuda_device):
    """Full-size parity that is immune to tie-breaking chaos.  The network is piecewise smooth: its only
    discontinuities are the leaky-ReLU branch and the pooling arg-max.  We (1) read back the decisions the
    GPU took, (2) check each one is CONSISTENT with exact arithmetic -- it may differ from the fp64 choice
    only where the fp64 margin is below 1e-4 (a genuine near-tie), and (3) evaluate the fp64 oracle with
    those decisions pinned: loss and every meta-gradient tensor must then agree to fp32 rounding
    (1e-4 of the tensor's max-norm; measured ~1e-6..1e-5)."""
    import torch.nn.functional as Fnn
    g = load_golden(case)
    from howtotrainyourmamlpytorch_b200 import MAMLFewShotClassifier
    a = g.args
    m = MAMLFewShotClassifier(im_shape=(2, a.image_channels, a.image_height, a.image_width), device=cuda_device, args=a)
    m._debug_keep_target_passes = True
    m.load_state_dict(g.state())
    batch, epoch = g.batch(0), g.iters[0][0]
    losses, preds, grads = m.meta_gradient(batch, epoch)
    dec = _gpu_decisions(m, g, batch, epoch)
    ref = O.manual_train_iter(g.state(torch.float64), a, batch, epoch, decisions=dec, keep_intermediates=True)
    # (2) consistency of the GPU's decisions with exact arithmetic
    n_slope_flip, n_arg_flip, worst_margin, n_dec = 0, 0, 0.0, 0
    for x in [i for i in ref["intermediates"] if "theta" in i]:
        passes = [f for f in x["sup_f"]] + [t[0] for t in x["tgt_f"] if t is not None]
        for f in passes:
            for blk in f["blocks"]:
                y = blk["y"]
                nat_pos = y > 0
                forced_pos = blk["slope"] > 0.5
                flip = nat_pos != forced_pos
                n_dec += y.numel()
                if flip.any():
                    n_slope_flip += int(flip.sum())
                    worst_margin = max(worst_margin, float(y[flip].abs().max()))
                act = y * torch.where(nat_pos, torch.ones_like(y), torch.full_like(y, 0.01))
                pmax = Fnn.max_pool2d(act, 2, 2)
                n_, c_ = act.shape[:2]
                pforced = act.view(n_, c_, -1).gather(2, blk["idx"].view(n_, c_, -1)).view(pmax.shape)
                gap = pmax - pforced
                if (gap > 0).any():
                    n_arg_flip += int((gap > 0).sum())
                    worst_margin = max(worst_margin, float(gap.max()))
    print("\n[%s] decisions checked: %d, leaky-branch flips vs fp64: %d, arg-max flips: %d, worst fp64 margin at a flip: %.2e"
          % (case, n_dec, n_slope_flip, n_arg_flip, worst_margin))
    # Mini-ImageNet 5-way 5-shot diverges in the inner loop (LR 0.1): by the last steps the fast weights are large and an
    # fp32 rounding difference in theta moves pre-activations by several 1e-4 (any fp32 implementation, the reference's
    # included) -- the consistency margin scales accordingly for that case only
    assert worst_margin <= (1e-3 if case == "mini_imagenet_mamlpp_5w5s" else 1e-4), worst_margin
    # (3) smooth parity with the decisions pinned
    ref_loss = float(ref["loss"])
    assert abs(float(losses["loss"]) - ref_loss) <= 1e-5 * abs(ref_loss), (float(losses["loss"]), ref_loss)
    rows, bad = [], []
    for n, v in ref["grads"].items():
        got = grads[n].cpu().double()
        err = float((got - v).abs().max())
        scale = max(float(v.abs().max()), 1e-30)
        if "conv.bias" in n or "conv-bias" in n:
            # dead parameter (true gradient 0): fp32 cancellation noise, proportional to the live gradients
            tol = 1e-5 * max(1.0, max(float(x.abs().max()) for x in ref["grads"].values()))
        else:
            # Mini-ImageNet 5-way 5-shot: the inner loop diverges at LR 0.1 (loss 29, gradients up to 240; the reference's
            # own fp32 run is 10 % away from its fp64 run).  Rounding differences of the fast weights are amplified step
            # by step (GPU decisions flip at fp64 margins up to 4e-4, see above), and the LSLR gradients -<theta_bar, g>
            # are dot products with heavy cancellation: measured 1.2e-4 of max-norm on the ordinary tensors and 1.2e-3 on
            # one LSLR vector with the 3xTF32 tensor-core weight gradient (2e-5 / 2e-4 with the fp32 FFMA one).
            if case == "mini_imagenet_mamlpp_5w5s":
                tol = (3e-3 if "names_learning_rates" in n else 3e-4) * scale + 1e-7
            else:
                tol = 1e-4 * scale + 1e-7
        rows.append("%-78s err %.2e (%.1e of max)" % (n, err, err / scale))
        if err > tol:
            bad.append((n, err, tol))
    _report(case + " decision-forced parity (loss %.7f vs %.7f)" % (float(losses["loss"]), ref_loss), rows)
    assert not bad, bad
    got_logits = torch.from_numpy(np.stack(preds)).double()
    assert float((got_logits - ref["logits"]).abs().max()) <= 1e-4 * float(ref["logits"].abs().max())


@pytest.mark.parametrize("case", ["tiny_pp", "tiny_odd", "tiny_maml"])
def test_tensor_core_convs_match_fp32_ffma_convs(case, cuda_device):
    """Kernel-level A/B: the tcgen05 3xTF32 implicit-GEMM convolutions against their exact-fp32 FFMA twins
    (`reserved` bit 1) on the same inputs -- every intermediate of the first support forward / backward must
    agree to 2e-5 (no chaos: a single pass has no inner-loop amplification)."""
    from howtotrainyourmamlpytorch_b200 import MAMLFewShotClassifier
    g = load_golden(case)
    a = g.args
    outs = []
    for force in (False, True):
        m = MAMLFewShotClassifier(im_shape=(2, a.image_channels, a.image_height, a.image_width), device=cuda_device, args=a)
        m._debug_force_fp32_convs = force
        m.load_state_dict(g.state())
        m.meta_gradient(g.batch(0), g.iters[0][0])
        eng = m._engine
        L = int(a.num_stages)
        taps = {}
        for l in range(L):
            taps["zh%d" % l] = eng.debug_read("sup_zh", 0, 0, l)
            taps["dz%d" % l] = eng.debug_read("sup_dz", 0, 0, l)
            if l < L - 1:
                taps["dp%d" % l] = eng.debug_read("sup_dp", 0, 0, l)
        taps["g0"] = eng.debug_read("g", 0, 0, 0)
        outs.append(taps)
    for k in outs[0]:
        x, y = torch.from_numpy(outs[0][k]), torch.from_numpy(outs[1][k])
        assert rel_err(x, y) <= 2e-5, (k, rel_err(x, y))


@pytest.mark.parametrize("case", ["tiny_pp", "tiny_maml", "omniglot_mamlpp_5w1s"])
def test_functional_network_operator(case, cuda_device):
    """Level B1: VGGReLUNormNetwork.forward(x, num_step, params) as a stand-alone operator vs the oracle's
    functional forward (F.conv2d / F.batch_norm / F.leaky_relu / F.max_pool2d / F.linear), with external fast weights
    carrying the reference's leading replica dim, and with params=None."""
    g = load_golden(case)
    a = g.args
    m = _model(g, cuda_device)
    xs, xt, ys, yt = g.batch(0)
    x = xt[0].reshape(-1, *xt.shape[-3:])
    state = g.state()
    inner = O.inner_param_names(a)
    gen = torch.Generator().manual_seed(5)
    fast_cpu = {n: state[n] + 0.05 * torch.randn(state[n].shape, generator=gen) for n in inner}
    for step in (0, int(a.number_of_training_steps_per_iter) - 1):
        ref = O._net_forward(x, fast_cpu, state, a, step)
        params = {n[len("classifier."):]: v.to(cuda_device).unsqueeze(0) for n, v in fast_cpu.items()}
        got = m.classifier.forward(x.to(cuda_device), num_step=step, params=params, training=True)
        assert got.shape == ref.shape
        assert float((got.cpu() - ref).abs().max()) <= 2e-5 * float(ref.abs().max()) + 1e-6, (case, step)
    ref0 = O._net_forward(x, {n: state[n] for n in inner}, state, a, 0)
    got0 = m.classifier.forward(x.to(cuda_device), num_step=0)
    assert float((got0.cpu() - ref0).abs().max()) <= 2e-5 * float(ref0.abs().max()) + 1e-6


@pytest.mark.parametrize("case", ["tiny_pp", "tiny_maml", "tiny_bern"])
def test_functional_network_operator_is_differentiable(case, cuda_device):
    """Level B1 used the way the reference uses it (few_shot_learning_system.py:138-139, :265-286): cross-entropy of
    ``classifier.forward(x, params=fast, num_step=s)`` differentiated with ``torch.autograd.grad`` w.r.t. the fast
    weights (leading replica dim included) and w.r.t. the BatchNorm gamma / beta the module owns -- against torch
    autograd through the oracle's functional forward.  Also: the forward leaves F.batch_norm's EMA update behind."""
    import torch.nn.functional as Fnn
    g = load_golden(case)
    a = g.args
    m = _model(g, cuda_device)
    xs, xt, ys, yt = g.batch(0)
    x = xs[0].reshape(-1, *xs.shape[-3:])
    y = ys[0].reshape(-1).long()
    state = g.state()
    inner = O.inner_param_names(a)
    step = min(1, int(a.number_of_training_steps_per_iter) - 1)
    # oracle: autograd through F.conv2d / F.batch_norm / ...
    leaves = {k: v.clone().requires_grad_(k in O.trainable_names(a) and "learning_rates" not in k) for k, v in state.items()}
    fast = {n: leaves[n] for n in inner}
    stats = []
    ref_logits = O._net_forward(x, fast, leaves, a, step, stats)
    ref_loss = Fnn.cross_entropy(ref_logits, y)
    wrt = [n for n, v in leaves.items() if v.requires_grad]
    ref_grads = dict(zip(wrt, torch.autograd.grad(ref_loss, [leaves[n] for n in wrt], allow_unused=True)))
    ref_run = O.apply_running_stats(state, a, stats)
    # engine operator
    params = {n[len("classifier."):]: dict(m.named_parameters())[n].detach().clone().unsqueeze(0).requires_grad_(True) for n in inner}
    before = {k: v.detach().cpu().clone() for k, v in m.state_dict().items() if "running" in k}
    logits = m.classifier.forward(x.to(cuda_device), num_step=step, params=params, training=True,
                                  backup_running_statistics=True)
    loss = Fnn.cross_entropy(logits, y.to(cuda_device))
    assert abs(float(loss) - float(ref_loss)) <= 2e-5 * abs(float(ref_loss))
    bn_params = [(n, p) for n, p in m.named_parameters() if "norm_layer" in n and p.requires_grad]
    got = torch.autograd.grad(loss, list(params.values()) + [p for _, p in bn_params], create_graph=False)
    names = ["classifier." + k for k in params] + [n for n, _ in bn_params]
    rows = []
    for n, gv in zip(names, got):
        r = ref_grads[n]
        gv = gv.detach().cpu().reshape(r.shape)
        if "conv.bias" in n:
            assert float((gv - r).abs().max()) <= 1e-4, n        # dead parameter: true gradient 0, both sides are rounding noise
            continue
        e = rel_err(gv, r)
        rows.append("%-60s %.2e" % (n, e))
        assert e <= 5e-5, (n, e)
    _report(case + " functional operator backward", rows)
    after = {k: v.detach().cpu() for k, v in m.state_dict().items() if "running" in k}
    for k in after:
        assert torch.allclose(after[k], ref_run[k], rtol=5e-5, atol=5e-6), k
    if a.per_step_bn_statistics:
        assert any(not torch.equal(after[k], before[k]) for k in after)
    # a second forward of the same shape before the backward of the first must not corrupt it (replay path)
    l1 = m.classifier.forward(x.to(cuda_device), num_step=step, params=params)
    l2 = m.classifier.forward(xt[0].reshape(-1, *xt.shape[-3:])[:x.shape[0]].to(cuda_device), num_step=step, params=params)
    g1 = torch.autograd.grad(Fnn.cross_entropy(l1, y.to(cuda_device)), list(params.values()))
    for n, gv in zip(names, g1):
        if "conv.bias" in n:
            continue
        assert rel_err(gv.detach().cpu().reshape(ref_grads[n].shape), ref_grads[n]) <= 5e-5, ("replay", n)
    m.classifier.zero_grad(params)
    m.classifier.restore_backup_stats()


def test_fused_and_cluster_paths_match_plain_paths(cuda_device):
    """The scheduling / fusion variants (cluster split-K convs, N-stacked 3xTF32 MMAs, tcgen05 weight gradient, fused
    BatchNorm backward, tangent conv split, double-buffered target passes, fused last block + head) against the plain
    one-kernel-per-op paths (one-tap FFMA wgrad included) they replaced
    (selected through the diagnostic environment switches, read when the engine handle is created)."""
    g = load_golden("tiny_pp")
    batch, epoch = g.batch(0), g.iters[0][0]
    plain = {"MAML_B200_TC_SPLIT": "1", "MAML_B200_BN_FUSE": "0", "MAML_B200_TAN_SPLIT": "0", "MAML_B200_TGT_SLOTS": "1",
             "MAML_B200_WGRAD_ROW": "0", "MAML_B200_TAIL_FUSE": "0", "MAML_B200_WGRAD_TC": "0", "MAML_B200_TC_STACK": "0"}
    saved = {k: os.environ.get(k) for k in plain}
    try:
        os.environ.update(plain)
        m0 = _model(g, cuda_device)
        l0, p0, g0 = m0.meta_gradient(batch, epoch)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    m1 = _model(g, cuda_device)
    l1, p1, g1 = m1.meta_gradient(batch, epoch)
    assert abs(float(l0["loss"]) - float(l1["loss"])) <= 1e-6 * abs(float(l0["loss"]))
    for n in g0:
        if "conv.bias" in n or "conv-bias" in n:
            assert float((g0[n] - g1[n]).abs().max()) <= 1e-5
        else:
            assert rel_err(g1[n], g0[n]) <= 2e-5, (n, rel_err(g1[n], g0[n]))


_POLICY_SWITCHES = [
    {"MAML_B200_PDL": "0"},                                  # no programmatic dependent launch
    {"MAML_B200_PDL": "1", "MAML_B200_PDL_CLUSTER": "3"},    # ... on every stream, cluster launches included
    {"MAML_B200_TC_PUSH": "0"},                              # pull-based split-K reduction (two cluster barriers)
    {"MAML_B200_TC_ZSTAGE": "0"},                            # tangent-mode statistics read the primal zh from global memory
    {"MAML_B200_TAIL_ONCHIP": "0"},                          # last-block kernels that exchange their stages through L2
    {"MAML_B200_TC_NB": "3", "MAML_B200_WG_NSTAGE": "2", "MAML_B200_TC_NB_FIT": "1"},     # shallow shared-memory rings
    {"MAML_B200_TC_SPLIT_SIDE": "1", "MAML_B200_TC_NB_SIDE": "2", "MAML_B200_BN_SIDE_CAP": "16"},   # side-stream caps
]


@pytest.mark.parametrize("case", ["tiny_pp", "tiny_bern"])
@pytest.mark.parametrize("switches", _POLICY_SWITCHES, ids=lambda d: "+".join("%s=%s" % (k[10:], v) for k, v in d.items()))
def test_launch_policy_switches_do_not_change_results(case, switches, cuda_device):
    """Round-2 launch policy (programmatic dependent launch, push-based split-K epilogue, on-chip last-block kernels,
    shared-memory ring depths, side-stream caps): every switch is scheduling only -- the meta-gradient must agree with
    the default build to summation-order noise."""
    g = load_golden(case)
    batch, epoch = g.batch(0), g.iters[0][0]
    m1 = _model(g, cuda_device)
    l1, p1, g1 = m1.meta_gradient(batch, epoch)
    saved = {k: os.environ.get(k) for k in switches}
    try:
        os.environ.update(switches)
        m0 = _model(g, cuda_device)
        l0, p0, g0 = m0.meta_gradient(batch, epoch)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    assert abs(float(l0["loss"]) - float(l1["loss"])) <= 1e-6 * abs(float(l0["loss"]))
    for n in g0:
        if "conv.bias" in n or "conv-bias" in n:
            assert float((g0[n] - g1[n]).abs().max()) <= 1e-5
        else:
            assert rel_err(g1[n], g0[n]) <= 2e-5, (n, rel_err(g1[n], g0[n]))


def test_device_trace(cuda_device):
    """maml_b200_trace: one entry per kernel start of an iteration (also inside the replayed CUDA graph)."""
    g = load_golden("tiny_pp")
    m = _model(g, cuda_device)
    batch, epoch = g.batch(0), g.iters[0][0]
    m.meta_gradient(batch, epoch)
    m.meta_gradient(batch, epoch)                 # second call replays the captured graph
    eng = m._engine
    eng.trace(True)
    m.meta_gradient(batch, epoch)
    tr = eng.trace_read()
    eng.trace(False)
    starts = [t for t, k, tag in tr if not (k & 0x80)]
    assert len(starts) == eng.last_launch_count()
    assert sorted(tag for t, k, tag in tr if not (k & 0x80)) == list(range(len(starts)))     # one entry per graph node
    assert max(starts) - min(starts) < 1e9           # nanoseconds: one tiny iteration spans far less than a second


def test_reference_experiment_builder_drives_the_class(cuda_device, tmp_path):
    """Level B0 as the reference uses it.  ``tests/golden/experiment_builder_tiny_maml.json`` holds every call the
    UNMODIFIED reference ``ExperimentBuilder`` makes on a model (``train_iteration`` with numpy episodes,
    ``evaluation_iteration`` with torch episodes, ``save_models``, and a second builder resuming from ``latest``),
    recorded while it drove the reference's own class (``oracle/gen_golden.py --builder``).  Replayed on THIS repo's
    ``MAMLFewShotClassifier``: the same keyword arguments are accepted, the losses dicts carry the reference's keys and
    values (the builder folds every entry into its summaries with ``float()``), the checkpoints land under the same names
    and ``load_model`` finds them again."""
    import json
    from howtotrainyourmamlpytorch_b200 import MAMLFewShotClassifier
    with open(os.path.join(GOLDEN_DIR, "experiment_builder_tiny_maml.json")) as fh:
        rec = json.load(fh)
    g = load_golden(rec["case"])
    a = g.args
    episodes = g.batch(0)

    def replay(model, call):
        kw = dict(call["kwargs"])
        if "data_batch" in kw:
            assert [list(t.shape) for t in episodes] == [d["shape"] for d in kw["data_batch"]]
            kw["data_batch"] = tuple(t.numpy() if d["type"] == "ndarray" else t for t, d in zip(episodes, kw["data_batch"]))
        if "model_save_dir" in kw:
            kw["model_save_dir"] = os.path.join(str(tmp_path), kw["model_save_dir"])
        if call["method"] == "save_model":
            os.makedirs(os.path.dirname(kw["model_save_dir"]), exist_ok=True)
            kw["state"] = dict(kw["state"])
        return getattr(model, call["method"])(**kw)

    model = _model(g, cuda_device)
    for call in rec["calls"]:
        out = replay(model, call)
        if "losses" not in call:
            continue
        losses, _ = out
        assert sorted(losses) == sorted(call["losses"]), call["method"]
        got, want = {k: float(v) for k, v in losses.items()}, call["losses"]
        train = call["method"] == "run_train_iter"
        # validation runs after the Adam step: noise-level gradient elements move differently through Adam's first step
        # (see test_train_iterations_post_state), so its loss agrees to ~1e-4 and one target prediction may flip
        assert abs(got["loss"] - want["loss"]) <= (1e-4 if train else 1e-3) * abs(want["loss"]), (call["method"], got, want)
        assert abs(got["accuracy"] - want["accuracy"]) <= (1e-6 if train else 0.06), (call["method"], got, want)
        for k in want:
            if k.startswith("loss_importance_vector") or k == "learning_rate":
                assert abs(got[k] - want[k]) <= 1e-7, (k, got[k], want[k])
    saved_dir = os.path.join(str(tmp_path), rec["resume_calls"][0]["kwargs"]["model_save_dir"])
    assert sorted(os.listdir(saved_dir)) == rec["saved_models"]
    m2 = MAMLFewShotClassifier(im_shape=(2, a.image_channels, a.image_height, a.image_width), device=cuda_device, args=a)
    for call in rec["resume_calls"]:
        st = replay(m2, call)
        assert {k: st[k] for k in call["state"]} == call["state"]
    for k, v in model.state_dict().items():
        assert torch.equal(v.cpu(), m2.state_dict()[k].cpu()), k
