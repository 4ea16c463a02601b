"""ORACLE TOOLING -- TEST INFRASTRUCTURE ONLY.

Generates the golden vectors under ``tests/golden/`` by importing the UNMODIFIED reference
from ``/root/reference`` (a pure-Python/PyTorch program; it runs on CPU in the authoring
container) and running ``MAMLFewShotClassifier.run_train_iter`` on seeded synthetic episodes.

  python oracle/gen_golden.py            # regenerates every case
  python oracle/gen_golden.py tiny_pp    # one case

Each ``tests/golden/<case>.npz`` holds: the args (JSON string), the initial ``state_dict``,
the fp32 reference outputs (loss, accuracy, last-step logits, every outer gradient captured
just before ``optimizer.step``, the post-Adam ``state_dict`` incl. running statistics, the
logged ``learning_rate``), and the fp64 reference loss / gradients (noise-floor anchor for
the tolerance policy, SURVEY.md appendix C).  Inputs are stored only for the tiny cases; the
full-size ones are regenerated from their seed by ``oracle.maml_oracle.synthetic_batch``.

The reference cannot travel to the GPU box (``/root/reference`` does not exist there), so
nothing under ``tests/`` reads it at run time: tests read these fixtures.
"""
import contextlib
import io
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from howtotrainyourmamlpytorch_b200.configs import CONFIGS  # noqa: E402
from howtotrainyourmamlpytorch_b200.utils.parser_utils import args_from_json  # noqa: E402
from oracle import maml_oracle as O  # noqa: E402

REF = "/root/reference"
# intra-op threads of every reference / oracle run in this script: fp32 CPU convolutions split their reductions by
# thread, so the CPU tests that compare the fp32 oracle with these fixtures run with the same count
# (tests/test_oracle_golden.py)
THREADS = 8

_TINY = dict(image_height=20, image_width=20, image_channels=3, cnn_num_filters=16,
             num_classes_per_set=3, num_samples_per_class=2, num_target_samples=2,
             number_of_training_steps_per_iter=3, number_of_evaluation_steps_per_iter=3,
             batch_size=3, total_epochs=100, multi_step_loss_num_epochs=10,
             dataset_name="mini_imagenet_tiny")

# case name -> (base config, overrides, list of (epoch, iteration-seed) train iterations)
# Inputs are N(0,1) unless the case says otherwise (4th tuple entry).  Bernoulli "Omniglot-like" images give
# exact max-pool ties whose resolution is rounding noise, so the reference's own fp32-vs-fp64 gradients differ
# by 10-100 % there (measured; see DESIGN.md "noise floor"): the direct comparison is loose for that case, but
# the decision-forced test (GPU decisions pinned in the fp64 oracle) and the tie statistics ARE meaningful --
# this is the input distribution bench.py runs (BASELINE.md section 4).
KIND = "normal"
CASES = {
    "tiny_pp":        ("mini_imagenet_mamlpp_5w1s", dict(_TINY), [(0, 0), (0, 1)]),
    "tiny_pp_late":   ("mini_imagenet_mamlpp_5w1s", dict(_TINY), [(12, 0)]),
    "tiny_pp_first":  ("mini_imagenet_mamlpp_5w1s", dict(_TINY, second_order=False), [(3, 0)]),
    "tiny_maml":      ("omniglot_maml_5w1s", dict(_TINY, image_channels=1, image_height=16, image_width=16,
                                                  dataset_name="omniglot_tiny"), [(0, 0), (1, 1)]),
    "tiny_odd":       ("omniglot_mamlpp_5w1s", dict(_TINY, image_channels=1, image_height=28, image_width=28,
                                                    cnn_num_filters=32, batch_size=2,
                                                    dataset_name="omniglot_tiny"), [(2, 0)]),
    # Bernoulli(0.93) "Omniglot-like" binary images: exact max-pool ties in every block-0 window whose four receptive
    # fields coincide -- the case first-max-wins exists for (stage-wise GPU test compares dz against the oracle)
    "tiny_bern":      ("omniglot_mamlpp_5w1s", dict(_TINY, image_channels=1, image_height=28, image_width=28,
                                                    cnn_num_filters=32, batch_size=2,
                                                    dataset_name="omniglot_tiny"), [(0, 0), (0, 1)], "bernoulli"),
    "omniglot_mamlpp_5w1s": ("omniglot_mamlpp_5w1s", dict(batch_size=2), [(0, 0)]),
    "omniglot_maml_5w1s":   ("omniglot_maml_5w1s", dict(batch_size=2), [(0, 0)]),
    "mini_imagenet_mamlpp_5w1s": ("mini_imagenet_mamlpp_5w1s", dict(batch_size=1), [(0, 0)]),
    "omniglot_mamlpp_20w5s": ("omniglot_mamlpp_20w5s", dict(batch_size=1), [(0, 0)]),
    # the benchmarked input distribution of BASELINE configs[1] (exact pooling ties)
    "omniglot_mamlpp_5w1s_bernoulli": ("omniglot_mamlpp_5w1s", dict(batch_size=2), [(0, 0)], "bernoulli"),
    # BASELINE configs[3] shape (Mini-ImageNet 5-way 5-shot), one task
    "mini_imagenet_mamlpp_5w5s": ("mini_imagenet_mamlpp_5w5s", dict(batch_size=1), [(0, 0)]),
}


def case_kind(case):
    c = CASES[case]
    return c[3] if len(c) > 3 else KIND


def make_args(case):
    base, over, iters = CASES[case][:3]
    d = dict(CONFIGS[base])
    d.update(over)
    d["experiment_name"] = case
    return args_from_json(None, **d), d, iters


def build_reference(args, dtype):
    sys.path.insert(0, REF)
    import few_shot_learning_system as ref_sys  # noqa: the reference, unmodified
    with contextlib.redirect_stdout(io.StringIO()):
        model = ref_sys.MAMLFewShotClassifier(
            im_shape=(2, args.image_channels, args.image_height, args.image_width),
            device=torch.device("cpu"), args=args)
    if dtype == torch.float64:
        model.double()
    return model


def run_reference_fp32(args, iters, store_inputs, kind=KIND):
    """fp32 reference run.  The true model gives the losses / logits / post-Adam state.  The outer
    gradients are captured on a twin model whose ``dataset_name`` lacks 'imagenet' -- the reference clamps
    ``param.grad`` in place between ``backward`` and ``optimizer.step`` (:332-335), so the twin is the only
    way to see the UNCLAMPED gradients without editing the reference.  The twin is reloaded from the true
    model's parameters before every iteration."""
    import copy
    import warnings
    warnings.filterwarnings("ignore")
    model = build_reference(args, torch.float32)
    args_nc = copy.copy(args)
    args_nc.dataset_name = args.dataset_name.replace("imagenet", "imgnet")
    twin = build_reference(args_nc, torch.float32)
    out = {}
    for k, v in model.state_dict().items():
        out["state/" + k] = v.detach().numpy().copy()
    for it, (epoch, seed_it) in enumerate(iters):
        batch = O.synthetic_batch(args, iteration=seed_it, kind=kind)
        if store_inputs:
            for nm, t in zip(("xs", "xt", "ys", "yt"), batch):
                out["it%d/%s" % (it, nm)] = t.numpy().copy()
        twin.load_state_dict(copy.deepcopy(model.state_dict()))
        captured = {}
        orig_step = twin.optimizer.step

        def step_and_capture(*a, **kw):
            for n, p in twin.named_parameters():
                if p.requires_grad:
                    captured[n] = (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p))
            return None          # the twin never updates

        twin.optimizer.step = step_and_capture
        with contextlib.redirect_stdout(io.StringIO()):
            twin.run_train_iter(data_batch=batch, epoch=epoch)
        twin.optimizer.step = orig_step
        with contextlib.redirect_stdout(io.StringIO()):
            losses, preds = model.run_train_iter(data_batch=batch, epoch=epoch)
        out["it%d/loss" % it] = np.float64(float(losses["loss"]))
        out["it%d/accuracy" % it] = np.float64(float(losses["accuracy"]))
        out["it%d/learning_rate" % it] = np.float64(float(losses["learning_rate"]))
        S = args.number_of_training_steps_per_iter
        out["it%d/msl" % it] = np.array([float(losses["loss_importance_vector_%d" % i]) for i in range(S)])
        out["it%d/logits" % it] = np.stack(preds).astype(np.float32)
        for n, g in captured.items():
            out["it%d/grad/%s" % (it, n)] = g.numpy().copy()
        for k, v in model.state_dict().items():
            out["it%d/post/%s" % (it, k)] = v.detach().numpy().copy()
    return out


def run_reference_validation(args, iters, state32, kind=KIND):
    """Reference ``run_validation_iter`` (few_shot_learning_system.py:371-397) from the INITIAL state on the first
    recorded batch: loss, accuracy, last-step logits and the running statistics afterwards (the reference's
    backup/restore of them is an alias, meta_neural_network_architectures.py:240-255, so they come out mutated)."""
    model = build_reference(args, torch.float32)
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in state32.items()})
    epoch, seed_it = iters[0]
    model.current_epoch = int(epoch)
    batch = O.synthetic_batch(args, iteration=seed_it, kind=kind)
    with contextlib.redirect_stdout(io.StringIO()):
        losses, preds = model.run_validation_iter(data_batch=batch)
    out = {"val/loss": np.float64(float(losses["loss"])), "val/accuracy": np.float64(float(losses["accuracy"])),
           "val/logits": np.stack(preds).astype(np.float32)}
    for k, v in model.state_dict().items():
        if "running" in k:
            out["val/post/" + k] = v.detach().numpy().copy()
    return out


def run_reference_fp64(args, iters, state32, big, kind=KIND):
    """fp64 reference gradients at the SAME parameters as each fp32 iteration started from
    (iteration 0 only -- later iterations start from fp32-updated parameters)."""
    model = build_reference(args, torch.float64)
    sd = {k: torch.from_numpy(v).double() for k, v in state32.items()}
    model.load_state_dict(sd)
    epoch, seed_it = iters[0]
    batch = O.synthetic_batch(args, iteration=seed_it, kind=kind)
    xs, xt, ys, yt = batch
    model.current_epoch = int(epoch)
    data = (xs.double(), xt.double(), ys.long(), yt.long())
    with contextlib.redirect_stdout(io.StringIO()):
        losses, _ = model.train_forward_prop(data_batch=data, epoch=int(epoch))
        model.optimizer.zero_grad()
        losses["loss"].backward()
    out = {"it0/loss64": np.float64(float(losses["loss"]))}
    for n, p in model.named_parameters():
        if p.requires_grad:
            g = p.grad.detach() if p.grad is not None else torch.zeros_like(p)
            out["it0/grad64/" + n] = g.numpy().astype(np.float32 if big else np.float64)
    return out


def write_reference_checkpoint(case="tiny_pp"):
    """A checkpoint WRITTEN BY THE REFERENCE (its own save_model, few_shot_learning_system.py:399-409) after the recorded
    train iterations of ``case`` -> tests/golden/ref_ckpt_<case>/train_model_latest.  tests/test_host_logic.py loads it
    through this repo's load_model and compares with the post-state fixtures."""
    import warnings
    warnings.filterwarnings("ignore")
    args, argdict, iters = make_args(case)
    model = build_reference(args, torch.float32)
    for epoch, seed_it in iters:
        batch = O.synthetic_batch(args, iteration=seed_it, kind=case_kind(case))
        with contextlib.redirect_stdout(io.StringIO()):
            model.run_train_iter(data_batch=batch, epoch=epoch)
    d = os.path.join(ROOT, "tests", "golden", "ref_ckpt_" + case)
    os.makedirs(d, exist_ok=True)
    state = {"best_val_acc": 0.25, "best_val_iter": 1, "current_iter": len(iters), "best_epoch": 0,
             "train_loss_mean": 1.5, "per_epoch_statistics": {"train_loss_mean": [1.5]}}
    model.save_model(model_save_dir=os.path.join(d, "train_model_latest"), state=state)
    return d


def write_episode_fixture():
    """Episodes drawn by the reference's own ``FewShotLearningDatasetParallel.get_set`` (data.py:478-524) from a small
    synthetic IN-MEMORY dataset (the object is built without its file-scanning __init__) -> tests/golden/episodes.npz:
    for Omniglot-like (1 channel, rot90 train augmentation) and ImageNet-like (3 channels, mean / std normalisation)
    settings, several seeds, augmentation on and off.  The GPU sampler must reproduce them bit for bit."""
    sys.path.insert(0, REF)
    sys.argv = [sys.argv[0]]
    import data as ref_data  # noqa: the reference, unmodified
    from howtotrainyourmamlpytorch_b200.data import synthetic_class_images
    blob = {}
    for tag, dataset_name, C, binary in (("omni", "omniglot_dataset", 1, True), ("imnet", "mini_imagenet_full_size", 3, False)):
        H = W = 8
        classes = synthetic_class_images(12, 7, H, W, C, seed=11 if C == 1 else 12, binary=binary)
        args, _, _ = make_args("tiny_pp")
        args.dataset_name = dataset_name
        args.image_channels, args.image_height, args.image_width = C, H, W
        args.num_classes_per_set, args.num_samples_per_class, args.num_target_samples = 4, 2, 3
        ds = object.__new__(ref_data.FewShotLearningDatasetParallel)
        ds.args = args
        ds.dataset_name = dataset_name
        ds.data_loaded_in_memory = True
        ds.image_channel = C
        ds.num_classes_per_set, ds.num_samples_per_class, ds.num_target_samples = 4, 2, 3
        ds.dataset_size_dict = {"train": {k: len(v) for k, v in classes.items()}}
        ds.datasets = {"train": {k: v for k, v in classes.items()}}
        cases = []
        for seed in (5, 123456, 99):
            for aug in (False, True):
                xs, xt, ys, yt, _ = ds.get_set("train", seed=seed, augment_images=aug)
                key = "%s/seed%d_aug%d" % (tag, seed, int(aug))
                blob[key + "/xs"] = xs.numpy().astype(np.float32); blob[key + "/xt"] = xt.numpy().astype(np.float32)
                blob[key + "/ys"] = np.asarray(ys, dtype=np.float32); blob[key + "/yt"] = np.asarray(yt, dtype=np.float32)
                cases.append((seed, int(aug)))
        blob[tag + "/cases"] = np.array(cases)
        blob[tag + "/meta"] = np.array(json.dumps({"dataset_name": dataset_name, "C": C, "H": H, "W": W, "classes": 12,
                                                   "samples": 7, "seed": 11 if C == 1 else 12, "binary": binary,
                                                   "N": 4, "K": 2, "T": 3}))
    path = os.path.join(ROOT, "tests", "golden", "episodes.npz")
    np.savez_compressed(path, **blob)
    return path


class _CallRecorder(object):
    """Stands in for a model: forwards everything to ``model`` and logs the public calls an experiment driver makes on
    it (method, keyword arguments as JSON, what came back)."""

    def __init__(self, model, root):
        self._model, self._root, self.calls = model, root, []

    def __getattr__(self, name):
        attr = getattr(self._model, name)
        if name not in ("run_train_iter", "run_validation_iter", "save_model", "load_model"):
            return attr

        def call(*args, **kwargs):
            assert not args, "%s called with positional arguments" % name
            rec = {"method": name, "kwargs": {}}
            for k, v in kwargs.items():
                if k == "data_batch":
                    rec["kwargs"][k] = [{"type": type(t).__name__, "dtype": str(t.dtype), "shape": list(t.shape)} for t in v]
                elif k == "model_save_dir":
                    rec["kwargs"][k] = os.path.relpath(v, self._root)
                elif k == "state":
                    rec["kwargs"][k] = {sk: sv for sk, sv in v.items() if isinstance(sv, (int, float, str))}
                else:
                    rec["kwargs"][k] = v
            with contextlib.redirect_stdout(io.StringIO()):
                out = attr(**kwargs)
            if name in ("run_train_iter", "run_validation_iter"):
                rec["losses"] = {k: float(v) for k, v in out[0].items()}
            elif name == "load_model":
                rec["state"] = {sk: sv for sk, sv in out.items() if isinstance(sv, (int, float, str))}
            self.calls.append(rec)
            return out
        return call


def write_builder_fixture(case="tiny_maml"):
    """The calls the reference's own ``ExperimentBuilder`` (experiment_builder.py) makes on a model, recorded while it
    drives the reference's ``MAMLFewShotClassifier`` on the first recorded batch of ``case``: ``train_iteration`` (numpy
    episodes), ``evaluation_iteration`` (torch episodes), ``save_models`` after one iteration, and a second builder that
    resumes from ``latest`` -> tests/golden/experiment_builder_<case>.json.  The GPU test replays them on this repo's
    class."""
    import shutil
    import tempfile
    import warnings
    import tqdm
    warnings.filterwarnings("ignore")
    sys.path.insert(0, REF)
    sys.argv = [sys.argv[0]]
    import experiment_builder as ref_builder  # noqa: the reference, unmodified

    class _Data(object):                       # stands in for MetaLearningSystemDataLoader (no dataset on disk)
        def __init__(self, args, current_iter):
            self.dataset = type("D", (), {"seed": {"train": 0, "val": 0}})()

    args, _, iters = make_args(case)
    g = np.load(os.path.join(ROOT, "tests", "golden", case + ".npz"))
    xs, xt, ys, yt = (torch.from_numpy(g["it0/" + n]) for n in ("xs", "xt", "ys", "yt"))
    tmp = tempfile.mkdtemp()
    try:
        args.experiment_name = os.path.join(tmp, "exp")
        args.continue_from_epoch = "from_scratch"
        args.max_models_to_save = 2
        args.total_epochs_before_pause = 1
        model = build_reference(args, torch.float32)
        model.load_state_dict({k[len("state/"):]: torch.from_numpy(g[k]) for k in g.files if k.startswith("state/")})
        rec = _CallRecorder(model, tmp)
        with contextlib.redirect_stdout(io.StringIO()):
            eb = ref_builder.ExperimentBuilder(args=args, data=_Data, model=rec, device=torch.device("cpu"))
        with contextlib.redirect_stdout(io.StringIO()), tqdm.tqdm(total=2, disable=True) as pbar:
            _, _, it = eb.train_iteration(train_sample=(xs.numpy(), xt.numpy(), ys.numpy(), yt.numpy(), 0), sample_idx=0,
                                          epoch_idx=float(iters[0][0]), total_losses={}, current_iter=0, pbar_train=pbar)
            eb.evaluation_iteration(val_sample=(xs, xt, ys, yt, 0), total_losses={}, pbar_val=pbar, phase="val")
            eb.state["current_iter"] = it
            eb.save_models(model=rec, epoch=0, state=eb.state)
        saved = sorted(os.listdir(eb.saved_models_filepath))
        args.continue_from_epoch = "latest"
        rec2 = _CallRecorder(build_reference(args, torch.float32), tmp)
        with contextlib.redirect_stdout(io.StringIO()):
            ref_builder.ExperimentBuilder(args=args, data=_Data, model=rec2, device=torch.device("cpu"))
        out = {"case": case, "calls": rec.calls, "saved_models": saved, "resume_calls": rec2.calls}
    finally:
        shutil.rmtree(tmp)
    path = os.path.join(ROOT, "tests", "golden", "experiment_builder_%s.json" % case)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")
    return path


def check_against_oracle(args, blob, iters, kind=KIND):
    """Immediately validate both restatements against what was just generated."""
    state = {k[len("state/"):]: torch.from_numpy(v) for k, v in blob.items() if k.startswith("state/")}
    epoch, seed_it = iters[0]
    batch = O.synthetic_batch(args, iteration=seed_it, kind=kind)
    worst = {}
    for nm, fn in (("autograd", O.autograd_train_iter), ("manual", O.manual_train_iter)):
        for dt, suffix in ((torch.float32, ""), (torch.float64, "64")):
            st = {k: v.to(dt) for k, v in state.items()}
            res = fn(st, args, batch, epoch)
            ref_loss = float(blob["it0/loss" + suffix])
            err = abs(float(res["loss"]) - ref_loss) / max(abs(ref_loss), 1e-30)
            gerr = 0.0
            for n, g in res["grads"].items():
                ref = torch.from_numpy(blob["it0/grad%s/%s" % (suffix, n)]).to(torch.float64)
                denom = float(ref.abs().max())
                if denom < 1e-6:
                    continue  # dead conv-bias gradients: pure noise in the reference
                gerr = max(gerr, float((g.double() - ref).abs().max()) / denom)
            worst[nm + suffix] = (err, gerr)
    # validation leg (fp32): loss, logits and the mutated running statistics
    for nm, fn in (("autograd", O.autograd_train_iter), ("manual", O.manual_train_iter)):
        res = fn(state, args, batch, epoch, training_phase=False, current_epoch=epoch)
        ref_loss = float(blob["val/loss"])
        err = abs(float(res["loss"]) - ref_loss) / max(abs(ref_loss), 1e-30)
        lerr = float((res["logits"].float() - torch.from_numpy(blob["val/logits"])).abs().max())
        rerr = 0.0
        for k, v in res["running"].items():
            rerr = max(rerr, float((v - torch.from_numpy(blob["val/post/" + k])).abs().max()))
        worst[nm + "_val"] = (err, max(lerr, rerr))
    return worst


def main():
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    which = sys.argv[1:] or list(CASES.keys())
    torch.set_num_threads(THREADS)
    if "--episodes" in which:
        print(write_episode_fixture())
        return
    if "--checkpoint" in which:
        print(write_reference_checkpoint("tiny_pp"))
        return
    if "--builder" in which:
        print(write_builder_fixture("tiny_maml"))
        return
    for case in which:
        args, argdict, iters = make_args(case)
        kind = case_kind(case)
        big = not case.startswith("tiny_")
        blob = run_reference_fp32(args, iters, store_inputs=not big, kind=kind)
        state32 = {k[len("state/"):]: v for k, v in blob.items() if k.startswith("state/")}
        blob.update(run_reference_validation(args, iters, state32, kind))
        blob.update(run_reference_fp64(args, iters, state32, big, kind))
        blob["args_json"] = np.array(json.dumps(argdict))
        blob["iters_json"] = np.array(json.dumps(iters))
        blob["kind"] = np.array(kind)
        path = os.path.join(ROOT, "tests", "golden", case + ".npz")
        np.savez_compressed(path, **blob)
        worst = check_against_oracle(args, blob, iters, kind)
        print(case, "%.1f KB" % (os.path.getsize(path) / 1024.0),
              {k: ("%.1e" % a, "%.1e" % b) for k, (a, b) in worst.items()}, flush=True)


if __name__ == "__main__":
    main()
