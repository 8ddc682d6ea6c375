"""Drop-in for reference ``src/ml/train.py``.

    python -m cubecobrarecommender_b200.ml.train epochs batch_size name reg noise [seed] [--validation-split F]
                                                 [--rank-at K1,K2,...] [--rank-cuts]
                                                 [--rank-baselines graph,popularity]

Same positional arguments (reference train.py:28-38), same inputs (``data/maps/nameToId.json``,
``data/cube/*.json``, ``output/full_adj_mtx.npy``), same M-hat construction (train.py:69-71), loss and
optimiser (train.py:83-88).  The model is saved under ``ml_files/<name>/`` in this package's npz
checkpoint format (TensorFlow SavedModel is not available; see DESIGN.md).  Under ``torchrun`` the cubes
of every batch and the regulariser rows are sharded over the ranks and gradients are all-reduced.
"""
from __future__ import annotations

import os
import random
import sys
import time

import numpy as np
import torch


def reset_random_seeds(seed):
    os.environ['PYTHONHASHSEED'] = str(seed)
    torch.manual_seed(seed)
    np.random.seed(seed)
    random.seed(seed)


def progress_line(steps, seconds, logs):
    """Keras' end-of-epoch progress line: ``steps/steps - Ns - key: value - ...`` in the order of ``logs``."""
    return f"{steps}/{steps} - {seconds:.0f}s" + "".join(f" - {k}: {v:.4f}" for k, v in logs.items())


def shard_range(n, rank, world):
    """[lo, hi) of the contiguous shard of n items that rank ``rank`` of ``world`` takes (sizes differ by at most one)."""
    return (n * rank) // world, (n * (rank + 1)) // world


def evaluate(model, generator, reg, *, group=None, metrics=True, engine=None):
    """Keras' ``model.evaluate(generator)``: ``{"loss", "output_1_loss", "output_2_loss", "output_1_accuracy",
    "output_2_accuracy"}`` over every cube of ``generator``, as sample-weighted means over the whole set:
    output_1_loss = sum BCE / (K C), output_2_loss = sum_v KL_v / K, loss = output_1_loss + reg * output_2_loss, the
    accuracies = hits / (K C) and hits / K.  Cube v is corrupted by the generator's fixed validation noise and paired
    with reg row v of its fixed draw (``DataGenerator.validation_draws``), so the result does not depend on the batch
    size or the number of ranks beyond summation order.  Under ``torchrun`` each rank evaluates a contiguous shard of the
    cubes and one all_reduce adds the sums.  ``engine``: a DAEEngine to run on (``fit`` passes its training engine);
    none of its parameters, gradients, Adam slots or counters change.  Note that M-hat is built from every cube, the
    held-out ones included."""
    import torch.distributed as dist
    from .engine import DAEEngine
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    k = generator.N_cubes
    if k < 1:
        raise ValueError("evaluate: the generator holds no cubes")
    if engine is None:
        lb = max(generator.batch_size // world, 1)
        engine = DAEEngine(model, generator.mhat_device(), batch=lb, reg_rows=lb, reg=reg,
                           max_cube_size=max(generator.csr.max_size, 1), group=group)
    seed, counter, reg_rows = generator.validation_draws()
    lo, hi = shard_range(k, rank, world)
    step = min(engine.B, engine.R) if engine.R else engine.B
    sums = torch.zeros(4, dtype=torch.float64, device=model.device)
    ids = torch.arange(k, dtype=torch.int32, device=model.device)
    for b0 in range(lo, hi, step):
        b1 = min(b0 + step, hi)
        engine.sample_eval_batch(generator.indptr, generator.indices_dev, ids[b0:b1], generator.alias_prob,
                                 generator.alias_idx, generator.noise, generator.noise_std, seed, counter)
        engine.evaluate_batch(b1 - b0, reg_rows[b0:b1], sums, metrics=metrics)
    if world > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    engine.check_overflow()
    t = sums.cpu().numpy()
    c = float(generator.N_cards)
    bce, kl = t[0] / (k * c), t[1] / k
    out = {"loss": float(bce + reg * kl), "output_1_loss": float(bce), "output_2_loss": float(kl)}
    if metrics:
        out.update({"output_1_accuracy": float(t[2] / (k * c)), "output_2_accuracy": float(t[3] / k)})
    return out


def evaluate_recommendations(model, generator, *, at=(10, 50), holdout=0.2, group=None):
    """Leave-k-out ranking quality of the recommendations over every cube of ``generator``: each cube of s >= 2 cards
    hides ``min(s - 1, max(1, floor(holdout * s + 0.5)))`` of them (``DataGenerator.holdout_split``: the same cards in
    every call), the model sees the rest, and every hidden card is ranked among all the cards the cube does not show,
    in the order ``MLRecommender.recommend_device`` lists them.  ``model``: a ``CC_Recommender`` (ranked through
    ``MLRecommender``) or any recommender with ``target_ranks_device(visible, hidden)`` -- ``MLRecommender``,
    ``graph.GraphRecommender``, ``graph.PopularityRecommender`` -- so the baselines are scored on the same hidden cards
    by the same code (see ``ranking_baselines``).  Returns ``{"recall_at_k", "ndcg_at_k",
    "hit_rate_at_k"}`` for each k in ``at``, ``"mrr"``, ``"mpr"`` (mean percentile rank: 0.5 for a random ranking) --
    each a mean over the evaluated cubes, see ``ranking.ranking_sums`` -- plus ``"cubes"`` (evaluated) and ``"skipped"``
    (fewer than two cards).  Under ``torchrun`` each rank takes a contiguous shard of the cubes and one all_reduce adds
    the sums; the only host read is the final one.  Parameters, gradients, the tf32 shadow, Adam slots and step
    counters are left untouched, and no random stream is drawn from.  M-hat is built from every cube, the held-out
    ones included."""
    return _ranking_eval("evaluate_recommendations", model, generator, at, group,
                         lambda: generator.holdout_split(holdout), "target_ranks_device",
                         lambda vis: generator.N_cards - np.diff(vis.indptr))


def evaluate_cuts(model, generator, *, at=(10, 50), inject=0.2, group=None):
    """Ranking quality of the cut list over every cube of ``generator``: each cube of s >= 1 cards gets
    ``max(1, floor(inject * s + 0.5))`` intruders, cards of another cube that it does not hold
    (``DataGenerator.intruder_split``: the same cards in every call), the model sees the corrupted cube, and every
    intruder is placed where the cube's cut list (its cards by ascending probability, ties to the smaller index) would
    list it, among the s + m cards of the corrupted cube.  A good cutter lists the intruders first.  ``model``: a
    ``CC_Recommender`` (ranked through ``MLRecommender``) or any recommender with ``cut_ranks_device(corrupted,
    intruders)`` -- ``MLRecommender``, ``graph.GraphRecommender`` (``simple_cuts``), ``graph.PopularityRecommender``.
    Returns the keys of ``evaluate_recommendations`` (recall, NDCG and hit rate at each k in ``at``, ``"mrr"``,
    ``"mpr"``: 0.5 for a random ordering), ``"cubes"`` (evaluated) and ``"skipped"`` (no cards, or no intruder
    because the donor holds nothing the cube lacks).  Under ``torchrun`` each rank takes a contiguous shard of the
    split made over the whole set and one all_reduce adds the sums; the only host read is the final one.  Parameters,
    gradients, the tf32 shadow, Adam slots and step counters are left untouched, and no random stream is drawn from.
    M-hat is built from every cube, the held-out ones included."""
    return _ranking_eval("evaluate_cuts", model, generator, at, group, lambda: generator.intruder_split(inject),
                         "cut_ranks_device", lambda corrupted: np.diff(corrupted.indptr))


def _ranking_eval(what, model, generator, at, group, split, method, n_candidates):
    """The metrics of ``ranking.ranking_sums`` over the ranks that recommender method ``method(inputs, targets)`` gives
    this rank's shard of ``split() = (inputs, targets, evaluated)``; ``n_candidates(inputs)``: each cube's candidates."""
    import torch.distributed as dist
    from .inference import MLRecommender
    from .model import CC_Recommender
    from .ranking import metric_names, ranking_sums
    at = tuple(int(k) for k in at)
    if not at or min(at) < 1:
        raise ValueError(f"{what}: every k in `at` must be >= 1, got {at}")
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    k = generator.N_cubes
    if k < 1:
        raise ValueError(f"{what}: the generator holds no cubes")
    inputs, targets, _ = split()
    inp, tgt = inputs.shard(rank, world), targets.shard(rank, world)          # the cubes of shard_range(k, rank, world)
    rec = MLRecommender(model) if isinstance(model, CC_Recommender) else model
    ranks = getattr(rec, method)(inp, tgt)
    dev = ranks.device
    hp = torch.from_numpy(np.ascontiguousarray(tgt.indptr, dtype=np.int64)).to(dev, non_blocking=True)
    n_cand = torch.from_numpy(n_candidates(inp)).to(dev, non_blocking=True)
    sums = ranking_sums(ranks, hp, n_cand, at)
    if world > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    t = sums.cpu().numpy()
    cubes = int(round(t[0]))
    out = {name: float(v / cubes) if cubes else float("nan") for name, v in zip(metric_names(at), t[1:])}
    out.update({"cubes": cubes, "skipped": k - cubes})
    return out


BASELINES = ("graph", "popularity")


def ranking_baselines(train_generator, val_generator, *, names=BASELINES, at, holdout=0.2, group=None, task="adds",
                      inject=0.2):
    """``{name: evaluate_recommendations(...)}`` of simple recommenders on ``val_generator``'s cubes, the same hidden
    cards and metrics as the autoencoder's ranking evaluation, to read its numbers against.  ``"graph"``: the
    co-occurrence recommender (``simple_recs``, reference ``recommend.py:7-18``) with M built from the cubes of
    ``train_generator`` only, so no held-out co-occurrence leaks into it (the autoencoder's M-hat, by contrast, is built
    from every cube).  ``"popularity"``: the cards listed by the most training cubes, the same list for every cube.
    ``task="cuts"``: ``{name: evaluate_cuts(..., inject=inject)}`` instead, the same intruders as the autoencoder's cut
    evaluation; the graph cuts like ``simple_cuts`` (reference ``cut_cards.py:7-18``), popularity cuts the least-listed
    cards first.  Under ``torchrun`` every rank builds the whole graph (no all_reduce of the counts) and ranks its shard
    of the validation cubes; the graph is freed before the function returns."""
    from .. import graph as G
    names = tuple(names)
    unknown = [n for n in names if n not in BASELINES]
    if unknown:
        raise ValueError(f"unknown ranking baseline(s) {unknown}; choose from {list(BASELINES)}")
    if task not in ("adds", "cuts"):
        raise ValueError(f"task must be 'adds' or 'cuts', got {task!r}")
    out = {}
    for name in names:
        if name == "graph":
            g = G.build_graph(train_generator.csr, train_generator.device, allreduce=False, want_m64=True,
                              want_mhat=False, want_neg=False)
            rec = G.GraphRecommender(g.m64)
            del g                                           # the int32 counts go now, M with the recommender below
        else:
            rec = G.PopularityRecommender(train_generator.csr, train_generator.device)
        if task == "adds":
            out[name] = evaluate_recommendations(rec, val_generator, at=at, holdout=holdout, group=group)
        else:
            out[name] = evaluate_cuts(rec, val_generator, at=at, inject=inject, group=group)
        del rec
    return out


def fit(model, generator, epochs, reg, *, group=None, log=print, steps_per_epoch=None, max_cube_size=None,
        initial_epoch=0, checkpoint_dir=None, save_every=None, overflow_check_every=50, metrics=True,
        validation_data=None, validation_split=0.0, validation_freq=1, ranking_at=None, ranking_holdout=0.2,
        ranking_cuts=False, ranking_inject=0.2):
    """``autoencoder.fit(generator, epochs=epochs)`` (reference train.py:99-102).  Returns the history
    ``[{"loss", "output_1_loss", "output_2_loss", "output_1_accuracy", "output_2_accuracy"}]`` per epoch (means over
    the epoch's steps, like Keras' progress line).  ``metrics`` mirrors ``compile(..., metrics=['accuracy'])`` (reference
    train.py:87): Keras resolves the name to binary accuracy on the sigmoid output and categorical accuracy on the
    softmax output; both are counted inside the loss kernels.

    Beyond the reference (SURVEY.md 8f-3): ``initial_epoch`` (Keras' own argument name) continues a run -- the epoch
    shuffle is a function of (seed, epoch), Adam's step counter lives in the model -- and every ``save_every`` epochs the
    model, its Adam slots and the number of completed epochs are written to ``checkpoint_dir`` (rank 0 writes; in p2p
    data-parallel mode the sliced Adam slots are gathered first).

    Held-out validation, with Keras' semantics: ``validation_data`` (a DataGenerator) or ``validation_split`` (the last
    fraction of the cubes, see ``DataGenerator.split``; ignored when ``validation_data`` is given) is evaluated (see
    ``evaluate``) after every epoch with ``(epoch + 1) % validation_freq == 0``, and that epoch's history entry and
    progress line gain ``val_loss``, ``val_output_1_loss``, ``val_output_2_loss`` and, with ``metrics``, the two
    ``val_*_accuracy`` keys.  ``ranking_at`` (a sequence of k): the same epochs also run ``evaluate_recommendations``
    on the validation cubes with ``holdout=ranking_holdout`` and add ``val_recall_at_k``, ``val_ndcg_at_k`` and
    ``val_hit_rate_at_k`` per k, ``val_mrr`` and ``val_mpr``.  ``ranking_cuts`` (needs ``ranking_at``): the same
    epochs also run ``evaluate_cuts`` with ``inject=ranking_inject`` and add ``val_cut_recall_at_k``,
    ``val_cut_ndcg_at_k`` and ``val_cut_hit_rate_at_k`` per k, ``val_cut_mrr`` and ``val_cut_mpr``.  M-hat is built
    from every cube, the validation cubes included."""
    import torch.distributed as dist
    from .engine import DAEEngine
    if ranking_cuts and ranking_at is None:
        raise ValueError("ranking_cuts reports the metrics of ranking_at: it needs ranking_at=(k1, k2, ...)")
    if ranking_at is not None:
        ranking_at = tuple(int(k) for k in ranking_at)
        if validation_data is None and not validation_split:
            raise ValueError("ranking_at needs validation data (validation_data or validation_split)")
        if not ranking_at or min(ranking_at) < 1:
            raise ValueError(f"every k in ranking_at must be >= 1, got {ranking_at}")
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    gb = generator.batch_size
    if gb % world:
        raise ValueError(f"batch_size {gb} must be divisible by the number of ranks {world}")
    lb = gb // world
    val = validation_data
    if val is None and validation_split:
        generator, val = generator.split(validation_split)
    if int(validation_freq) < 1:
        raise ValueError(f"validation_freq must be >= 1, got {validation_freq}")
    sizes = [generator.csr.max_size] + ([val.csr.max_size] if val is not None else [])
    eng = DAEEngine(model, generator.mhat_device(), batch=lb, reg_rows=lb, reg=reg,
                    max_cube_size=max_cube_size or max(max(sizes), 1), global_batch=gb,
                    global_reg_rows=gb, group=group, metrics=metrics)
    history = []
    nsteps = steps_per_epoch or len(generator)
    if initial_epoch:
        generator.reset_indices(initial_epoch)
    for epoch in range(initial_epoch, epochs):
        log(f"Epoch {epoch + 1}/{epochs}")
        t0 = time.time()
        acc = torch.zeros(3, dtype=torch.float64, device=model.device)
        macc = torch.zeros(2, dtype=torch.float64, device=model.device)
        for b in range(nsteps):
            ids_t = generator.batch_ids(b, rank, world)           # a slice of the epoch's device-side permutation
            eng.sample_batch(generator.indptr, generator.indices_dev, ids_t, generator.alias_prob, generator.alias_idx,
                             generator.noise, generator.noise_std, seed=generator.seed + 7919 * rank)
            acc += eng.train_step()
            if metrics:
                macc += eng.metrics2
            if overflow_check_every and (b + 1) % overflow_check_every == 0:
                eng.check_overflow()                                # (one 4-byte read: the only host sync inside an epoch)
        eng.check_overflow()
        mean = (acc / max(nsteps, 1)).cpu().numpy()
        history.append({"loss": float(mean[2]), "output_1_loss": float(mean[0]), "output_2_loss": float(mean[1])})
        if metrics:
            mm = (macc / max(nsteps, 1)).cpu().numpy()
            history[-1].update({"output_1_accuracy": float(mm[0]), "output_2_accuracy": float(mm[1])})
        if val is not None and (epoch + 1) % int(validation_freq) == 0:
            vlogs = evaluate(model, val, reg, group=group, metrics=metrics, engine=eng)
            history[-1].update({"val_" + key: v for key, v in vlogs.items()})
            if ranking_at is not None:
                rlogs = evaluate_recommendations(model, val, at=ranking_at, holdout=ranking_holdout, group=group)
                history[-1].update({"val_" + key: v for key, v in rlogs.items() if key not in ("cubes", "skipped")})
            if ranking_cuts:
                clogs = evaluate_cuts(model, val, at=ranking_at, inject=ranking_inject, group=group)
                history[-1].update({"val_cut_" + key: v for key, v in clogs.items() if key not in ("cubes", "skipped")})
        log(progress_line(nsteps, time.time() - t0, history[-1]))
        generator.on_epoch_end()
        if checkpoint_dir and save_every and (epoch + 1) % save_every == 0 and epoch + 1 < epochs:
            eng.gather_adam_state()
            if rank == 0:
                model.save(checkpoint_dir, epoch=epoch + 1)
    eng.gather_adam_state()      # p2p data parallel: m / v live sliced over the ranks until a checkpoint needs them
    return history


def parse_args(argv):
    """The reference's positional arguments ``epochs batch_size name reg noise [seed]`` and the optional flags."""
    args = list(argv)
    resume = "--resume" in args
    if resume:
        args.remove("--resume")
    rank_cuts = "--rank-cuts" in args
    if rank_cuts:
        args.remove("--rank-cuts")
    flags = {"--save-every": None, "--validation-split": 0.0, "--rank-at": None, "--rank-baselines": None}
    for flag in flags:
        if flag in args:
            i = args.index(flag)
            if i + 1 >= len(args):
                raise SystemExit(f"{flag} needs a value")
            flags[flag] = args[i + 1]
            del args[i:i + 2]
    if len(args) < 5:
        raise SystemExit("usage: train.py epochs batch_size name reg noise [seed] [--save-every N] [--resume] "
                         "[--validation-split F] [--rank-at K1,K2,...] [--rank-cuts] [--rank-baselines graph,popularity]")
    split = float(flags["--validation-split"])
    if not 0.0 <= split < 1.0:
        raise SystemExit(f"--validation-split must lie in [0, 1), got {split}")
    rank_at = None
    if flags["--rank-at"] is not None:
        try:
            rank_at = tuple(int(v) for v in flags["--rank-at"].split(","))
        except ValueError:
            raise SystemExit(f"--rank-at takes comma-separated integers, got {flags['--rank-at']!r}") from None
        if min(rank_at) < 1:
            raise SystemExit(f"--rank-at values must be >= 1, got {flags['--rank-at']}")
        if split == 0.0:
            raise SystemExit("--rank-at ranks the held-out cubes: it needs --validation-split F")
    if rank_cuts and rank_at is None:
        raise SystemExit("--rank-cuts reports the metrics of --rank-at: it needs --rank-at K1,K2,...")
    baselines = None
    if flags["--rank-baselines"] is not None:
        baselines = tuple(v for v in flags["--rank-baselines"].split(",") if v)
        unknown = [v for v in baselines if v not in BASELINES]
        if not baselines or unknown:
            raise SystemExit(f"--rank-baselines takes a comma-separated list of {', '.join(BASELINES)}, "
                             f"got {flags['--rank-baselines']!r}")
        if rank_at is None:
            raise SystemExit("--rank-baselines reports the metrics of --rank-at: it needs --rank-at K1,K2,...")
    return {"epochs": int(args[0]), "batch_size": int(args[1]), "name": args[2], "reg": float(args[3]),
            "noise": float(args[4]), "seed": int(args[5]) if len(args) == 6 else 0, "seed_given": len(args) == 6,
            "resume": resume, "save_every": int(flags["--save-every"]) if flags["--save-every"] is not None else None,
            "validation_split": split, "rank_at": rank_at, "rank_cuts": rank_cuts, "rank_baselines": baselines}


def main(argv=None):
    """``train.py epochs batch_size name reg noise [seed]`` (reference train.py:28-38), plus optional flags the
    reference does not have: ``--save-every N`` writes a checkpoint to ``ml_files/<name>`` every N epochs, ``--resume``
    continues from the checkpoint found there (weights, Adam slots, step counter, completed epochs),
    ``--validation-split F`` holds the last fraction F of the cubes out of training and reports ``val_*`` losses and
    accuracies on them after every epoch, ``--rank-at 10,50`` adds the leave-k-out ranking metrics of those cubes
    (``val_recall_at_10``, ``val_ndcg_at_10``, ``val_hit_rate_at_10``, ..., ``val_mrr``, ``val_mpr``), and
    ``--rank-cuts`` adds the same metrics of the cut list (``evaluate_cuts``: ``val_cut_recall_at_10``, ...,
    ``val_cut_mpr``), and ``--rank-baselines graph,popularity`` prints the same metrics of those baselines
    (``ranking_baselines``) on the same cubes before the first epoch, one ``baseline <name> - recall_at_10: ...`` line
    each, followed with ``--rank-cuts`` by one ``baseline <name> cuts - recall_at_10: ...`` line each."""
    from ..non_ml import utils
    from .generator import DataGenerator
    from .model import CC_Recommender
    opts = parse_args(sys.argv[1:] if argv is None else argv)
    epochs, batch_size, name, reg, noise, seed = (opts[k] for k in ("epochs", "batch_size", "name", "reg", "noise", "seed"))
    resume, save_every = opts["resume"], opts["save_every"]
    if opts["seed_given"]:
        reset_random_seeds(seed)
    import torch.distributed as dist
    if "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
    map_file = '././data/maps/nameToId.json'
    folder = "././data/cube/"
    print('Loading Cube Data . . .\n')
    num_cards, name_lookup, card_to_int, int_to_card = utils.get_card_maps(map_file)
    cubes = utils.build_cubes_csr(folder, num_cards, name_lookup, card_to_int)
    print('Loading Adjacency Matrix . . .\n')
    adj_mtx = np.load('././output/full_adj_mtx.npy')
    print('Creating Graph for Regularization . . . \n')
    y_mtx = adj_mtx.copy()
    np.fill_diagonal(y_mtx, 1)
    y_mtx = (y_mtx / y_mtx.sum(1)[:, None])                                   # train.py:69-71
    print('Setting Up Data for Training . . .\n')
    print('Setting Up Model . . . \n')
    dest = f'././ml_files/{name}'
    precision = os.environ.get("CC_PRECISION", "tf32")
    initial_epoch = 0
    if resume and os.path.exists(os.path.join(dest, "cc_recommender.npz")):
        autoencoder = CC_Recommender.load(dest, device="cuda", precision=precision)
        initial_epoch = autoencoder.completed_epochs
        print(f'Resuming from {dest}: {initial_epoch} epochs done, Adam step {int(autoencoder.store.step.item())}\n')
    else:
        autoencoder = CC_Recommender(num_cards, device="cuda", seed=seed, precision=precision)
    generator = DataGenerator(y_mtx, cubes, batch_size=batch_size, noise=noise, seed=seed)
    if opts["rank_baselines"]:
        from .ranking import metric_names
        train_gen, val_gen = generator.split(opts["validation_split"])          # the halves fit's split makes
        for bname, logs in ranking_baselines(train_gen, val_gen, names=opts["rank_baselines"],
                                             at=opts["rank_at"], holdout=0.2).items():   # fit's ranking_holdout
            print(f"baseline {bname}" + "".join(f" - {key}: {logs[key]:.4f}" for key in metric_names(opts["rank_at"])))
        if opts["rank_cuts"]:
            for bname, logs in ranking_baselines(train_gen, val_gen, names=opts["rank_baselines"], at=opts["rank_at"],
                                                 task="cuts", inject=0.2).items():          # fit's ranking_inject
                print(f"baseline {bname} cuts" + "".join(f" - {key}: {logs[key]:.4f}"
                                                         for key in metric_names(opts["rank_at"])))
        del train_gen, val_gen
    fit(autoencoder, generator, epochs, reg, initial_epoch=initial_epoch, checkpoint_dir=dest, save_every=save_every,
        validation_split=opts["validation_split"], ranking_at=opts["rank_at"], ranking_cuts=opts["rank_cuts"])
    if not dist.is_initialized() or dist.get_rank() == 0:
        autoencoder.save(dest, epoch=epochs)
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
