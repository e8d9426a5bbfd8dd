"""``python -m idelucs_b200`` — the reference CLI surface (idelucs/__main__.py:274-318: same
flags and defaults) driving the B200-native hot path.  Orchestration only: voters x epochs,
majority vote over voters (k-means on one-hot votes, utils.py:582-602) or HDBSCAN on the latent space when
--n_clusters=0 (the ``hdbscan`` package if importable, else scikit-learn's algorithm with its all-pairs work on the GPU,
``hdbscan.hdbscan_device``), metrics (silhouette on the GPU, ``metrics.silhouette_score_device``) and TSV output:
assignments.tsv and metrics.tsv under Results/<fasta stem>/<time>/.  ``--gpus N`` (N >= 2) trains data-parallel on N GPUs with
train.ShardedTrainer's graph-captured step (run_gpus), with --global_batch_loss on the losses of the global batch; the tail is the
same."""
import argparse
import os
import sys
import time

import numpy as np


def run(args):
    import torch
    from . import models
    from .utils import SummaryFasta
    start = time.time()
    # the all-pairs passes after training (HDBSCAN, silhouette) are split over every visible GPU; training uses one
    devices = list(range(torch.cuda.device_count()))
    use_hdbscan = False
    if args["n_clusters"] == 0:   # idelucs/__main__.py:75-83: 200 output units, clusters from HDBSCAN on the latent space
        args["n_clusters"], use_hdbscan = 200, True
    model = models.IID_model(args)
    model.names, model.lengths, model.GT, model.cluster_dis = SummaryFasta(model.sequence_file, model.GT_file)
    print(model.cluster_dis)
    print(f"No. Sequences: \t {len(model.lengths):,}")
    print(f"Min. Length: \t {np.min(model.lengths):,}")
    print(f"Max. Length: \t {np.max(model.lengths):,}")
    print(f"Avg. Length: \t {round(float(np.mean(model.lengths)), 2):,}")
    model.build_dataloader()
    predictions, latent, probabilities = [], None, None
    min_loss, model_latent = np.inf, None
    for voter in range(args["n_voters"]):
        sys.stdout.write(f"\r........... Training Model ({voter + 1}/{args['n_voters']})................")
        sys.stdout.flush()
        model.net.apply(models.weights_init)
        model.epoch = 0
        voter_min = np.inf
        for _ in range(args["n_epochs"]):
            voter_min = min(voter_min, model.contrastive_training_epoch())
        y_pred, probabilities, latent = model.predict(device_latent=True)
        if voter_min < min_loss:
            min_loss, model_latent = voter_min, latent
        if not use_hdbscan:   # relabel in order of first appearance (__main__.py:131-141)
            predictions.append(_relabel(y_pred))
    return _report(args, model.names, model.GT, predictions, latent, use_hdbscan, devices, start)


def _relabel(y_pred):
    y_pred = y_pred.astype(np.int32)
    first = {}
    return np.array([first.setdefault(int(c), len(first)) for c in y_pred], dtype=np.int32)


def _report(args, names, GT, predictions, latent, use_hdbscan, devices, start):
    """the tail after the voters: vote ensemble or HDBSCAN, assignments.tsv, metrics.tsv and the printout"""
    from .utils import compute_results, external_results, label_features
    if use_hdbscan:   # __main__.py:149-156 (the last voter's latent space, like the reference)
        msz = len(names) // 100 + 1
        try:
            import hdbscan
        except ImportError:   # scikit-learn's HDBSCAN with its all-pairs work on the GPU (same results as sklearn.cluster.HDBSCAN)
            from .hdbscan import default_devices, hdbscan_device
            with default_devices(devices):
                labels, probabilities = hdbscan_device(latent, max(msz, 2))
        else:
            clusterer = hdbscan.HDBSCAN(min_cluster_size=msz, gen_min_span_tree=True, prediction_data=True)
            clusterer.fit(latent.cpu().numpy().astype(np.float64))
            labels, probabilities = clusterer.labels_, clusterer.probabilities_
        y_pred = labels + 1
        args["n_clusters"] = int(np.max(y_pred)) + 1
    else:
        y_pred, probabilities = label_features(np.array(predictions), args["n_clusters"])
    out_dir = os.path.join(os.getcwd(), "Results", os.path.basename(args["sequence_file"]).split(".")[0],
                           time.strftime("%b_%d_%H-%M-%S"))
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "assignments.tsv"), "w") as fh:
        fh.write("sequence_id\tassignment\tconfidence_score\n")
        for name, c, pr in zip(names, y_pred, probabilities):
            fh.write(f"{name}\t{int(c)}\t{float(pr):.6f}\n")
    print("\n")
    y_true = None
    if GT is not None:
        labels = {c: i for i, c in enumerate(sorted(set(GT)))}
        y_true = np.array([labels[c] for c in GT])
    # __main__.py:163-232: the metrics of the last voter's latent space
    n_found = len(np.unique(y_pred))
    if 1 < n_found < len(y_pred):
        results, _ = compute_results(y_pred, latent, y_true, devices=devices)
        note = None
    else:   # silhouette and Davies-Bouldin are undefined; the run still reports what it can
        results = {"Davies-Boulding": float("nan"), "Silhouette-Score": float("nan")}
        if y_true is not None:
            results.update(external_results(y_pred, y_true)[0])
        note = f"Silhouette and Davies-Bouldin need 2 to {len(y_pred) - 1} clusters, got {n_found}: written as nan"
    with open(os.path.join(out_dir, "metrics.tsv"), "w") as fh:
        fh.write("\t".join(results) + "\n")
        fh.write("\t".join(repr(float(v)) for v in results.values()) + "\n")
    if y_true is not None:
        print(f"ACC \t {results['ACC']:.5f}")
        print(f"ARI \t {results['ARI']:.5f}")
        print(f"NMI \t {results['NMI']:.5f}")
    if note:
        print(note)
    print(f"Silhouette \t {results['Silhouette-Score']:.5f}")
    print(f"Davies-Bouldin \t {results['Davies-Boulding']:.5f}")
    print(f"Elapsed \t {time.time() - start:.1f} s   results in {out_dir}")
    return y_pred


def _free_port():
    import socket
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def run_gpus(args, gpus):
    """--gpus N >= 2: one worker process per GPU (torch.multiprocessing, NCCL rendezvous on a free local port), each training the
    same NetLinear replica on its shard of the sequences with train.ShardedTrainer's graph-captured step; rank 0 then runs the
    tail of run() on the gathered predictions.  A failing rank makes mp.spawn stop the others and raise here."""
    import torch.multiprocessing as mp
    mp.spawn(_rank_main, args=(gpus, _free_port(), args), nprocs=gpus, join=True)


def _rank_main(rank, world, port, args):
    import torch
    import torch.distributed as dist
    from . import featurise as ft
    from . import parallel
    from .seqset import read_fasta_native, SeqSet
    from .train import ShardedTrainer
    from .utils import SummaryFasta
    start = time.time()
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    use_hdbscan = args["n_clusters"] == 0
    n_clusters = 200 if use_hdbscan else args["n_clusters"]
    if rank == 0:
        names, lengths, GT, cluster_dis = SummaryFasta(args["sequence_file"], args["GT_file"])
        print(cluster_dis)
        print(f"No. Sequences: \t {len(lengths):,}")
        print(f"Min. Length: \t {np.min(lengths):,}")
        print(f"Max. Length: \t {np.max(lengths):,}")
        print(f"Avg. Length: \t {round(float(np.mean(lengths)), 2):,}")
    # every rank packs only its own contiguous shard (parallel.shard_ranges over the record lengths)
    _, _, byte_off = read_fasta_native(args["sequence_file"], pinned=False)
    n_total = byte_off.size - 1
    lo, hi = parallel.shard_ranges(np.diff(byte_off), world)[rank]
    ss = SeqSet.from_fasta(args["sequence_file"], device=dev, rows=(lo, hi))
    # --batch_sz is the global batch: batch_sz / N pairs per rank, and ceil(pairs / batch_sz) steps per epoch on every rank — the
    # number of optimiser updates of the reference's loader
    steps = -(-(len(ft.mimic_schedule(args["n_mimics"])) - 1) * n_total // args["batch_sz"])
    tr = ShardedTrainer(ss, k=args["k"], n_clusters=n_clusters, n_mimics=args["n_mimics"], batch_sz=args["batch_sz"] // world,
                        lamb=args["lambda"], weight=args["weight"], lr=args["lr"], seed=0, seq_id0=lo, world=world,
                        optimizer=args["optimizer"], global_batch_loss=args.get("global_batch_loss", False))
    tr.enable_cuda_graph()
    tr.reset_optimizer()   # (the capture's warm-up steps trained the network: start from a fresh optimiser)
    predictions, latent = [], None
    for voter in range(args["n_voters"]):
        if rank == 0:
            sys.stdout.write(f"\r........... Training Model ({voter + 1}/{args['n_voters']})................")
            sys.stdout.flush()
        tr.reinit(voter)
        voter_min = np.inf
        for _ in range(args["n_epochs"]):
            for _ in range(steps):
                tr.step()
            voter_min = min(voter_min, tr.epoch_loss(steps))
        y_pred, _, latent = tr.predict(ss, k=args["k"])
        lo_p, hi_p = tr._flat_param.clone(), tr._flat_param.clone()
        dist.all_reduce(lo_p, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_p, op=dist.ReduceOp.MAX)
        if not (torch.equal(lo_p, tr._flat_param) and torch.equal(hi_p, tr._flat_param)):
            raise RuntimeError("rank %d: the parameter replicas differ after voter %d" % (rank, voter + 1))
        if rank == 0 and not use_hdbscan:
            predictions.append(_relabel(y_pred.cpu().numpy()))
    dist.destroy_process_group()   # (no NCCL kernel keeps the other GPUs busy while rank 0 finishes)
    if rank != 0:
        return
    _report(args, names, GT, predictions, latent, use_hdbscan, list(range(torch.cuda.device_count())), start)


def main(argv=None):
    parser = argparse.ArgumentParser(prog="idelucs")
    parser.add_argument("--sequence_file", action="store", type=str)
    parser.add_argument("--n_clusters", action="store", type=int, default=0,
                        help="Expected or maximum number of clusters (0: fine-grained clusters via HDBSCAN)")
    parser.add_argument("--n_epochs", action="store", type=int, default=100)
    parser.add_argument("--n_mimics", action="store", type=int, default=3, help="data augmentations per sequence")
    parser.add_argument("--batch_sz", action="store", type=int, default=256)
    parser.add_argument("--GT_file", action="store", type=str, default=None)
    parser.add_argument("--k", action="store", type=int, default=6, help="k-mer length")
    parser.add_argument("--optimizer", action="store", type=str, default="RMSprop")
    parser.add_argument("--scheduler", action="store", type=str, default="None")
    parser.add_argument("--weight", action="store", type=float, default=0.25, help="weight of the IIC term")
    parser.add_argument("--lambda", action="store", type=float, default=2.8, help="cluster balance")
    parser.add_argument("--lr", action="store", type=float, default=1e-3)
    parser.add_argument("--n_voters", action="store", type=int, default=5)
    parser.add_argument("--model_size", action="store", type=str, default="linear")
    parser.add_argument("--plot", action="store", type=bool, default=False)
    parser.add_argument("--gpus", action="store", type=int, default=argparse.SUPPRESS,
                        help="train data-parallel on this many GPUs (default 1); --batch_sz stays the global batch")
    parser.add_argument("--global_batch_loss", action="store_true", default=argparse.SUPPRESS,
                        help="with --gpus N >= 2: evaluate both losses on the global batch (the ranks exchange the IIC joint and the "
                             "InfoNCE latents), as one GPU does, instead of on each GPU's batch_sz / N pairs")
    args = vars(parser.parse_args(argv))
    gpus = args.pop("gpus", 1)
    global_batch_loss = args.pop("global_batch_loss", False)   # (one GPU already trains on the global batch)
    print("\nTraining Parameters:")
    for key in args:
        print(f"{key} \t -> {args[key]}")
    if not args["sequence_file"]:
        parser.error("--sequence_file is required")
    if gpus == 1:
        run(args)
        return
    from .train import OPTIMIZERS
    if gpus < 1:
        parser.error(f"--gpus must be at least 1, got {gpus}")
    if args["model_size"] != "linear":
        parser.error(f"--gpus {gpus} trains the fused NetLinear step: --model_size must be 'linear', got '{args['model_size']}'")
    if args["scheduler"] != "None":
        parser.error(f"--gpus {gpus} runs with a constant learning rate: --scheduler must be 'None', got '{args['scheduler']}'")
    if args["optimizer"] not in OPTIMIZERS:
        parser.error(f"--optimizer must be one of {', '.join(OPTIMIZERS)}, got '{args['optimizer']}'")
    if args["batch_sz"] % gpus:
        parser.error(f"--batch_sz {args['batch_sz']} is the global batch: it must be a multiple of --gpus {gpus}")
    import torch
    if gpus > torch.cuda.device_count():
        parser.error(f"--gpus {gpus}: only {torch.cuda.device_count()} CUDA devices are visible")
    print(f"gpus \t -> {gpus}")
    if global_batch_loss:
        print("global_batch_loss \t -> True")
        args["global_batch_loss"] = True
    run_gpus(args, gpus)


if __name__ == "__main__":
    main()
