"""Fine-tune / evaluate ViT + CaRA on VTAB-1k -- the reference's entry point on the B200 kernels.

Usage (as in the reference README, from the repo root):
    PYTHONPATH=. python image_classification/vit_cp.py --dataset=cifar --dim=16
    PYTHONPATH=. python image_classification/vit_cp.py --dataset=cifar --dim=16 --evaluate=ckpt.pt

Flags ``--dim --lr --dataset --evaluate --model`` are the reference's (vit_cp.py:85-116); the step semantics are
its loop body (vit_cp.py:45-50): forward, cross-entropy, backward, AdamW(lr, wd=1e-4) over ``CP*`` + ``head``,
cosine schedule stepped with the epoch index (vit_cp.py:55-56,187), test every 10 epochs and keep the best
checkpoint (vit_cp.py:57-68).  Additive flags: ``--epochs``, ``--batch-size``, ``--synthetic`` (VTAB-shaped
random data when ./data/vtab-1k is absent), ``--no-merge`` (evaluate through the adapter kernels instead of
folding the CP delta into the frozen weights first), ``--weight-dropout exact|skip`` (default exact = the
reference's train-mode dropout on the materialised delta), ``--retrain-mode``, ``--allow-random-init``, ``--img-size``
(fine-tune at another resolution, e.g. 384: the position embedding is resampled and the data resized to match).  Multi-GPU: launch with torchrun; the batch is sharded
over the ranks and only the flat CP+head gradient (<= 1.1 MB) is all-reduced.
"""
import os
import random
import sys
from argparse import ArgumentDefaultsHelpFormatter, ArgumentParser

import numpy as np
import torch as th

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from vtab import get_classes_num, get_data, to_device  # noqa: E402
from vtab_config import config  # noqa: E402

from cara_b200 import train as T  # noqa: E402
from cara_b200.merge import merge_cara  # noqa: E402
from cara_b200.vit import _GEOMETRY, create_model  # noqa: E402
from cara_b200.wdrop import set_weight_dropout  # noqa: E402
from src.cara.cara import cara  # noqa: E402


@th.no_grad()
def test(model, dl, img_size=224):
    """Top-1 accuracy (reference vit_cp.py:73-82; avalanche's Accuracy replaced by a running mean)."""
    model.eval()
    correct = total = 0
    for x, y in dl:
        x, y = to_device(x, y, size=img_size)
        correct += int((model(x).argmax(dim=1).view(-1) == y).sum())
        total += int(y.numel())
    return correct / max(total, 1)


def train(args, model, dl, tdl, opt, epochs, world_size=1, rank=0):
    """Reference vit_cp.py:19-70, including two things that are easy to miss: the learning rate of each step
    (T.EpochCosineSchedule: epoch 0 runs at warmup_lr_init = 1e-6, the scheduler is stepped after opt.step()), and the
    fact that ``test()`` leaves the model in eval mode (vit_cp.py:75) and the loop never calls ``model.train()`` again
    -- from the first periodic test (epoch 10) on, the reference trains WITHOUT weight dropout and DropPath.
    ``--retrain-mode`` restores train mode after every test instead."""
    model.train()
    acc, old_name = 0.0, None
    sched = T.EpochCosineSchedule(base_lr=args.lr)
    opt.param_groups[0]["lr"] = sched.lr
    # The loader drops the last partial batch (vtab.py:84-88), so every step has the same shape: zero_grad + forward +
    # CE + backward (+ the gradient all-reduce and AdamW) are captured once into a CUDA graph and replayed (at the
    # reference's batch of 64 the launches of a step take longer to enqueue from Python than to run).
    step = None
    for epoch in range(epochs):
        for x, y in dl:
            x, y = to_device(x, y, size=args.img_size)
            if world_size > 1:
                lo, hi = T.shard_batch(x.shape[0], rank, world_size)
                x, y = x[lo:hi], y[lo:hi]
            if step is None and not args.no_graph:
                step = T.GraphedStep(model, opt, x, y, world_size)
            loss = step(x, y) if step is not None else T.train_step(model, opt, x, y, world_size)
            opt.param_groups[0]["lr"] = sched.after_step(epoch)
        if rank == 0:
            print(f"e: {epoch}, l: {round(float(loss), 7)}, a:{acc}", flush=True)
        if epoch % 10 == 0 and epoch != 0:
            sched.after_test(epoch)
            acc = test(model, tdl, args.img_size)
            if args.retrain_mode:
                model.train()
            step = None                       # the mode (dropout / DropPath kernels) is baked into the captured graph
            if acc > args.best_acc and rank == 0:
                args.best_acc = acc
                if old_name is not None:
                    os.remove(old_name)
                old_name = f"./vit_{args.dataset}_{round(acc, 5)}_seed_{args.seed}.pt"
                th.save(model.state_dict(), old_name)
    return model, old_name


def build_model(args, data_config, num_classes):
    """vit_cp.py:155-166 of the reference: backbone (+ ./ViT-B_16.npz), cara(), fresh classifier, on the GPU."""
    vit = create_model(args.model, checkpoint_path="./ViT-B_16.npz", drop_path_rate=0.1, img_size=args.img_size,
                       allow_missing_checkpoint=args.synthetic or args.allow_random_init)
    vit = cara({"model": vit, "rank": args.dim, "scale": data_config["scale"], "l_mu": data_config["init_mean"],
                "l_std": data_config["init_std"]})
    vit.reset_classifier(num_classes)
    vit = vit.cuda()
    set_weight_dropout(vit, args.weight_dropout)
    return vit


def load_for_evaluate(vit, path, merge=True):
    """The ``--evaluate`` branch (reference vit_cp.py:168-173): load a fine-tuned state_dict (the reference's own
    ``th.save(vit.state_dict())`` files load as they are: same 164 keys, nn.Linear [out,in] layout) and, unless
    ``--no-merge``, fold the CP delta into the frozen weights once with the reconstruction kernel."""
    vit.load_state_dict(th.load(path, map_location="cuda"))
    if merge:
        merge_cara(vit)
    return vit


def _parse_args(argv=None):
    p = ArgumentParser(formatter_class=ArgumentDefaultsHelpFormatter)
    p.add_argument("--dim", default=32, type=int, help="Number of trainable ranks.")
    p.add_argument("--lr", default=1e-3, type=float, help="Learning rate")
    p.add_argument("--dataset", default="svhn", type=str, choices=sorted(config), help="Dataset to train")
    p.add_argument("--evaluate", default=None, type=str, help="Evalute model only")
    p.add_argument("--model", type=str, default="vit_base_patch16_224_in21k")
    p.add_argument("--epochs", type=int, default=100)
    p.add_argument("--batch-size", type=int, default=64, help="global train batch")
    p.add_argument("--synthetic", action="store_true", help="force VTAB-shaped synthetic data")
    p.add_argument("--no-merge", action="store_true", help="evaluate without folding the CP delta into W")
    p.add_argument("--no-graph", action="store_true", help="enqueue every train step eagerly (no CUDA graph replay)")
    p.add_argument("--weight-dropout", default="exact", choices=["exact", "skip"],
                   help="exact: nn.Dropout(0.1) on the materialised CP delta in train mode, as the reference "
                        "(cara.py:35,57,81,92; slow path, cara_b200.wdrop); skip: fused fast path without it")
    p.add_argument("--retrain-mode", action="store_true",
                   help="call model.train() after each periodic test (the reference stays in eval mode, vit_cp.py:75)")
    p.add_argument("--allow-random-init", action="store_true",
                   help="keep the random initialisation when ./ViT-B_16.npz is missing (implied by --synthetic)")
    p.add_argument("--gpu-preprocess", action="store_true",
                   help="decode on the CPU, resize + normalise on the GPU (bit-identical to the reference's transforms)")
    p.add_argument("--img-size", default=None, type=int,
                   help="input resolution (default: the model's own, 224 for the *_224 models); a positive multiple "
                        "of the patch size, e.g. 384 for ViT-B/16 (577 tokens)")
    args = p.parse_args(argv)
    geom = _GEOMETRY.get(args.model, {})                  # (an unknown name is reported by create_model)
    patch = geom.get("patch_size", 16)
    if args.img_size is None:
        args.img_size = geom.get("img_size", 224)
    elif args.img_size <= 0 or args.img_size % patch != 0:
        p.error("--img-size %d is not a positive multiple of the patch size %d of %s" % (args.img_size, patch, args.model))
    return args


def main(sd=None):
    args = _parse_args()
    print(args)
    name = args.dataset
    data_config = config[name]
    seed = data_config["seed"] if sd is None else sd
    scale = data_config["scale"]
    args.best_acc = 0.0
    args.seed = seed
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    th.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        th.distributed.init_process_group("nccl")
    print(f"\n\nSeed: {seed}")
    np.random.seed(seed)
    random.seed(seed)
    th.manual_seed(seed)
    th.cuda.manual_seed_all(seed)

    train_dl, test_dl = get_data(name, evaluate=True, batch_size=args.batch_size,
                                 synthetic=True if args.synthetic else None, gpu_preprocess=args.gpu_preprocess,
                                 img_size=args.img_size)
    vit = build_model(args, data_config, get_classes_num(name))

    if args.evaluate is not None:
        print("Only evaluation")
        load_for_evaluate(vit, args.evaluate, merge=not args.no_merge)
        acc = test(vit, test_dl, args.img_size)
        print(f"Accuracy: {acc}")
        sys.exit(0)

    trainable = T.freeze_backbone(vit)
    print(f"Total parameters: {sum(p.numel() for n, p in trainable if 'head' not in n)}")
    print(vit.head)
    opt = T.FusedAdamW(T.FlatTrainable(trainable), lr=args.lr, weight_decay=1e-4)
    vit, old_name = train(args, vit, train_dl, test_dl, opt, args.epochs, world, rank)
    print("\n\n Evaluating....")
    acc = test(vit, test_dl, args.img_size)
    print(acc)
    if acc > args.best_acc and rank == 0:
        args.best_acc = acc
        if old_name is not None:
            os.remove(old_name)
        th.save(vit.state_dict(), f"./vit_{name}_{round(args.best_acc, 5)}_seed_{seed}.pt")
    if rank == 0:
        print(f"Accuracy: {args.best_acc}")


if __name__ == "__main__":
    main()
