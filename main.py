#!/usr/bin/env python
"""Entry point with the reference's flag surface (main.py of WilliamYi96/HGR-Net), hosted on hgrnet_b200.

    python main.py --train False [--hgr_synthetic 10,100,1000] ...

The drivers mirror the reference's ``main()`` / ``train()`` / ``test()`` (main.py:72-267); the hot path
behind ``tree_model`` runs in libhgr_b200.so.  Real-data runs need the upstream producers that are out of
scope here (an OpenAI-CLIP compatible ``clip`` package with weights, and the reference's ``dataset`` package
with ImageNet-21K on disk); ``--hgr_synthetic L0,L1,...`` replaces them by a synthetic hierarchy with those
level sizes, a table-lookup text encoder and random image features, so that the whole loop can be exercised.
"""
from __future__ import annotations

import json
import sys

import torch

from hgrnet_b200 import evaluate
from hgrnet_b200.flags import build_parser


def cosine_lr(optimizer, base_lr, warmup_length, steps):
    """utils.py:82-95."""
    import math

    def _adjust(step):
        for group in optimizer.param_groups:
            if step < warmup_length:
                lr = base_lr * (step + 1) / warmup_length
            else:
                lr = 0.5 * (1 + math.cos(math.pi * (step - warmup_length) / max(1, steps - warmup_length))) * base_lr
            group["lr"] = lr
    return _adjust


def train(opts, epoch, model, train_loader, num_batches, optimizer, optimizer2, scheduler, device):
    """main.py:72-101.  ``optimizer`` is a ``hgrnet_b200.optim.MasterStepper``: the reference's fp32-cast / step / fp16-cast
    sequence (main.py:90-94) on persistent fp32 masters instead of two whole-model re-allocations per step."""
    if not opts.open_eval:
        model.train()
    for i, data in enumerate(train_loader):
        scheduler(i + epoch * num_batches)
        imgs, targets = data["img"][0].to(device), data["label"][0].to(device)
        loss = model.train_batch(imgs, targets, opts.training_method, opts.sample_strategy)
        params = [p for name, p in model.named_parameters() if p.requires_grad and name != "layer_weight" and p.grad is not None]
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        optimizer.step()
        if opts.weights == "adaptive" and optimizer2 is not None:
            optimizer2.step()
        if i % opts.print_freq == 0:
            out_str = "loss: {:.2f}, {}/{}".format(loss, i, num_batches)
            print(out_str, flush=True)
            with open(model.save_path + "arugements.log", "a") as f:
                f.writelines(out_str + "\n")


def _synthetic_setup(opts, device):
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.hierarchy import synthetic_hierarchy
    from hgrnet_b200.synthetic import FeatureLoader, TableEncoder, node_id_tokens, synthetic_embeddings
    levels = [int(x) for x in opts.hgr_synthetic.split(",")]
    hier = synthetic_hierarchy(levels, seed=1)
    n = len(hier)
    dim = 1024 if opts.arch == "RN50" else 512
    enc = TableEncoder(synthetic_embeddings(n, dim, 1, normalize=False)).to(device)
    leaves = hier.nodes[n - levels[-1]:]
    # two seeded nested splits of the leaves (the shape of the 2-hops / 3-hops sets inside "rest"), for --hgr_eval_splits
    order = torch.randperm(len(leaves), generator=torch.Generator().manual_seed(5)).tolist()
    hops3 = [leaves[i] for i in sorted(order[:max(1, len(leaves) // 2)])]
    hops2 = [leaves[i] for i in sorted(order[:max(1, len(leaves) // 8)])]
    splits = {"train": hier.nodes, "rest": leaves, "all": hier.nodes, "hops2": hops2, "hops3": hops3}
    model = tree_model(opts, splits[opts.model_train], splits[opts.model_test], clip_model=enc, hierarchy=hier,
                       node_tokens=node_id_tokens(n))
    g = torch.Generator().manual_seed(3)
    test_ids = [hier.index[c] for c in splits[opts.data_test]]
    nb = 8
    def loader(batch):
        labels = [test_ids[int(torch.randint(0, len(test_ids), (1,), generator=g))] for _ in range(nb)]
        feats = [synthetic_embeddings(batch, dim, 50 + i, normalize=False) for i in range(nb)]
        return FeatureLoader(feats, labels)
    return model, splits, loader


def main(argv=None):
    parser = build_parser()
    opts = parser.parse_args(argv)
    device = "cuda:{}".format(opts.device)
    if opts.hgr_synthetic:
        print("Creating models (synthetic hierarchy / encoders)")
        model, splits, make_loader = _synthetic_setup(opts, device)
        loader_test = make_loader(opts.test_batch_size)
        loader_train, num_batches = make_loader(opts.batch_size), 8
    else:
        splits = json.load(open(opts.split_path, "r"))
        print("Creating models")
        from hgrnet_b200.head import tree_model
        model = tree_model(opts, candidates_train=splits[opts.model_train], candidates_test=splits[opts.model_test])
        try:
            from dataset import DataManager, DataManager_test  # the reference's loaders (upstream, out of scope)
        except ImportError as e:
            raise SystemExit("real-data runs need the reference's `dataset` package on PYTHONPATH (image I/O is an "
                             "upstream component); use --hgr_synthetic to exercise the head without it") from e
        loader_test = DataManager_test(opts=opts, split=opts.data_split_test, node_set=model.nodes,
                                       candidates=splits[opts.data_test], resolution=model.resolution).get_data_loader()
        data = DataManager(opts=opts, split=opts.data_split_train, node_set=model.nodes,
                           candidates=splits[opts.data_train], resolution=model.resolution)
        loader_train, num_batches = data.get_data_loader(), data.n_episodes

    if opts.train:
        with open(model.save_path + "arugements.log", "a") as f:           # main.py:232-237
            for k, v in vars(opts).items():
                f.writelines(k + " : " + str(v) + "\n")
        print("Training.")
        params = [p for name, p in model.named_parameters() if p.requires_grad and name != "layer_weight"]
        from hgrnet_b200.optim import MasterStepper
        optimizer = MasterStepper(params, lambda ps: torch.optim.AdamW(ps, lr=opts.lr, weight_decay=opts.wd))
        optimizer2 = torch.optim.SGD([model.layer_weight], lr=opts.w_lr) if opts.weights == "adaptive" else None
        scheduler = cosine_lr(optimizer, opts.lr, opts.warmup_length, opts.epochs * num_batches)
        for epoch in range(opts.from_epoch + 1, opts.epochs):
            train(opts, epoch, model, loader_train, num_batches, optimizer, optimizer2, scheduler, device)
            model.save(opts, epoch)
            print("Model saved.")
            if opts.test_after_train:
                evaluate.test(opts, model, device, splits, loader=loader_test)
    else:
        print("Direct testing.")
        evaluate.test(opts, model, device, splits, loader=loader_test)


if __name__ == "__main__":
    sys.exit(main())
