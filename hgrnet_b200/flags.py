"""Command-line surface: every flag of the reference's ``main.py`` (main.py:16-68) with the
same name, default and type -- including the ``type=eval`` booleans (``--train False``) and the
three flags the reference parses but never reads (``--debug``, ``--template``,
``--num_workers``; SURVEY.md section 5) -- plus a small ``hgr_*`` group for this build.
"""
from __future__ import annotations

import argparse


def _bool(s):  # the reference uses type=eval for True/False flags (main.py:41,46,47)
    if isinstance(s, bool):
        return s
    if s in ("True", "true", "1"):
        return True
    if s in ("False", "false", "0"):
        return False
    raise argparse.ArgumentTypeError("expected True or False, got %r" % (s,))


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(description="HGR")
    p.add_argument("--exp_name", default="HGR", type=str)
    p.add_argument("--folder", default="adaptive", type=str)
    p.add_argument("--device", default=0, type=int)
    p.add_argument("--print_freq", default=1000, type=int)
    p.add_argument("--debug", default=False, action="store_true")
    p.add_argument("--test_after_train", default=False, action="store_true")
    # model
    p.add_argument("--arch", default="RN50", type=str)
    # imagenet
    p.add_argument("--template", default="TEMPLATES_STANDARD", type=str)
    p.add_argument("--model_train", default="all", type=str)
    p.add_argument("--model_test", default="rest", type=str)
    p.add_argument("--data_train", default="train", type=str)
    p.add_argument("--data_test", default="rest", type=str)
    # data
    p.add_argument("--graph_path", default="data/process_results/graph_edges_cls.json", type=str)
    p.add_argument("--split_path", default="data/process_results/splits_for_tree.json", type=str)
    p.add_argument("--num_workers", default=12, type=int)
    p.add_argument("--batch_size", default=256, type=int)
    p.add_argument("--test_batch_size", default=512, type=int)
    p.add_argument("--k_shots", default=-1, type=int)
    p.add_argument("--serial_batches", type=_bool, default=True, choices=[True, False])
    p.add_argument("--n_episodes", default=-1, type=int)
    p.add_argument("--data_split_train", default="train", type=str, help="train, ls_train")
    p.add_argument("--data_split_test", default="zsl_test", type=str, help="val, ls_test, zsl_test")
    # train
    p.add_argument("--open_eval", type=_bool, default=True, choices=[True, False])
    p.add_argument("--train", default=True, type=_bool, choices=[True, False])
    p.add_argument("--lr", default=3e-7, type=float)
    p.add_argument("--w_lr", default=1e-4, type=float)
    p.add_argument("--epochs", default=10, type=int)
    p.add_argument("--wd", default=0.0, type=float)
    p.add_argument("--warmup_length", default=0, type=int)
    p.add_argument("--num_compare", default=256, type=int)
    p.add_argument("--weights", default="adaptive", type=str,
                   help="equal, increasing, decreasing, adaptive, nl_increasing, nl_decreasing")
    p.add_argument("--training_method", default="OM", type=str, help="flat, hierarchical, OM")
    p.add_argument("--sample_strategy", default="topk", type=str, help="random, simi, topk, brothers")
    p.add_argument("--k", default=1, type=int)
    p.add_argument("--out_ratio", default=0.25, type=float, help="0.0, 0.25, 0.5, 0.75, 1.0")
    p.add_argument("--in_ratio", default=0.5, type=float, help="0.0, 0.25, 0.5, 0.75, 1.0")
    p.add_argument("--weighting", default="both", type=str, help="in,out")
    p.add_argument("--scale", default=1.0, type=float)
    # resume
    p.add_argument("--fetch", default=False, action="store_true")
    p.add_argument("--fetch_path", type=str)
    p.add_argument("--load", default=False, action="store_true")
    p.add_argument("--load_path", default="none", type=str)
    p.add_argument("--from_epoch", default=-1, type=int)
    # ---- additions of this build (all default to the reference's behaviour) ----
    g = p.add_argument_group("hgrnet_b200")
    g.add_argument("--hgr_bank", default="node", choices=["node", "chain"],
                   help="class bank: 'node' = one normalised text embedding per node (the reference, "
                        "clip_tree.py:318-325); 'chain' = hierarchy-aggregated (out_ratio/--weights over the "
                        "ancestor chain) through the CSR aggregation kernel")
    g.add_argument("--hgr_hier_metrics", type=_bool, default=True, choices=[True, False],
                   help="also compute TOR/POR (hit_ratio/path_ratio/point_ratio, main.py:152-191) during test")
    g.add_argument("--hgr_synthetic", default="", type=str,
                   help="run on a synthetic hierarchy and synthetic features, e.g. '10,100,1000' level sizes")
    g.add_argument("--hgr_eval_splits", default="", type=str,
                   help="comma-separated split-file keys (e.g. 2-hops,3-hops,all): test scores every batch against all of "
                        "them in one pass and prints one line per split")
    g.add_argument("--hgr_mistake_metrics", type=_bool, default=False, choices=[True, False],
                   help="also report the mistake rate, the mistake severity (mean LCA height of the wrong top-1) and "
                        "the LCA distance@k of the top-k during test, per split with --hgr_eval_splits")
    g.add_argument("--hgr_class_metrics", type=_bool, default=False, choices=[True, False],
                   help="also report the class-averaged Hit@k (the mean over the classes with test rows of each "
                        "class's Hit@k / rows) during test, per split with --hgr_eval_splits")
    return p


def parse_args(argv=None):
    return build_parser().parse_args(argv)
