#!/usr/bin/env python
"""filter.py — drop-in for /root/reference/filter.py (same argv, same files), B200-native.

    python -u filter.py --dataset D --model M --checkpoint "D_M||0|0.pt"        (submit_job.py:20-21)

Reads ``models/{checkpoint}`` (a LinkGNN state_dict in the reference's layout) when the model has
parameters, optionally ``filtered_edges/{sorted_edge_path}.pt`` when the checkpoint name encodes
extra edges, and writes ``filtered_edges/{spec}_{sorted_edge_path}_{num}_{run}_sorted_edges.pt``:
a float32 ``[E,3]`` tensor of (u, v, score) sorted by score descending (filter.py:160-165).

Differences from the reference, all on the fast side of the same semantics:
  * candidates are enumerated on the GPU (K6), scored in one launch per slab (K2 / K3) with the GNN
    embeddings computed once, and ordered by K4 with the deterministic tie rule
    "score desc, then (v, u) asc" (the reference's unstable CPU sort leaves ties arbitrary);
  * ``--topk K`` keeps only the first K rows (rank.py only ever reads a prefix, rank.py:294);
    without it every candidate is written, like the reference;
  * with ``--topk`` a GNN filter scores every candidate on the tcgen05 tensor cores (fp16 operands) and
    re-scores the band around the k-th score in fp32: the saved list is the fp32 list, bit for bit
    (``--mlp_precision``, filter_step.filter_topk_multi);
  * ``--per_node_topk M`` keeps only the M best candidates (u, v) of every node v (score descending, ties by u):
    every node gets proposals, not just the neighbourhoods of the hubs, and the list has at most n * M rows.  The
    kept rows are ordered like the global list (and cut to ``--topk`` when given), so the file is read the same way.
    The budget belongs to v, the second column; (v, u) need not be in u's list (the rank graph is symmetrised, so
    either row adds the undirected edge);
  * under ``torchrun`` the owners are sharded across the GPUs and merged with one all-gather.
"""
from __future__ import annotations

import argparse
import os
from pathlib import Path

import torch


def _budget(text: str) -> int:
    m = int(text)
    if m < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1 (got {m})")
    return m


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="filter step (B200-native)")
    p.add_argument("--dataset", type=str, required=True)
    p.add_argument("--model", type=str, required=True)
    p.add_argument("--checkpoint", type=str, required=True)
    # model configs; overwrite defaults if specified (reference flags, incl. its type=bool quirk)
    p.add_argument("--num_layers", type=int)
    p.add_argument("--hidden_channels", type=int)
    p.add_argument("--dropout", type=float)
    p.add_argument("--batch_size", type=int)
    p.add_argument("--lr", type=float)
    p.add_argument("--epochs", type=int)
    p.add_argument("--use_feature", type=bool)
    p.add_argument("--use_learnable_embedding", type=bool)
    p.add_argument("--device", type=int, default=0)
    # additions
    p.add_argument("--topk", type=int, default=None, help="keep only the K best rows (default: all)")
    p.add_argument("--mlp_precision", choices=["prefilter", "fp32", "f16", "bf16"], default="prefilter",
                   help="GNN filters: 'prefilter' = tcgen05 fp16-operand scores select a band around the top-k that is "
                        "re-scored in fp32 (the fp32 list, bit for bit); 'fp32' = FFMA arm for every candidate; "
                        "'f16' (alias 'bf16') = tensor-core scores only (approximate list)")
    p.add_argument("--per_node_topk", type=_budget, default=None, metavar="M",
                   help="per-node proposal budget: keep only the M best candidates (u, v) of every node v, then order "
                        "them like the global list (and keep the first --topk rows when given); default: off")
    p.add_argument("--slab_pairs", type=int, default=1 << 27)
    p.add_argument("--random_init", action="store_true",
                   help="score with seeded random weights when models/{checkpoint} does not exist")
    return p.parse_args(argv)


def main(argv=None):
    from edge_proposal_sets_b200 import _lib, filter_step
    from edge_proposal_sets_b200.data import get_data
    from edge_proposal_sets_b200.graph import add_edges
    from edge_proposal_sets_b200.models import build_model, default_model_configs

    args = default_model_configs(parse_args(argv))
    print(args)
    Path("filtered_edges").mkdir(exist_ok=True)
    if not torch.cuda.is_available():
        raise SystemExit("filter.py: no CUDA device (this build has no CPU fallback)")
    _lib.load()
    distributed = int(os.environ.get("WORLD_SIZE", "1")) > 1
    local = int(os.environ.get("LOCAL_RANK", args.device))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if distributed:
        torch.distributed.init_process_group("nccl", device_id=device)
    rank = torch.distributed.get_rank() if distributed else 0

    edge_index, edge_weight, split_edge, data = get_data(args, device)
    model = build_model(args, data, device)
    print(f"using model {model}")
    use_params = sum(p.numel() for p in model.parameters() if p.requires_grad) > 0
    print("using params?", use_params)
    if use_params:
        path = f"models/{args.checkpoint}"
        if os.path.exists(path):
            model.load_state_dict(torch.load(path, map_location=device))
        elif args.random_init:
            torch.manual_seed(1234)
            model.reset_parameters()
        else:
            raise FileNotFoundError(f"{path} (train it with rank.py --save_models, or pass --random_init)")
    model.eval()

    spec, sorted_edge_path, num_sorted_edge, run = args.checkpoint.split("|")[:4]
    num_sorted_edge, run = int(num_sorted_edge), run.split(".")[0]
    name = "collab" if args.dataset.startswith("collab") else args.dataset
    extra = torch.zeros([2, 0], dtype=torch.long)
    if sorted_edge_path:
        print("Loading corresponding extra edges from ", sorted_edge_path)
        print(f"Using {num_sorted_edge} highest scoring edges")
        extra = filter_step.load_extra_edges(f"filtered_edges/{sorted_edge_path}.pt", num_sorted_edge)
    data.adj_t = add_edges(name, edge_index.to(device), edge_weight.to(device), extra.to(device), data.num_nodes)

    ra_adj = None
    if args.model == "resource_allocation":       # filter.py:130-139 rebuilds A from the raw train split
        ra_adj = filter_step.ra_graph_from_train_edges(split_edge["train"]["edge"].to(device), data.num_nodes)
    stats = {}
    k = args.topk
    if distributed and k is None:
        raise SystemExit("filter.py: --topk is required under torchrun (only top-k lists are merged)")
    sorted_edges = filter_step.filter_topk(args.model, model, data.x, data.adj_t, k=k, slab_pairs=args.slab_pairs,
                                           distributed=distributed, ra_adj=ra_adj, stats=stats,
                                           per_node=args.per_node_topk).cpu()
    print(f"using {stats.get('candidates_scored')} edges" + (" (this rank)" if distributed else ""))
    if rank == 0:
        print(sorted_edges)
        filename = f"filtered_edges/{spec}_{sorted_edge_path}_{num_sorted_edge}_{run}_sorted_edges.pt"
        torch.save(sorted_edges, filename)
        print("Saving to ", filename)
    if distributed:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
