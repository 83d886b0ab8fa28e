#!/usr/bin/env python
"""run.py -- the reference's training entry point (run.py:22-45 flags, :115-120 model switch, :140-145 checkpoint load and
RMSprop, :163-243 epoch loop and checkpoint names) over the B200 path of this repo.

Only the two models on the hot path are built (``--model RegionalTemporalGCN`` with ``--dataloading_type 2``, and
``--model TemporalGCN``); the other names of the reference's switch are refused.  The reference's data files are not
shipped (``dataset/processed/.../tpims_data_small.pkl`` is a missing large blob, SURVEY section 2 #11), so the node series
comes from ``--dataset_path`` when it holds ``node_data.npy`` ([N, 8, T_total] float32, MinMax-scaled as
load_dataset.py:430 leaves it) and is synthetic U[0,1) otherwise; the graph is the TPIMS topology of the reference's link
CSVs (committed fixture).  The epoch runs on the device (regt_b200/loop.py): gradients of all training snapshots accumulate,
ONE RMSprop step per epoch (run.py:190-195), test RMSE / MSE over the held-out snapshots (run.py:202-226; the value the
reference prints as "MAE" is the MSE, SURVEY 3.3).
"""
import argparse
import os
import os.path as osp
import sys

ROOT = osp.dirname(osp.abspath(__file__))
for p in (ROOT, osp.join(ROOT, "regt-gcn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def build_parser() -> argparse.ArgumentParser:
    """the reference's flag set, verbatim (run.py:24-44), plus additive ones at the end."""
    parser = argparse.ArgumentParser()
    parser.add_argument("--seed", default=42, type=int, help="seed number")
    parser.add_argument("--epochs", default=30, type=int, help="Max epochs")
    parser.add_argument("--lr", default=1e-3, type=float, help="Learning rate")
    parser.add_argument("--decay", default=1e-4, type=float, help="Weight decay")
    parser.add_argument("--momentum", default=0.9, type=float, help="Momentum (parsed and unused, as in the reference)")
    parser.add_argument("--bs", "--batch_size", default=32, type=int,
                        help="Batch size (unused by the reference; here: snapshots per fused step)")
    parser.add_argument("--tr", "--train_ratio", default=0.8, type=float, help="Train ratio")
    parser.add_argument("--tf", "--train_feature", default="available", type=str, help="Train feature (occrate / avaialble)")
    parser.add_argument("--edge_cut", default=None, type=str, help="The type of edge cut (random/neural/None)")
    parser.add_argument("--dataset_path", default="./dataset", type=str, help="Dataset path")
    parser.add_argument("--checkpoint_path", default="../checkpoints/", type=str, help="Checkpoints path")
    parser.add_argument("--dataloading_type", default=2, type=int, help="Dataset number (Truckparking dataset '1' / '2')")
    parser.add_argument("--decomp_type", default=None, type=str, help="Regional or Random decomposition type")
    parser.add_argument("--num_timesteps_in", default=8, type=int, help="Number of timesteps for input")
    parser.add_argument("--num_timesteps_out", default=4, type=int, help="Number of timesteps for output")
    parser.add_argument("--model", default="TemporalGCN", type=str, help="RegionalTemporalGCN | TemporalGCN")
    parser.add_argument("--is_preprocessed", action="store_true", help="If the dataset is preprocessed")
    parser.add_argument("--is_pretrained", action="store_true")
    parser.add_argument("--pretrained_model", default="", type=str, help="Pretrained model name")
    parser.add_argument("--pretrained_model_epoch", default="0", type=str, help="Pretrained model epochs")
    parser.add_argument("--logs", action="store_true")
    # additive (reference defaults reproduce the reference)
    parser.add_argument("--hidden", default=256, type=int, help="hidden width (reference: 256)")
    parser.add_argument("--precision", default="auto", type=str, help="auto | fp32 | tf32x3 | bf16")
    parser.add_argument("--share_periods", action="store_true",
                        help="run the cell once per time step of a batch of windows and share it across them (exact in real "
                             "arithmetic, sums in another order; off: every window runs its own periods)")
    parser.add_argument("--synthetic_steps", default=600, type=int, help="length of the synthetic series when no node_data.npy is found")
    return parser


def load_series(args, N: int):
    import numpy as np
    import torch
    path = osp.join(args.dataset_path, "node_data.npy")
    if osp.exists(path):
        nd = torch.from_numpy(np.load(path).astype("float32"))
        if nd.dim() != 3 or nd.shape[0] != N or nd.shape[1] != 8:
            raise SystemExit(f"{path}: expected [N={N}, 8, T_total], got {tuple(nd.shape)}")
        return nd, path
    g = torch.Generator().manual_seed(args.seed)
    return torch.rand(N, 8, args.synthetic_steps, generator=g), "synthetic U[0,1)"


def main(argv=None):
    args = build_parser().parse_args(argv)
    import torch
    from models import RegionalTemporalGCN, TemporalGCN
    from regt_b200 import workloads as W
    from regt_b200.loop import FlatRMSprop, SlidingWindows, evaluate, train_epoch

    torch.manual_seed(args.seed)                                                       # run.py:69-71
    if not torch.cuda.is_available():
        raise SystemExit("run.py needs a CUDA device: this repository has no CPU path (use the reference for CPU runs)")
    device = torch.device("cuda:0")                                                    # run.py:73
    full, rei, rea, N = W.tpims_graph()
    if args.model == "RegionalTemporalGCN":
        if args.dataloading_type != 2:
            raise SystemExit("RegionalTemporalGCN needs --dataloading_type 2 (regional edge lists), as in run.py:94-106")
        model = RegionalTemporalGCN(node_features=8, num_nodes=N, periods=args.num_timesteps_in,
                                    output_dim=args.num_timesteps_out, hidden=args.hidden, precision=args.precision)   # run.py:116
        graph = (full, *rei, *rea)
    elif args.model == "TemporalGCN":
        model = TemporalGCN(node_features=8, periods=args.num_timesteps_in, output_dim=args.num_timesteps_out,
                            hidden=args.hidden, precision=args.precision)                                              # run.py:120
        graph = (full, torch.cat(rea))
    else:
        raise SystemExit(f"--model {args.model}: only RegionalTemporalGCN and TemporalGCN are on this repository's path "
                         "(the reference's other baselines are out of scope, DESIGN.md section 9)")
    model = model.to(device)
    pretrained_idx = 0
    ck_dir = osp.join("pretrained", args.tf, args.model)
    if args.is_pretrained:                                                             # run.py:140-142
        state = torch.load(osp.join(ck_dir, args.pretrained_model), map_location=device)
        model.load_state_dict(state)                                                   # strict, as the reference
        pretrained_idx = int(args.pretrained_model_epoch)
    graph = tuple(g.to(device) for g in graph)
    nd, src = load_series(args, N)
    windows = SlidingWindows(nd.to(device), args.num_timesteps_in, args.num_timesteps_out)
    n_train = int(args.tr * len(windows))                                              # temporal_signal_split, run.py:111
    print(f"{args.model}: N={N} T_in={args.num_timesteps_in} T_out={args.num_timesteps_out} hidden={args.hidden} "
          f"precision={model.precision}; series: {src}; {n_train} train / {len(windows) - n_train} test snapshots")
    opt = FlatRMSprop(list(model.parameters()), lr=args.lr, weight_decay=args.decay, skip=model.dead_parameters())   # run.py:145
    for epoch in range(args.epochs + 1):                                               # run.py:230
        last_loss, _ = train_epoch(model, windows, graph, opt, 0, n_train, batch=max(1, args.bs), share_periods=args.share_periods)
        mae, rmse, _ = evaluate(model, windows, graph, n_train, len(windows), batch=max(1, args.bs),
                                share_periods=args.share_periods)
        print("Train Loss: {:.4f}, Test RMSE: {:.4f}, MAE: {:.4f}".format(float(last_loss), rmse, rmse * rmse))      # run.py:236
        if epoch % 10 == 0:                                                            # run.py:242-243
            os.makedirs(ck_dir, exist_ok=True)
            torch.save(model.state_dict(), osp.join(ck_dir, "model_in{}_out{}_epoch{}.pt".format(
                args.num_timesteps_in, args.num_timesteps_out, pretrained_idx + epoch)))
    return 0


if __name__ == "__main__":
    sys.exit(main())
