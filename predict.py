#!/usr/bin/env python
"""predict.py -- the reference's inference entry point (predict.py:19-40 flags, :138 checkpoint load, :142-194 metrics) over
the B200 path: forward-only fused kernels (no saved activations) + on-device MAE / RMSE / MAPE-vs-p95 (regt_eval_metrics).
Data and graph as in run.py of this repository; the matplotlib figure of the reference (--visualize) is not built."""
import argparse
import os.path as osp
import sys

ROOT = osp.dirname(osp.abspath(__file__))
for p in (ROOT, osp.join(ROOT, "regt-gcn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def build_parser() -> argparse.ArgumentParser:
    import run as R
    parser = R.build_parser()
    # predict.py:37-39 adds these two and drops the --is_pre* / --pretrained_model* group (kept here: harmless)
    parser.add_argument("--pretrained_idx", default="30", type=str, help="Pretrained index num")
    parser.add_argument("--visualize", type=bool, default=False, help="Flag for network visualization (not built)")
    return parser


def main(argv=None):
    args = build_parser().parse_args(argv)
    import torch
    import run as R
    from models import RegionalTemporalGCN, TemporalGCN
    from regt_b200 import workloads as W
    from regt_b200.loop import SlidingWindows, evaluate
    if not torch.cuda.is_available():
        raise SystemExit("predict.py needs a CUDA device: this repository has no CPU path")
    device = torch.device("cuda:0")
    full, rei, rea, N = W.tpims_graph()
    if args.model == "RegionalTemporalGCN":
        model = RegionalTemporalGCN(node_features=8, num_nodes=N, periods=args.num_timesteps_in, output_dim=args.num_timesteps_out,
                                    hidden=args.hidden, precision=args.precision)
        graph = (full, *rei, *rea)
    elif args.model == "TemporalGCN":
        model = TemporalGCN(node_features=8, periods=args.num_timesteps_in, output_dim=args.num_timesteps_out, hidden=args.hidden,
                            precision=args.precision)
        graph = (full, torch.cat(rea))
    else:
        raise SystemExit(f"--model {args.model}: only RegionalTemporalGCN and TemporalGCN are on this repository's path")
    model = model.to(device)
    ck = osp.join("pretrained", args.tf, args.model, "model_in{}_out{}_epoch{}.pt".format(
        args.num_timesteps_in, args.num_timesteps_out, int(args.pretrained_idx)))                      # predict.py:138
    model.load_state_dict(torch.load(ck, map_location=device))
    graph = tuple(g.to(device) for g in graph)
    nd, _ = R.load_series(args, N)
    windows = SlidingWindows(nd.to(device), args.num_timesteps_in, args.num_timesteps_out)
    n_train = int(args.tr * len(windows))
    mae, rmse, mape = evaluate(model, windows, graph, n_train, len(windows), batch=max(1, args.bs),    # predict.py:142-194
                               share_periods=args.share_periods)
    print(f"Test Results: RMSE: {rmse}, MAE: {mae}, MAPE: {mape}")                                     # predict.py:252
    return mae, rmse, mape


if __name__ == "__main__":
    main()
