#!/usr/bin/env python
"""Input-gradient benchmark at the C4 shape (128x128, batch 64, Cin = 7 + season label, running-statistics BatchNorm, frozen model):

  * the stem data-gradient kernel alone (sbgm_stem_dgrad_tc), warm, CUDA events, and its HBM traffic over the time against the
    7.7 TB/s of the B200 data sheet (df read once per 16-bit plane, dx and dplanes written once, fp32);
  * one forward + input-VJP call, torch.autograd.grad(score, [x, cond_img, lsm_cond, topo_cond], v): eager and replayed from the
    captured graphs;
  * the full training step (loss_fn -> backward, trainable parameters, train-mode BatchNorm) on the same card.

    python tools/bench_input_grad.py [--precision bf16|bf16x3] [--iters 20] [--out FILE]

Prints one JSON line (also written to FILE) with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch

HBM_BYTES_PER_S = 7.7e12


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        return [s.strip() for s in q.split(",")]
    except Exception as exc:                          # the measurement stands without it; say so in the output
        return [torch.cuda.get_device_name(0), f"unknown ({type(exc).__name__})", "unknown"]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_input_grad.py measures on the GPU; no CUDA device found")
    import __graft_entry__
    __graft_entry__.build()
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import _lib, score_sampling
    from sbgm_danra_b200._lib import FMT_BF16X2, call
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.engine import Act
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    from sbgm_danra_b200.train_engine import TRAIN_PRECISIONS, PackPlan, stem_dgrad_weight

    dev, n, s = "cuda:0", args.batch, args.size
    ck = dict(n_lr=2, geo=True, seasons=True)
    cfg = config_for(**ck)
    sd = synth_state_dict(cfg)
    b = synth_batch(batch=n, size=s, **ck)
    c = lambda v: None if v is None else v.to(dev)
    x, y, cond, lsm, topo, sdf = (c(v) for v in (b.x, b.y, b.cond_img, b.lsm_cond, b.topo_cond, b.sdf_cond))
    t = torch.linspace(0.2, 0.9, n, device=dev)
    v = torch.randn(n, 1, s, s, device=dev)
    res = {"metric": "input_grad_c4", "precision": args.precision, "batch": n, "size": s}

    # stem data gradient alone
    fmt = TRAIN_PRECISIONS[args.precision]
    cin = sd["encoder.conv1.weight"].shape[1]
    cc = cin - 1
    df = Act.from_nchw(torch.randn(n, 64, s // 2, s // 2, device=dev), fmt)
    plan = PackPlan(fmt)
    table = stem_dgrad_weight(plan, sd["encoder.conv1.weight"].to(dev))
    plan.run()
    dx = torch.empty(n, 1, s, s, device=dev)
    dpl = torch.empty(n, cc, s, s, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    us = 1e3 * timed(lambda: call("sbgm_stem_dgrad_tc", df.ptr, df.plane, fmt, table.data_ptr(), table.stride(1), dx.data_ptr(),
                                  dpl.data_ptr(), n, cc, n, s, s, None, st), 200)
    planes = 2 if fmt == FMT_BF16X2 else 1
    traffic = planes * n * (s // 2) ** 2 * 64 * 2 + n * cin * s * s * 4
    res.update(stem_dgrad_us=round(us, 2), stem_dgrad_MB=round(traffic / 1e6, 1), stem_dgrad_GBps=round(traffic / us / 1e3, 1),
               stem_dgrad_share_of_hbm_bound=round(traffic / HBM_BYTES_PER_S / (us * 1e-6), 3))

    # forward + input VJP, frozen model, eager and replayed
    net = build_model(cfg, sd, args.precision, dev).requires_grad_(False)

    def vjp():
        leaves = [a.detach().requires_grad_() for a in (x, cond, lsm, topo)]
        return torch.autograd.grad(net(leaves[0], t, y, *leaves[1:]), leaves, v)

    os.environ["SBGM_B200_TRAIN_GRAPHS"] = "0"
    res["vjp_eager_ms"] = round(timed(vjp, args.iters), 3)
    os.environ["SBGM_B200_TRAIN_GRAPHS"] = "1"
    net._train_runners.clear()
    res["vjp_graph_ms"] = round(timed(vjp, args.iters), 3)
    del net
    net = build_model(cfg, sd, args.precision, dev).train()
    score_sampling.manual_seed(0)

    def train_step():
        net.zero_grad(set_to_none=True)
        loss_fn(net, x, marginal_prob_std_fn, y=y, cond_img=cond, lsm_cond=lsm, topo_cond=topo, sdf_cond=sdf).backward()

    res["train_step_ms"] = round(timed(train_step, args.iters), 3)
    name, power, clock = card()
    res.update(gpu=name, power_limit=power, max_sm_clock=clock)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
