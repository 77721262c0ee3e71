"""Per-tile timeline of the fused kernel from its own %globaltimer stamps (fm_set_trace): where the time of the expert-FFN
phase goes.  Usage: python scripts/trace_gantt.py [--cfg B] [--world-note ...]   (environment knobs FM_* apply).
Prints medians over the leader CTAs of: claim -> dependencies resolved -> first k-block landed -> last MMA issued ->
accumulator complete -> epilogue stores issued -> published, per GEMM kind, plus the idle gaps between tiles."""
import argparse
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from flashmoe_b200.config import BASELINE_CONFIGS, MoEConfig
from flashmoe_b200.runtime import MoEContext

CFGS = dict(BASELINE_CONFIGS)
CFGS["small"] = MoEConfig(num_experts=8, expert_top_k=2, sequence_len=512, hidden_size=256, intermediate_size=512)


def analyse(tr, cfg, label=""):
    tr = tr.astype(np.int64)
    t00 = tr[:, 0].min()
    us = lambda a: (a - t00) / 1e3  # noqa: E731
    names = {0: "start", 11: "gate_gemv", 10: "zero_issued", 15: "topk_warp0", 12: "gate_topk", 1: "gate_done", 2: "barrier", 8: "disp_prefix", 9: "disp_rows_done",
             3: "dispatch_end", 7: "first_tma_issued", 4: "ffn_start", 5: "ffn_end", 6: "kernel_end"}
    print(f"--- {label} phases (us after the first CTA's start; min / median / max over CTAs)")
    for i, nm in names.items():
        v = us(tr[:, i][tr[:, i] > 0])
        if len(v):
            print(f"  {nm:14s} {v.min():8.1f} {np.median(v):8.1f} {v.max():8.1f}")
    lead = tr[0::2]  # leader CTAs of the pairs hold the scheduler / MMA stamps
    part = tr[1::2]
    rows = []
    for c in range(lead.shape[0]):
        n = int((lead[c, 32:48] > 0).sum())
        for i in range(n):
            rows.append(dict(c=c, i=i, claim=lead[c, 112 + i], ready=lead[c, 16 + i], first=lead[c, 32 + i], last=lead[c, 48 + i],
                             acc=lead[c, 64 + i], stores=lead[c, 80 + i], pub=lead[c, 96 + i],
                             p_acc=part[c, 64 + i], p_stores=part[c, 80 + i], p_pub=part[c, 96 + i],
                             prev_last=lead[c, 48 + i - 1] if i else lead[c, 4], prev_acc=lead[c, 64 + i - 1] if i else 0))
    if not rows:
        print("  no tile stamps")
        return
    span = np.array([r["acc"] - r["first"] for r in rows]) / 1e3
    thr = 2.0 * np.median(span) if len(span) else 0
    nk = {0: cfg.H // 64, 1: cfg.P // 64}
    kinds = np.array([1 if s > 0.6 * span.max() and span.max() > 1.8 * span.min() else 0 for s in span])
    ffn0 = np.median(lead[:, 4][lead[:, 4] > 0])
    ffn_end = tr[:, 5].max()
    print(f"--- {label} tiles recorded (first 16 per pair): {len(rows)}; GEMM0-like {int((kinds == 0).sum())}, GEMM1-like {int((kinds == 1).sum())}")
    for kd in (0, 1):
        sel = [r for r, k in zip(rows, kinds) if k == kd]
        if not sel:
            continue
        f = lambda a, b: np.array([r[a] - r[b] for r in sel]) / 1e3  # noqa: E731
        main = f("acc", "first")
        issue = f("last", "first")
        print(f"  GEMM{kd} (nk={nk[kd]}): n={len(sel)}")
        for nm, v in (("claim->ready", f("ready", "claim")), ("ready->first k-block landed", f("first", "ready")),
                      ("first landed->last MMA issued", issue), ("first landed->accumulator complete", main),
                      ("  per k-block (us)", main / nk[kd]),
                      ("accumulator complete->stores issued (leader epi)", f("stores", "acc")),
                      ("stores issued->published (leader)", f("pub", "stores")),
                      ("accumulator complete->stores issued (partner epi)", f("p_stores", "p_acc")),
                      ("MMA idle before this tile (first landed - prev last issued)", f("first", "prev_last")),
                      ):
            v = v[np.isfinite(v)]
            print(f"    {nm:62s} med {np.median(v):7.2f}  p10 {np.percentile(v, 10):7.2f}  p90 {np.percentile(v, 90):7.2f}")
    t0rows = [r for r in rows if r["i"] == 0]
    if t0rows:
        g = lambda key: np.median([(r[key] - t00) / 1e3 for r in t0rows])  # noqa: E731
        print(f"  per pair, first tile: claimed {g('claim'):.1f}, rows ready {g('ready'):.1f}, first k-block landed {g('first'):.1f} us (medians)")
    # tensor-busy fraction per pair over the FFN phase (first 16 tiles only are stamped; config B has <= 10 per pair)
    busy = {}
    for r in rows:
        busy[r["c"]] = busy.get(r["c"], 0) + (r["acc"] - r["first"])
    b = np.array(list(busy.values())) / 1e3
    t_first = np.array([min(r["first"] for r in rows if r["c"] == c) for c in busy]) - t00
    t_lastacc = np.array([max(r["acc"] for r in rows if r["c"] == c) for c in busy]) - t00
    print(f"  per pair: mainloop-busy med {np.median(b):.1f} us; first k-block landed at med {np.median(t_first) / 1e3:.1f} "
          f"(min {t_first.min() / 1e3:.1f}, max {t_first.max() / 1e3:.1f}) us; last accumulator complete med {np.median(t_lastacc) / 1e3:.1f} max {t_lastacc.max() / 1e3:.1f} us; "
          f"kernel end {us(tr[:, 6].max()):.1f} us")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", default="B")
    ap.add_argument("--label", default="")
    ap.add_argument("--save", default="")
    args = ap.parse_args()
    cfg = CFGS[args.cfg]
    g = torch.Generator().manual_seed(0)
    x = torch.randn(cfg.mini_batch, cfg.sequence_len, cfg.H, generator=g).bfloat16().cuda()
    wg = torch.randn(cfg.H, cfg.E, generator=g).bfloat16().cuda()
    we = torch.randn(cfg.E, 2, cfg.P, cfg.H, generator=g).bfloat16().cuda()
    ctx = MoEContext(cfg, timeout_ms=5000)
    out = torch.empty_like(x)
    for _ in range(5):
        ctx.forward(x, wg, we, out=out)
    ctx.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        ctx.forward(x, wg, we, out=out)
    e1.record()
    ctx.synchronize()
    print(f"=== {args.label or args.cfg}: {e0.elapsed_time(e1) / 20 * 1e3:.1f} us / forward")
    ctx.set_trace(True)
    ctx.forward(x, wg, we, out=out)
    ctx.synchronize()
    tr = ctx.read("trace")
    if args.save:
        np.save(args.save, tr)
    analyse(tr, cfg, args.label or args.cfg)
    ctx.close()


if __name__ == "__main__":
    main()
