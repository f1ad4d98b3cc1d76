#!/usr/bin/env python
"""Micro-benchmark of every hand-written kernel at the BASELINE shapes (1 GPU).

    python tools/kernel_bench.py [--only k2,k3,...] [--iters 20] [--json out.json]

Each kernel is timed with CUDA events on the launching stream over ROTATING operand sets whose
total size exceeds the 126 MB L2 (so every launch streams from HBM), after 3 warm-up launches.
Reported: average launch time, algorithmic bytes, achieved GB/s and the fraction of the measured
copy bandwidth in MEASURED_PEAKS.json.  Under ``ncu`` (profiles/) pass ``--iters 2``.
"""
import argparse
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

import frl_b200  # noqa: E402,F401
from frl_b200 import _native, criteria  # noqa: E402

DEV = torch.device("cuda", 0)
L2_BYTES = 126 << 20


def peak_gbs():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    return json.load(open(p))["hbm_gbs"] if os.path.exists(p) else 6650.0


WARMUP = 3
MAX_SETS = 0          # > 0: cap the number of rotating operand sets (ncu runs)


def timed(name, fn_of_set, n_sets, bytes_per_launch, iters, note=""):
    for i in range(WARMUP):
        fn_of_set(i % n_sets)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn_of_set(i % n_sets)
    e1.record()
    torch.cuda.synchronize()
    us = 1e3 * e0.elapsed_time(e1) / iters
    gbs = bytes_per_launch / us / 1e3
    rec = {"kernel": name, "us": round(us, 2), "bytes": int(bytes_per_launch), "GBps": round(gbs, 1),
           "frac_of_measured_hbm": round(gbs / peak_gbs(), 3), "sets": n_sets, "note": note}
    print(json.dumps(rec), flush=True)
    return rec


def sets_for(bytes_per_set):
    n = max(2, -(-2 * L2_BYTES // max(bytes_per_set, 1)))
    return min(n, MAX_SETS) if MAX_SETS > 0 else n


def bench_k2(iters):
    out = []
    # AdamW next to Adam: same bytes (28 B/param), one more multiply per element
    for label, n, algo in (("mlp", 54_703_144, "sgd"), ("mlp", 54_703_144, "adam"), ("mlp", 54_703_144, "adamw"),
                           ("r18", 11_689_512, "sgd"), ("r50x4", 25_790_618, "adam")):
        n = (n + 7) // 8 * 8
        p = torch.randn(n, device=DEV)
        lp = torch.empty(n, device=DEV, dtype=torch.bfloat16)
        g = torch.randn(n, device=DEV).bfloat16()
        s0, s1 = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
        if algo == "sgd":
            def fn(i, p=p, g=g, s0=s0, lp=lp, n=n):
                _native.sgd_momentum(p, g, s0, lp, n, lr=0.01, mu=0.9, dampening=0.0, wd=1e-5,
                                     first_step=False)
            bpp = 20
        else:
            def fn(i, p=p, g=g, s0=s0, s1=s1, lp=lp, n=n, k=getattr(_native, algo)):
                k(p, g, s0, s1, None, lp, n, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, wd=1e-5, step=3)
            bpp = 28
        out.append(timed("K2 %s %s bf16-grad (%d elems)" % (algo, label, n), fn, 1, bpp * n, iters,
                         "one set: the arena itself is %d MB" % (bpp * n >> 20)))
    return out


def bench_k2mt(iters):
    """K2-mt / K1 on the parameter lists of BASELINE configs 4/5: 62 / 167 tensors, gradients in
    separately allocated bf16 tensors (what cuDNN hands to autograd), segment table in HBM."""
    import torchvision
    from frl_b200.multi_tensor import GradSegTable

    class Slot:
        def __init__(self, index, offset, numel):
            self.index, self.offset, self.numel = index, offset, numel

    out = []
    r50x4_heads = [(2048, 1000), (2048, 100), (2048, 10), (2048, 4)]
    for label, arch, heads, algo in (("r18", "resnet18", [(512, 1000)], "sgd"),
                                     ("r50x4", "resnet50", r50x4_heads, "adam"),
                                     ("r50x4", "resnet50", r50x4_heads, "adamw")):
        net = getattr(torchvision.models, arch)(weights=None)
        sizes = [p.numel() for n, p in net.named_parameters() if not n.startswith("fc.")]
        for i, o in heads:
            sizes += [i * o, o]
        slots, off = [], 0
        for i, n in enumerate(sizes):
            slots.append(Slot(i, off, n))
            off = (off + n + 7) // 8 * 8
        n = off
        grads = [torch.randn(s.numel, device=DEV).bfloat16() for s in slots]
        table = GradSegTable(slots, DEV)
        for s_, g in zip(slots, grads):
            table.point(s_, g.data_ptr(), g.dtype)
        table.upload()
        p = torch.randn(n, device=DEV)
        lp = torch.empty(n, device=DEV, dtype=torch.bfloat16)
        s0, s1 = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
        flat = torch.empty(n, device=DEV, dtype=torch.bfloat16)
        n_real = sum(sizes)
        if algo == "sgd":
            def fn(i, p=p, s0=s0, lp=lp, table=table):
                _native.sgd_momentum_mt(p, s0, lp, table, lr=0.01, mu=0.9, dampening=0.0, wd=1e-5, first_step=False)
            bpp = 20
        else:
            def fn(i, p=p, s0=s0, s1=s1, lp=lp, table=table, k=getattr(_native, algo + "_mt")):
                k(p, s0, s1, None, lp, table, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, wd=1e-5, step=3)
            bpp = 28
        out.append(timed("K2-mt %s %s: %d tensors, %d params, gradients read in place" % (algo, label, len(sizes), n_real),
                         fn, 1, bpp * n_real, iters))
        if algo == "adamw":
            continue                  # same table and gradients as the Adam row: K1 is timed there
        out.append(timed("K1 flatten_grads %s: %d tensors -> bf16 arena, one launch" % (label, len(sizes)),
                         lambda i, table=table, flat=flat: _native.flatten_grads(table, flat, scale=1.0), 1,
                         4 * n_real, iters))
    return out


def bench_k3(iters):
    n = 54_703_144
    out = []
    for dt in (torch.bfloat16, torch.float32):
        ns = sets_for(n * (2 if dt == torch.bfloat16 else 4))
        gs = [torch.randn(n, device=DEV).to(dt) for _ in range(ns)]
        out3 = torch.zeros(3, device=DEV)
        scratch = torch.zeros((_native.reduce_scratch_bytes() + 3) // 4, dtype=torch.int32, device=DEV)
        out.append(timed("K3 sumsq_clip %s (%d elems)" % (str(dt).replace("torch.", ""), n),
                         lambda i: _native.grad_sumsq_clip(gs[i], n, pre_scale=1.0, max_norm=1.0,
                                                           out3=out3, scratch=scratch),
                         ns, n * gs[0].element_size(), iters))
        del gs
    return out


def bench_k4(iters):
    B, C, R = 4096, 1000, 64
    out = []
    for dt in (torch.bfloat16, torch.float32):
        esz = 2 if dt == torch.bfloat16 else 4
        per = B * C * esz + B * R * esz + B * R * 4 + B * 8
        ns = sets_for(per)
        mods = [torch.nn.CrossEntropyLoss(), torch.nn.MSELoss()]
        sets = []
        for _ in range(ns):
            lo = torch.randn(B, C, device=DEV).to(dt).requires_grad_(True)
            ro = torch.randn(B, R, device=DEV).to(dt).requires_grad_(True)
            sets.append((lo, ro, torch.randint(0, C, (B,), device=DEV), torch.randn(B, R, device=DEV)))
        held = {}

        def fwd(i):
            lo, ro, y, r = sets[i]
            held[i] = criteria.fused_task_losses(mods, [lo, ro], [(y,), (r,)], [1.0, 1.0])

        name = str(dt).replace("torch.", "")
        out.append(timed("K4 criteria forward %s [4096,1000] CE + [4096,64] MSE" % name, fwd, ns, per, iters))
        for i in range(ns):
            fwd(i)

        def bwd(i):
            held[i][0].backward(retain_graph=True)
            sets[i][0].grad = sets[i][1].grad = None

        # backward reads logits + lse and writes dlogits (+ the small head)
        out.append(timed("K4 criteria backward %s (includes autograd dispatch)" % name, bwd, ns,
                         2 * (B * C * esz + B * R * esz) + B * R * 4 + B * 12, iters))
    return out


def bench_k5(iters):
    out = []
    n = 4096 * 4096
    ns = sets_for(n * 6)
    src = [torch.randn(n, device=DEV) for _ in range(ns)]
    dst = [torch.empty(n, device=DEV, dtype=torch.bfloat16) for _ in range(ns)]
    sc, bi = torch.tensor([2.0], device=DEV), torch.tensor([-1.0], device=DEV)
    out.append(timed("K5 preproc_affine f32->bf16 [4096,4096] (1 channel)",
                     lambda i: _native.preproc_affine(src[i], dst[i], inner=n, channels=1, scale=sc, bias=bi),
                     ns, n * 6, iters))
    out.append(timed("K5 cast_scale f32->bf16 [4096,4096]",
                     lambda i: _native.cast_scale(src[i], dst[i], 1.0), ns, n * 6, iters))
    del src, dst
    B, Cc, H = 256, 3, 224
    n = B * Cc * H * H
    ns = sets_for(n * 3)
    src = [torch.randint(0, 256, (n,), device=DEV, dtype=torch.uint8) for _ in range(ns)]
    dst = [torch.empty(n, device=DEV, dtype=torch.bfloat16) for _ in range(ns)]
    sc, bi = torch.rand(3, device=DEV), torch.rand(3, device=DEV)
    out.append(timed("K5 preproc_affine u8->bf16 [256,3,224,224] per-channel",
                     lambda i: _native.preproc_affine(src[i], dst[i], inner=H * H, channels=Cc, scale=sc, bias=bi),
                     ns, n * 3, iters))
    return out


def bench_k6(iters):
    out = []
    rows = cols = 4096
    ns = sets_for(rows * cols * 2 * 3)
    dy = [torch.randn(rows, cols, device=DEV).bfloat16() for _ in range(ns)]
    act = [torch.randn(rows, cols, device=DEV).bfloat16() for _ in range(ns)]
    dz = [torch.empty(rows, cols, device=DEV, dtype=torch.bfloat16) for _ in range(ns)]
    db = torch.empty(cols, device=DEV, dtype=torch.bfloat16)
    out.append(timed("K6 colsum bf16 [4096,4096]", lambda i: _native.colsum(dy[i], db), ns,
                     rows * cols * 2 + cols * 2, iters))
    out.append(timed("K6b drelu_colsum bf16 [4096,4096]",
                     lambda i: _native.drelu_colsum(dy[i], act[i], dz[i], db), ns,
                     rows * cols * 2 * 3 + cols * 2, iters))
    dy1 = [torch.randn(rows, 1000, device=DEV).bfloat16() for _ in range(ns)]
    db1 = torch.empty(1000, device=DEV, dtype=torch.bfloat16)
    out.append(timed("K6 colsum bf16 [4096,1000]", lambda i: _native.colsum(dy1[i], db1), ns,
                     rows * 1000 * 2 + 2000, iters))
    return out


def bench_k8(iters):
    out = []
    n_rows, width, B = 16384, 4096, 4096
    src = torch.randn(n_rows, width).pin_memory()
    dst = torch.empty(B, width, device=DEV)
    idx = torch.randperm(n_rows, device=DEV)[:B].contiguous()
    for blocks in (8, 16, 32):
        out.append(timed("K8 gather_rows (LSU) pinned host -> HBM, %d CTAs" % blocks,
                         lambda i: _native.gather_rows(src, idx, dst, max_blocks=blocks), 1,
                         B * width * 4, max(iters // 2, 2), "PCIe-bound (55 GB/s DMA ceiling), not HBM"))
    out.append(timed("K8 gather_rows_tma pinned host -> HBM, 2 CTAs",
                     lambda i: _native.gather_rows_tma(src, idx, dst, max_blocks=2), 1, B * width * 4,
                     max(iters // 2, 2), "PCIe-bound"))
    return out


BENCHES = {"k2": bench_k2, "k2mt": bench_k2mt, "k3": bench_k3, "k4": bench_k4, "k5": bench_k5, "k6": bench_k6,
           "k8": bench_k8}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="k2,k2mt,k3,k4,k5,k6,k8")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--json", default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--max-sets", type=int, default=0)
    args = ap.parse_args()
    global WARMUP, MAX_SETS
    WARMUP, MAX_SETS = args.warmup, args.max_sets
    torch.cuda.set_device(0)
    recs = []
    for key in args.only.split(","):
        recs += BENCHES[key](args.iters)
        torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"peak_hbm_gbs": peak_gbs(), "kernels": recs}, f, indent=1)


if __name__ == "__main__":
    main()
