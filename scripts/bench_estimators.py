#!/usr/bin/env python
"""Step time of the batched pipeline per estimator configuration, on bench.py's headline workload.

    python scripts/bench_estimators.py [--steps 20] [--warmup 5] [--rounds 2] [--batch 16]

Workload as bench.py --config 2: B synthetic 1024x768 images (tests/helpers.py, the same seeds), K=2000, border=5, CUDA-graph replay,
a 256 MiB write between timed steps to flush the L2.  The configurations are alternated and the whole round repeated (--rounds), so
that drift of the shared machine shows up as spread instead of as a difference.  Then one profiled step per configuration (per-launch
CUDA events, L.profile) gives the per-stage times, including the two hand-crafted pyramid kernels.  The card's name and power limit are
read in the same run (read-only nvidia-smi query).  Prints a plain-text report.
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

H, W, K, BORDER = 768, 1024, 2000, 5
# name -> (shape estimator, num_Baum_iters, orientation)
CONFIGS = [
    ("default: AffNet x1 + OriNet", "affnet", 1, "orinet"),
    ("AffNet x1 + hist", "affnet", 1, "hist"),
    ("AffNet x1 + none", "affnet", 1, "none"),
    ("Baumberg x16 + hist", "baumberg", 16, "hist"),
    ("Baumberg x16 + none", "baumberg", 16, "none"),
    ("0 + hist", None, 0, "hist"),
]
NEW_KERNELS = ("orientation_hist_pyr_kernel", "baumberg_pyr_kernel")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi: %s)" % r.stderr.strip()
    except Exception as e:   # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--batch", type=int, default=16)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_estimators.py needs a CUDA device (no CPU fallback)")
    import affnet_b200._lib as L
    from affnet_b200.architectures import AffNetFast, OriNetFast
    from affnet_b200.HandCraftedModules import AffineShapeEstimator, OrientationDetector
    from affnet_b200.HardNet import HardNet
    from affnet_b200.pipeline import DetectDescribePipeline
    from helpers import load_weights, synthetic_image
    dev = torch.device("cuda", 0)
    sd = load_weights()
    a, o, h = AffNetFast(PS=32), OriNetFast(PS=32), HardNet()
    a.load_state_dict(sd["affnet"]); o.load_state_dict(sd["orinet"]); h.load_state_dict(sd["hardnet"])
    a, o, h = a.eval().to(dev), o.eval().to(dev), h.eval().to(dev)
    B = args.batch
    imgs = torch.cat([synthetic_image(H, W, 1234 + i) for i in range(B)]).to(dev)    # bench.py's rank-0 inputs
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    pipes = []
    for name, shape, n, ori in CONFIGS:
        aff = {"affnet": a, "baumberg": AffineShapeEstimator(patch_size=19), None: None}[shape]
        orim = {"orinet": o, "hist": OrientationDetector(patch_size=19), "none": None}[ori]
        p = DetectDescribePipeline(B, H, W, aff, h, orim, num_features=K, border=BORDER, do_ori=ori != "none", device=dev, num_Baum_iters=n)
        p.capture()
        pipes.append(p)

    def timed(p):
        for _ in range(args.warmup):
            p.replay(imgs)
        torch.cuda.synchronize()
        evs = []
        for _ in range(args.steps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); p.replay(imgs); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        total = sum(x.elapsed_time(y) for x, y in evs)
        return total / args.steps

    print("# scripts/bench_estimators.py --steps %d --warmup %d --rounds %d --batch %d: %d x %dx%d synthetic, K=%d, border=%d, CUDA-graph "
          "replay, 256 MiB L2 flush between timed steps" % (args.steps, args.warmup, args.rounds, B, B, W, H, K, BORDER))
    print("# card: %s" % card())
    times = {name: [] for name, *_ in CONFIGS}
    for r in range(args.rounds):
        for (name, *_), p in zip(CONFIGS, pipes):
            ms = timed(p)
            times[name].append(ms)
            p.check()
            print("round %d  %-28s %7.3f ms/step  launches %d  keypoints/img %.0f" % (r + 1, name, ms, p.launches, p.count.float().mean().item()))
    print("# summary (ms per step over the rounds; min - max)")
    for name, *_ in CONFIGS:
        t = times[name]
        print("%-28s %7.3f - %7.3f" % (name, min(t), max(t)))

    print("# one profiled step per configuration (non-graph launch path, per-launch CUDA events), ms")
    for (name, *_), p in zip(CONFIGS, pipes):
        lst = []
        for i in range(3):
            flush.fill_(1.0)
            torch.cuda._sleep(4_000_000)      # the host enqueues the whole step behind this spin: no interval holds host launch latency
            lst = L.profile(lambda: p.run(imgs))
        agg = {}
        for k, ms in lst:
            agg.setdefault(k, [0, 0.0])
            agg[k][0] += 1
            agg[k][1] += ms
        top = sorted(agg.items(), key=lambda kv: -kv[1][1])
        print("%-28s sum %.3f  %s" % (name, sum(v[1] for v in agg.values()), ", ".join("%s x%d %.3f" % (k, v[0], v[1]) for k, v in top[:6])))
        for k in NEW_KERNELS:
            if k in agg:
                print("    %s: %.4f ms per launch (B*cap = %d rows)" % (k, agg[k][1] / agg[k][0],
                                                                       B * (int(1.5 * K) if k == "baumberg_pyr_kernel" else K)))


if __name__ == "__main__":
    main()
