#!/usr/bin/env python
"""Benchmark of the HesAffNet + HardNet detect-and-describe hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|5] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the whole path (pyramid -> Hessian/NMS -> top-k -> sample -> AffNet -> filter -> sample
-> OriNet -> sample -> HardNet) over one batch of B synthetic images per GPU.  Headline workload (--config 2, the default):
1024x768, K=2000 keypoints, B=16 (BASELINE.json configs[1] tiled B times = configs[3]'s per-GPU shard).  --config 3: 1920x1080, K=4000,
B=64; --config 5: 3840x2160, K=8000, border=33 (the 5-octave pyramid), B=1.  N>1: one process per GPU (torchrun), B images per rank
(weak scaling), one NCCL all-gather of descriptors/LAFs/counts per step.  Prints ONE JSON line; with the default config the line
also carries `extra`: the same metric for B=1, B=64 (configs[3] as written) and configs 3 and 5.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIGS = {   # BASELINE.json configs[...]: (H, W, K, border, default batch per GPU, label)
    "2": (768, 1024, 2000, 5, 16, "configs[1] tiled = configs[3] shard"),
    "3": (1080, 1920, 4000, 5, 64, "configs[2]"),
    "5": (2160, 3840, 8000, 33, 1, "configs[4] (border=33: the 5-octave pyramid)"),
}
ALG_BYTES_PER_PX = 30.66                      # SURVEY.md §8(d): detect stage, 4 B read + 5 levels x 4 B x 1.333 written
FLOP_PER_PATCH = {"affnet": 19.19e6, "orinet": 19.32e6, "hardnet": 78.18e6}   # 2*MAC, SURVEY.md §8(d)
DTYPE = "fp16 operands (fp16 residual planes: AffNet/OriNet weights+activations, HardNet layer 2-3 weights), fp32 accumulate; stencils fp32"


def oracle_module():
    """The CPU oracle: imported ONLY by the CPU legs (cpu_baseline / --impl reference), never by the product arm."""
    op = os.path.join(ROOT, "oracle")
    if op not in sys.path:
        sys.path.insert(0, op)
    import affnet_oracle
    return affnet_oracle


def ncu_traffic(batch):
    """DRAM bytes per step of the tcgen05 kernel family from the committed `ncu --set full` capture (profiles/*_ncu_traffic.json,
    written by scripts/ncu_summary.py); None when no capture exists for this batch size."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    for f in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if f.endswith("_ncu_traffic.json"):
            d = json.load(open(os.path.join(pdir, f)))
            if d.get("batch") == batch:
                best = {"dram_bytes_per_step": d["family_bytes_per_step"], "launches": len(d["launches"]), "source": "profiles/" + f}
    return best


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, src="fallback")


def make_images(B, seed0, H, W):
    from helpers import synthetic_image
    return torch.cat([synthetic_image(H, W, seed0 + i) for i in range(B)])


def load_state_dicts():
    from helpers import load_weights
    return load_weights()


DUMP_BUDGET = 64_000_000     # bytes that --dump-outputs may write


def dump_outputs(out_dir, lafs, resp, desc, count):
    """--dump-outputs: what the timed path returned in its last step for this rank's images, as DIR/<name>.npy (float32; count as
    float64), so that two builds can be compared output for output.  Rows at or past an image's count are unspecified, so they are
    written as zeros.  Above DUMP_BUDGET only a fixed, seeded sample of keypoint slots is written (the same slots for every image;
    their indices in keypoint_slots.npy)."""
    B, K = resp.shape
    valid = torch.arange(K)[None, :] < count.long()[:, None]
    out = {"lafs": lafs.masked_fill(~valid[:, :, None, None], 0.0), "resp": resp.masked_fill(~valid, 0.0),
           "desc": desc.masked_fill(~valid[:, :, None], 0.0)}
    per_slot = B * (6 + 1 + 128) * 4                           # bytes of lafs, resp and desc per keypoint slot
    slots = (DUMP_BUDGET - 8 * B - 4096) // (per_slot + 8)      # count.npy, keypoint_slots.npy and the .npy headers
    if slots < K:
        keep = np.sort(np.random.default_rng(0).choice(K, slots, replace=False))
        out = {k: a[:, torch.from_numpy(keep)] for k, a in out.items()}
        out["keypoint_slots"] = keep.astype(np.float64)
    out["count"] = count.double()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a.numpy() if isinstance(a, torch.Tensor) else a))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append((time.time(), l)) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def in_window(self, t0, t1):
        return sum(1 for t, _ in self.lines if t0 <= t <= t1)

    def stop(self, window=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for t, l in self.lines:
            if window is not None and not (window[0] <= t <= window[1]):
                continue
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, pw) if p > 250] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def best_cpu_threads(H, W):
    """Pick the torch thread count that runs the reference's dominant CPU cost (HardNet on a patch batch + one
    dense blur) fastest on this host: all cores is NOT the fastest on a 128-core box (measured 40x slower)."""
    O = oracle_module()
    sd = load_state_dicts()
    P = torch.rand(256, 1, 32, 32)
    x = torch.rand(1, 1, H, W)
    best, best_t = None, 1e30
    n = os.cpu_count() or 1
    for t in sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n}):
        torch.set_num_threads(t)
        O.hardnet_forward(P[:32], sd["hardnet"])
        t0 = time.perf_counter()
        O.hardnet_forward(P, sd["hardnet"]); O.gaussian_blur(x, 1.6)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = t, dt
    return best


class CpuArm:
    """The reference's own CPU implementation of the path: the UNMODIFIED reference through oracle/ref_harness.py when its tree is
    present ($AFFNET_REF, /root/reference, baseline/_ref; kind "reference"), else the oracle port (kind "port").  The reference is
    Python with neither setup.py nor pyproject.toml: it cannot be pip-installed into baseline/_ref and does not travel to the GPU box."""

    def __init__(self, H, W, K, border):
        O = oracle_module()
        self.O, self.H, self.W, self.K, self.border = O, H, W, K, border
        self.sd = load_state_dicts()
        self.kind, self.what = "port", "oracle/affnet_oracle.py (PyTorch-CPU restatement; the reference tree is absent on this host)"
        try:
            import ref_harness as R
            if R.available():
                aff, ori, hn = R.load_nets()
                self.det = R.make_detector(aff, ori, num_features=K, border=border)
                self.hn, self.R = hn, R
                self.kind, self.what = "reference", "the unmodified reference at %s through oracle/ref_harness.py::run_full (train_AffNet_test_on_graffity.py:255-260)" % R.REF
        except Exception as e:   # noqa: BLE001
            self.what += " [reference import failed: %s]" % e

    def one(self, img):
        if self.kind == "reference":
            LAFs, resp, patches, d = self.R.run_full(self.det, self.hn, img, True)
            return d.shape[0]
        dL, r, d = self.O.detect_and_describe(img, self.sd["affnet"], self.sd["orinet"], self.sd["hardnet"], self.K, border=self.border, do_ori=True)
        return d.shape[0]

    def leg(self, imgs, threads):
        torch.set_num_threads(threads)
        self.one(imgs[0:1])   # warm-up
        t0 = time.perf_counter()
        n_desc = sum(self.one(imgs[i:i + 1]) for i in range(imgs.size(0)))
        dt = time.perf_counter() - t0
        return dt, imgs.size(0) * self.H * self.W / dt / 1e6, n_desc / dt / 1e3


def run_reference(args, rank, world, real_stdout):
    if rank != 0:
        return
    H, W, K, border, _, label = CONFIGS[args.config]
    threads = best_cpu_threads(H, W)
    per = max(1, min(args.ref_images, 24 // max(1, args.steps)))     # bounded sample: at most ~24 images in the whole run
    arm = CpuArm(H, W, K, border)
    imgs = make_images(per, 1234, H, W)
    times, mpix, kp = [], [], []
    for _ in range(max(1, args.steps)):
        dt, m, k = arm.leg(imgs, threads)
        times.append(dt); mpix.append(m); kp.append(k)
    v = float(np.mean(mpix))
    line = {"impl": "reference", "metric": "Mpix/s end-to-end HesAffNet(+OriNet)+HardNet", "value": v, "unit": "Mpix/s",
            "kpatches_per_s": float(np.mean(kp)), "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": float(np.mean(times)) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic images (seeded noise, blur sigma 2, stretched), pretrained weights from tests/golden",
            "config": {"workload": "%dx%d grayscale, %d kpts/img, %d image(s) per step (bounded CPU sample of the batch; %s)" % (W, H, K, per, label),
                       "do_ori": True, "border": border, "mrSize": 5.192},
            "cpu_baseline": {"value": v, "unit": "Mpix/s", "cores": threads, "host_cores": os.cpu_count(), "kind": arm.kind,
                             "sample": "%d image(s) of the workload per step, %s" % (per, arm.what)},
            "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(real_stdout, line)


def main():
    # NCCL may print its version banner on stdout: keep fd 1 clean for the single JSON line
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _main(real_stdout)
    finally:
        os.dup2(real_stdout, 1)


def emit(real_stdout, line):
    os.write(real_stdout, (json.dumps(line) + "\n").encode())


TC_FAMILY = ("tc_first2_kernel", "tc_conv_kernel", "tc_conv_pair_kernel", "tc_head_kernel", "tc_headx_kernel", "tcx_first_kernel", "tcx_conv_kernel")
STENCIL = ("blur_kernel", "octave_kernel", "pyramid_tail_kernel", "detect_level_kernel", "detect_fused_kernel", "detect_warp_kernel", "detect_rows_kernel", "resolve_kernel")


class Workload:
    """One configuration on this rank's GPU: pipeline, inputs, device-resident and end-to-end timed legs."""

    def __init__(self, ctx, H, W, K, border, B, use_graph, exchange=True):
        from affnet_b200.pipeline import DetectDescribePipeline
        self.ctx, self.H, self.W, self.K, self.border, self.B, self.use_graph = ctx, H, W, K, border, B, use_graph
        dev, rank, world = ctx["dev"], ctx["rank"], ctx["world"]
        a, o, h = ctx["nets"]
        self.xchg = None
        if world > 1 and exchange:
            from affnet_b200.exchange import make_exchange
            self.xchg, ctx["exchange_kind"] = make_exchange(world, B, K, dev)   # one gather per step, overlapped with the next step; the kernels write its blocks directly
        self.pipe = DetectDescribePipeline(B, H, W, a, h, o, num_features=K, border=border, do_ori=True, device=dev,
                                           outputs=self.xchg.outputs() if self.xchg else None)
        self.host_imgs = make_images(B, 1234 + rank * B, H, W).pin_memory()
        self.dev_imgs = self.host_imgs.to(dev)
        self.last = [None, None, None, None]
        self.step_i = 0
        if use_graph:
            self.pipe.capture()

    def _run(self, imgs):
        """One step into the next output slot; with an exchange: wait for the gather that last read the slot, compute, queue its gather."""
        slot = (self.step_i & 1) if self.xchg else 0
        if self.xchg:
            self.xchg.wait_slot(slot)
        out = self.pipe.replay(imgs, slot) if self.use_graph else self.pipe.run(imgs, slot)
        if self.xchg:
            self.xchg.submit(slot)
        self.step_i += 1
        self.last[:] = out
        return out

    def step_device(self):
        return self._run(self.dev_imgs)

    def timed(self, steps, warmup, sampler=None, keep_last=False):
        """keep_last: copy the last timed step's outputs to host memory as self.last_host (after the timed region, before the clock
        sampler's extra steps overwrite the pipeline's buffers)."""
        ctx = self.ctx
        dist, dev, flush = ctx["dist"], ctx["dev"], ctx["flush"]
        for _ in range(warmup):
            self.step_device()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t_begin = time.time()
        evs = []
        for _ in range(steps):
            flush.fill_(1.0)                                  # L2 flush between timed iterations (outside the events)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); self.step_device(); e1.record()
            evs.append((e0, e1))
        if self.xchg:   # the last steps' all-gathers finish inside the timed region
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); self.xchg.drain(); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        t_stop = time.time()
        if keep_last:
            self.last_host = [t.cpu() for t in self.last]
        clocks = None
        if sampler:
            # The sampler runs since before the warm-up; only samples that arrived inside the timed region count.  If the region was
            # too short for three of them, the same load keeps running (untimed, rank 0 only, hence without collectives) until it is.
            extra, t_end = 0, time.time() + 4.0
            while sampler.in_window(t_begin, time.time()) < 3 and time.time() < t_end:
                (self.pipe.replay(self.dev_imgs) if self.use_graph else self.pipe.run(self.dev_imgs)); torch.cuda.synchronize(); extra += 1
            clocks = sampler.stop(window=(t_begin, time.time() if extra else t_stop))
            clocks["sampled"] = "inside the timed region" if extra == 0 else "timed region + %d extra untimed steps of the same load" % extra
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        total_ms = sum(a_.elapsed_time(b_) for a_, b_ in evs)
        t = torch.tensor([total_ms], device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), clocks

    def check_exchange(self):
        if not self.xchg:
            return
        rank, B = self.ctx["rank"], self.B
        self.xchg.drain(); torch.cuda.synchronize()
        gd, gl, gc = self.xchg.last()
        own = slice(rank * B, (rank + 1) * B)
        if not (torch.equal(gc[own], self.last[3].int()) and bool((gc > 0).all()) and torch.equal(gd[own], self.last[2]) and torch.equal(gl[own], self.last[0])):
            raise RuntimeError("all-gather returned something else than this rank's results")

    def timed_e2e(self, steps, warmup):
        """Every step uploads ITS OWN batch from pinned host memory and downloads ITS OWN results.  Transfers run on copy streams and are
        software-pipelined against the compute of the neighbouring steps (double-buffered device staging), as a serving loop would do;
        all of it is inside the timed region: ONE event pair around all steps, closed after the last results reached host memory."""
        ctx = self.ctx
        dist, dev = ctx["dist"], ctx["dev"]
        B, K, pipe, use_graph, xchg = self.B, self.K, self.pipe, self.use_graph, self.xchg
        host_desc = torch.empty(B, K, 128).pin_memory(); host_lafs = torch.empty(B, K, 2, 3).pin_memory()
        host_resp = torch.empty(B, K).pin_memory(); host_cnt = torch.empty(B, dtype=torch.int32).pin_memory()
        copy_stream = torch.cuda.Stream(device=dev)     # device -> host
        up_stream = torch.cuda.Stream(device=dev)       # host -> device (separate, so uploads never queue behind a download)
        stage_in = [torch.empty_like(self.dev_imgs) for _ in range(2)]
        stage_out = [(torch.empty(B, K, 128, device=dev), torch.empty(B, K, 2, 3, device=dev), torch.empty(B, K, device=dev),
                      torch.empty(B, dtype=torch.int32, device=dev)) for _ in range(2)]
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        state = {"i": 0}

        def upload(slot):
            with torch.cuda.stream(up_stream):
                stage_in[slot].copy_(self.host_imgs, non_blocking=True)
                ev_in[slot].record(up_stream)

        def step():
            i = state["i"]; slot = i & 1
            cur = torch.cuda.current_stream()
            if i == 0:
                upload(slot)
            cur.wait_event(ev_in[slot])                       # this step's images are on the device
            ev_free = torch.cuda.Event(); ev_free.record(cur)
            up_stream.wait_event(ev_free)                     # the other input slot was consumed by the previous step
            upload(slot ^ 1)                                  # next step's images travel while this step computes
            out = self._run(stage_in[slot])
            if i >= 2:
                cur.wait_event(ev_done[slot])                 # the download that used this staging slot two steps ago has finished
            so = stage_out[slot]
            so[0].copy_(out[2], non_blocking=True); so[1].copy_(out[0], non_blocking=True); so[2].copy_(out[1], non_blocking=True); so[3].copy_(out[3], non_blocking=True)
            ev_out[slot].record(cur)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_out[slot])
                host_desc.copy_(so[0], non_blocking=True); host_lafs.copy_(so[1], non_blocking=True)
                host_resp.copy_(so[2], non_blocking=True); host_cnt.copy_(so[3], non_blocking=True)
                ev_done[slot].record(copy_stream)
            state["i"] = i + 1

        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        if xchg:
            xchg.drain()
        torch.cuda.current_stream().wait_stream(copy_stream)
        torch.cuda.current_stream().wait_stream(up_stream)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def summary(self, steps, warmup, e2e=True):
        """Device-resident + end-to-end throughput of this configuration (for the `extra` block)."""
        total_ms, _ = self.timed(steps, warmup)
        self.pipe.check()
        self.check_exchange()
        world = self.ctx["world"]
        pix = world * self.B * self.H * self.W
        n_desc = int(self.last[3].sum().item())
        ms = total_ms / steps
        out = {"workload": "%dx%d, %d kpts/img, border %d, %d image(s) per GPU per step" % (self.W, self.H, self.K, self.border, self.B),
               "value": pix / (ms * 1e-3) / 1e6, "unit": "Mpix/s", "ms_per_step": ms, "kpatches_per_s": world * n_desc / (ms * 1e-3) / 1e3, "steps": steps}
        if e2e:
            e_ms = self.timed_e2e(steps, warmup) / steps
            out["e2e"] = {"value": pix / (e_ms * 1e-3) / 1e6, "unit": "Mpix/s", "ms_per_step": e_ms,
                          "h2d_bytes_per_step": self.B * self.H * self.W * 4, "d2h_bytes_per_step": self.B * self.K * (128 + 6 + 1) * 4 + self.B * 4}
        return out

    def close(self):
        self.pipe = None
        self.xchg = None
        torch.cuda.empty_cache()


def _main(real_stdout):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="2", choices=sorted(CONFIGS), help="BASELINE.json configuration (2 = headline)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the configuration's)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-images", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra configurations (B=1, B=64, configs 3 and 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0's images) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world, real_stdout)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    args.warmup = max(args.warmup, 3)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)

    import affnet_b200._lib as L
    from affnet_b200.architectures import AffNetFast, OriNetFast
    from affnet_b200.HardNet import HardNet
    sd = load_state_dicts()
    a, o, h = AffNetFast(PS=32), OriNetFast(PS=32), HardNet()
    a.load_state_dict(sd["affnet"]); o.load_state_dict(sd["orinet"]); h.load_state_dict(sd["hardnet"])
    a, o, h = a.eval().to(dev), o.eval().to(dev), h.eval().to(dev)
    H, W, K, border, B0, label = CONFIGS[args.config]
    B = args.batch or B0
    if args.config == "5":      # BASELINE.json configs[4]: "bf16 HardNet tensor-core path"
        h.set_engine(L.ENGINE_TC2_BF16)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()   # nvidia-smi needs a few hundred ms to deliver its first sample: start it long before the timed region
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
    ctx = {"dev": dev, "dist": dist, "rank": rank, "world": world, "nets": (a, o, h), "flush": flush}
    use_graph = not args.no_graph
    wl = Workload(ctx, H, W, K, border, B, use_graph)
    pipe = wl.pipe

    total_ms, clocks = wl.timed(args.steps, args.warmup, sampler, keep_last=bool(args.dump_outputs))
    pipe.check()
    last_outputs = wl.last_host if args.dump_outputs else None
    wl.check_exchange()
    n_desc = int(wl.last[3].sum().item())
    e2e_ms = wl.timed_e2e(args.steps, args.warmup)

    # ---- per-kernel CUDA-event profile of the same step (non-graph launch path), rank 0 ---------------------------
    roof = None
    if rank == 0:
        per_kernel, order = {}, []
        prof_steps = 3
        for i in range(prof_steps):
            flush.fill_(1.0)
            torch.cuda._sleep(4_000_000)     # ~2 ms of GPU spin: the host enqueues the whole step behind it, so no interval holds host launch latency
            lst = L.profile(lambda: pipe.run(wl.dev_imgs))
            if i == prof_steps - 1:
                order = [(k, round(ms, 4)) for k, ms in lst]
            for name, ms in lst:
                per_kernel.setdefault(name, []).append(ms)
        step_ms = sum(sum(v) for v in per_kernel.values()) / prof_steps
        agg = sorted(((sum(v) / prof_steps, len(v) // prof_steps, k) for k, v in per_kernel.items()), reverse=True)
        pk = peaks()
        # dominant kernel family: every tcgen05 kernel of the three CNNs (layers 1+2 fused with the sampler in the "first" kernels, layers 3-6 in
        # the conv kernels, the 8x8 head GEMMs in tc_head_kernel / tc_headx_kernel)
        n_aff, n_ori, n_hard = B * int(1.5 * K), n_desc, n_desc
        tc_flop = n_aff * FLOP_PER_PATCH["affnet"] + n_ori * FLOP_PER_PATCH["orinet"] + n_hard * FLOP_PER_PATCH["hardnet"]
        tc_ms = sum(t for t, n, k in agg if k in TC_FAMILY)
        tc_launches = sum(n for t, n, k in agg if k in TC_FAMILY)
        ach = tc_flop / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
        roof = {"kernel": "tcgen05 kernels (%d launches/step: %s; fp16 operands with fp16 residual planes for AffNet/OriNet and HardNet layers 2-3, fp32 accumulate in TMEM)"
                          % (tc_launches, ", ".join("%s x%d" % (k, n) for t, n, k in agg if k in TC_FAMILY)),
                "bound": "tensor", "achieved": ach, "peak": pk["tensor_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tensor_sustained"],
                "traffic": ncu_traffic(B), "peak_source": pk["src"] + " bf16 sustained (kernel timed inside a long step)", "kernel_ms_per_step": tc_ms,
                "algorithmic_flop_per_step": tc_flop, "share_of_step": tc_ms / step_ms if step_ms else None,
                "note": "algorithmic flops = 2*MAC of the reference's fp32 convolutions; the residual-plane products (3 MMAs per K step for AffNet/OriNet, 2 for HardNet "
                        "layers 2-3) and the K=9 first layer padded to K=16 are extra tensor work that is not counted",
                "timing": "CUDA events after every launch over %d profiled steps right after the timed region" % prof_steps,
                "stages_ms": {k: round(t, 4) for t, n, k in agg}, "launches_ms": order}
        # HBM roofline of the stencil side (pyramid + detect kernels), reported alongside
        st_ms = sum(t for t, n, k in agg if k in STENCIL)
        roof["stencil"] = {"kernels": ", ".join("%s x%d" % (k, n) for t, n, k in agg if k in STENCIL), "bound": "hbm",
                           "achieved": ALG_BYTES_PER_PX * B * H * W / (st_ms * 1e-3) / 1e9 if st_ms else None,
                           "peak": pk["hbm"], "unit": "GB/s", "ms_per_step": st_ms}
        if roof["stencil"]["achieved"]:
            roof["stencil"]["frac"] = roof["stencil"]["achieved"] / pk["hbm"]

    launches_per_step = pipe.launches
    exchange_cost = None
    if world > 1:    # the same steps without the all-gather: what the exchange costs (VERDICT r01 item 6)
        wl.close(); wl = None; pipe = None
        w0 = Workload(ctx, H, W, K, border, B, use_graph, exchange=False)
        t0, _ = w0.timed(args.steps, args.warmup)            # same step and warm-up counts: the clocks sag over a long run, so the legs must be alike
        w0.close(); w0 = None
        exchange_cost = {"ms_per_step_without_exchange": t0 / args.steps, "ms_per_step_with_exchange": total_ms / args.steps,
                         "kind": ctx.get("exchange_kind")}
    extra = None
    if not args.no_extras and args.config == "2" and not args.batch:
        if wl is not None:
            wl.close(); wl = None; pipe = None
        extra = {}
        plan = [("b1", "2", 1, 10), ("b64_config4_shard", "2", 64, 3)] if world > 1 else [("b1", "2", 1, 10), ("b64_config4_shard", "2", 64, 3), ("config3", "3", 64, 2), ("config5", "5", 1, 5)]
        for name, cfg, b, st in plan:
            try:
                Hh, Ww, Kk, bb, _, lab = CONFIGS[cfg]
                h.set_engine(L.ENGINE_TC2_BF16 if cfg == "5" else L.ENGINE_TC2)     # configs[4] names the bf16 HardNet path
                w2 = Workload(ctx, Hh, Ww, Kk, bb, b, use_graph)
                extra[name] = w2.summary(st, 3, e2e=True)
                extra[name]["config"] = lab
                extra[name]["hardnet_operands"] = "bf16" if cfg == "5" else "fp16"
                w2.close()
            except Exception as e:   # noqa: BLE001  (an extra must never cost the headline line)
                extra[name] = {"error": str(e)[:300]}
            w2 = None
            torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        threads = best_cpu_threads(H, W)
        arm = CpuArm(H, W, K, border)
        dt, m, kps = arm.leg(make_images(args.ref_images, 1234, H, W), threads)
        cpu = {"value": m, "unit": "Mpix/s", "cores": threads, "host_cores": os.cpu_count(), "kind": arm.kind, "kpatches_per_s": kps,
               "sample": "%d of the %d images of one step, %s, fastest torch thread count of a sweep (%.1f s)" % (args.ref_images, B, arm.what, dt)}

    if rank == 0:
        ms_per_step = total_ms / args.steps
        pix = world * B * H * W
        value = pix / (ms_per_step * 1e-3) / 1e6
        e2e_v = pix / (e2e_ms / args.steps * 1e-3) / 1e6
        line = {"metric": "Mpix/s end-to-end HesAffNet(+OriNet)+HardNet", "value": value, "unit": "Mpix/s",
                "kpatches_per_s": world * n_desc / (ms_per_step * 1e-3) / 1e3, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPE.replace("fp16 operands", "fp16 operands (HardNet: bf16 operands, configs[4])") if args.config == "5" else DTYPE,
                "data": "synthetic images (seeded noise, blur sigma 2, stretched), pretrained weights from tests/golden",
                "config": {"workload": "%dx%d grayscale, %d kpts/img, batch of %d images per GPU per step (%s)" % (W, H, K, B, label),
                           "do_ori": True, "border": border, "mrSize": 5.192, "cuda_graph": use_graph, "l2": "256 MiB flush write between timed steps (device-resident leg); e2e leg: fresh inputs arrive by DMA every step, no flush",
                           "parallelism": ("images sharded across GPUs, one all-gather of descriptors+LAFs+counts per step (%s), written by the kernels straight into the send block, overlapped with the next step's compute"
                                           % {"ce": "peer-to-peer copy-engine pushes into symmetric memory + barrier", "nccl": "NCCL all_gather_into_tensor"}.get(ctx.get("exchange_kind"), "?")) if world > 1 else "single GPU"},
                "roofline": roof, "cpu_baseline": cpu, "clocks": clocks,
                "e2e": {"value": e2e_v, "unit": "Mpix/s", "h2d_bytes_per_step": B * H * W * 4,
                        "d2h_bytes_per_step": B * K * (128 + 6 + 1) * 4 + B * 4, "ms_per_step": e2e_ms / args.steps},
                "gpu_launches": launches_per_step * args.steps, "launches_per_step": launches_per_step,
                "descriptors_per_step": world * n_desc}
        if extra is not None:
            line["extra"] = extra
        if exchange_cost is not None:
            line["exchange"] = exchange_cost
        if last_outputs is not None:
            dump_outputs(args.dump_outputs, *last_outputs)
        emit(real_stdout, line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
