#!/usr/bin/env python
"""Benchmark of the embed+detect hot path (BASELINE.json metric: embed+detect frames/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--card C] [--batch B] [--size S]
                    [--dump-outputs DIR]

One "step" = model.embed(batch, msgs, is_video=False) followed by model.detect(imgs_w, is_video=False) on one batch of
synthetic frames (configs[1] of BASELINE.json by default: videoseal_1.0, 256-bit, 64 x 3x256x256 per GPU).  Under torchrun
every rank processes its own batch (frames are independent units: weak scaling, no data-path collective except the
all-gather of the [B, 1+K] logits that reassembles the detection output).  Prints ONE JSON line on rank 0.

--impl reference times the CPU restatement of the reference path (oracle/restate.py, pinned bit-exact to the reference
modules) on the host cores; the unmodified reference itself needs packages that are not installed here (DESIGN.md).
"""
import argparse
import atexit
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_FRAME = {  # SURVEY.md §8(d): 2*MAC over every Conv2d/Linear at processing size 256 (embed, detect)
    "videoseal_1.0": (56.55e9, 12.32e9), "pixelseal": (119.30e9, 12.32e9), "chunkyseal": (2248.96e9, 1227.24e9),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--card", default="videoseal_1.0")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--video", action="store_true", help="is_video=True: one message, key frames every step_size frames")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-clip-leg", action="store_true", help="skip the BASELINE configs[2] leg (512-frame 768x768 clip, strong scaling)")
    ap.add_argument("--clip-frames", type=int, default=512)
    ap.add_argument("--no-hbm-leg", action="store_true", help="skip the 768x768 leg that measures the HBM-bound kernels")
    ap.add_argument("--profile-out", default="", help="write the per-kernel table (JSON) here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what embed() and detect() returned in the last timed step as DIR/<name>.npy "
                         "(float32; a seeded sample of the frames when they exceed 64 MB), to compare builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)     # the sampler never outlives bench.py, also when it fails before stop()
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def conv_flops(name: str, B: int, B_unet: int = 0) -> float:
    """algorithmic FLOPs (2*MAC) of one launch of a named plan step, from its shape tag (model.cuh step names).
    B_unet: frames that go through the U-Net (key frames only in video mode); the extractor sees all B frames."""
    try:
        kind, rest = name.rsplit(".", 1)
        dims, hs = rest.split("@")
        h = int(hs)
        M = (B_unet if (B_unet and kind.startswith("unet.")) else B) * h * h
        if kind in ("unet.conv3x3", "unet.conv3x3+outc", "unet.conv3x3d", "unet.conv3x3d+outc", "unet.down3x3s2", "unet.down3x3s2d", "unet.up3x3"):
            cin, cout = (int(x) for x in dims.split("-"))
            return 2.0 * M * cout * 9 * cin
        if kind == "unet.uptap1x1":
            cin, cout = (int(x) for x in dims.split("-"))
            return 2.0 * M * cout * cin
        if kind in ("unet.conv1x1", "unet.conv1x1d"):
            cin, cout = (int(x) for x in dims.split("-"))
            return 2.0 * M * cout * cin
        if kind == "cnx.down2x2s2":
            cin, cout = (int(x) for x in dims.split("-"))
            return 2.0 * M * cout * 4 * cin
        if kind in ("cnx.pwconv1", "cnx.pwconv2"):
            c = int(dims)
            return 2.0 * M * c * 4 * c
        if kind == "cnx.stem_gemm":
            return 2.0 * M * int(dims) * 48
        if kind == "cnx.head3x3":
            c = int(dims)
            return 2.0 * M * c * 9 * c
    except Exception:
        pass
    return 0.0


def pointwise_bytes(name: str, S: int = 256) -> float:
    """algorithmic HBM bytes of one launch of a full-resolution (pw.*) step, from its shape tag `kind.HxW@frames[+preds]`
    (SURVEY.md section 8(d): fp32 API tensors, the delta at processing size is L2 traffic and is not counted)."""
    try:
        kind, rest = name[3:].split(".", 1) if name.count(".") >= 2 else (name[3:].split("@")[0], "0x0@" + name.split("@")[1])
        dims, n = rest.split("@")
        preds = n.endswith("+preds")
        n = int(n.replace("+preds", ""))
        h, w = (int(x) for x in dims.split("x"))
        if kind == "resize":
            return n * 3 * 4.0 * (h * w + S * S)                      # read the frames, write them at processing size
        if kind in ("jnd_blend", "blend"):
            return n * 4.0 * h * w * (3 + 3 + (1 if preds else 0))    # read imgs, write imgs_w (+ preds_w, 1 channel for Y cards)
        if kind == "jnd_lowres":
            return n * 4.0 * S * S * (3 + 1)
    except Exception:
        pass
    return 0.0


def ncu_traffic(tag: str):
    """per-launch dram__bytes_read+write of a kernel from the committed ncu summaries (profiles/ncu_traffic.json), or None"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(tag)
    return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


DUMP_BYTES = 64 * 10**6


def dump_outputs(outs: dict, out_dir: str, seed: int = 0):
    """Write the per-frame outputs `outs` (name -> tensor with frames along dim 0) as out_dir/<name>.npy in float32.  When they
    exceed DUMP_BYTES, the same seeded sample of frames (in frame order) is taken from every array."""
    import numpy as np
    import torch
    n = next(iter(outs.values())).shape[0]
    per_frame = sum(4 * t[0].numel() for t in outs.values())
    keep = min(n, DUMP_BYTES // per_frame)
    if keep == 0:
        raise SystemExit(f"--dump-outputs: one frame of outputs is {per_frame} bytes, more than the {DUMP_BYTES}-byte budget")
    idx = None
    if keep < n:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:keep].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outs.items():
        t = t.detach().float().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (t if idx is None else t[idx]).numpy())
    return {"dir": out_dir, "arrays": sorted(outs), "frames": n if idx is None else idx.tolist()}


def build_card_on_disk(card_name: str, seed: int = 0):
    """synthetic checkpoint (no network) + a card YAML pointing at it, under a temp dir"""
    import tempfile
    import yaml
    from videoseal_b200 import synth
    d = tempfile.mkdtemp(prefix="vsb200_bench_")
    card = yaml.safe_load(open(os.path.join(ROOT, "videoseal_b200", "cards", card_name + ".yaml")))
    ckpt = os.path.join(d, card_name + ".pth")
    synth.write_synthetic_checkpoint(card, ckpt, seed)
    card["checkpoint_path"] = ckpt
    cpath = os.path.join(d, card_name + ".yaml")
    yaml.safe_dump(card, open(cpath, "w"))
    return cpath, card


def cpu_oracle_setup(card_name: str, size: int):
    import torch
    import yaml
    from oracle import restate
    card = yaml.safe_load(open(os.path.join(ROOT, "videoseal_b200", "cards", card_name + ".yaml")))
    spec = restate.spec_from_card(card)
    orc = restate.OracleModel(spec, restate.synth_state_dict(spec, 0))
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(8, 3, size, size, generator=g)
    msgs = torch.randint(0, 2, (8, spec["nbits"]), generator=g)

    def run(n):
        with torch.no_grad():
            t0 = time.perf_counter()
            o = orc.embed(imgs[:n], msgs[:n], is_video=False)
            orc.detect(o["imgs_w"], is_video=False)
            return time.perf_counter() - t0
    return run


def cpu_pick_threads(run):
    """the host may expose more logical CPUs than this process can use: calibrate the torch thread count on one frame"""
    import torch
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    best, best_t = 1, float("inf")
    for th in sorted({avail, min(avail, 64), min(avail, 32), min(avail, 16), min(avail, 8)}):
        torch.set_num_threads(th)
        run(1)
        t = run(1)
        if t < best_t:
            best, best_t = th, t
    torch.set_num_threads(best)
    return best, best_t


def cpu_oracle_fps(card_name: str, size: int, runs: int, budget_s: float):
    """embed+detect frames/s of the CPU restatement of the reference path (test infrastructure, timed as the baseline).
    1 warm-up + `runs` timed runs (evals/speed.py:51-52) on a sample sized to fit `budget_s` seconds."""
    run = cpu_oracle_setup(card_name, size)
    threads, t1 = cpu_pick_threads(run)
    sample = int(max(1, min(8, budget_s / max(1e-3, t1 * (runs + 1)))))
    run(sample)
    times = [run(sample) for _ in range(runs)]
    return sample * len(times) / sum(times), times, threads, sample


def clip_leg(model, dev, world: int, rank: int, frames: int, size: int, steps: int, seed: int = 7):
    """BASELINE configs[2]: a `frames`-frame 3 x size x size clip, is_video=True, sharded over the ranks in contiguous frame ranges
    aligned to step_size (videoseal_b200.dist.shard_bounds); every rank embeds and detects its shard and ONE NCCL all-gather
    reassembles the watermarked frames on every rank (plus one for the [F, 1+K] logits).  STRONG scaling: the clip is fixed.
    Three variants are timed with CUDA events (max over ranks): no frame gather (outputs stay sharded), gather after the step
    (serial), and gather issued right after embed() so that it runs on NCCL's stream while detect() computes (overlapped; this is
    `value`).  The all-gather alone is timed too: it is the collective that limits the real config."""
    import torch
    import torch.distributed as dist
    from videoseal_b200 import dist as vdist
    K = model.spec["nbits"]
    step_size = int(model.step_size)
    bounds = vdist.shard_bounds(frames, world, step_size)
    s, e = bounds[rank]
    n_loc = e - s
    equal = all(b[1] - b[0] == n_loc for b in bounds)
    g = torch.Generator().manual_seed(seed + rank)
    local = [torch.rand(n_loc, 3, size, size, generator=g).to(dev) for _ in range(2)]   # per-rank shard only: the clip never lives on one GPU
    msgs = torch.randint(0, 2, (1, K), generator=torch.Generator().manual_seed(seed)).to(dev)
    gath_imgs = torch.empty(frames, 3, size, size, device=dev) if world > 1 else None
    gath_log = torch.empty(frames, 1 + K, device=dev) if world > 1 else None
    sizes = [b[1] - b[0] for b in bounds]

    def gather(dst, src, async_op=False):
        if equal:
            return dist.all_gather_into_tensor(dst, src.contiguous(), async_op=async_op)
        dst.copy_(vdist.all_gather_ragged(src.contiguous(), sizes))
        return None

    def step(i, mode):
        out = model.embed(local[i % 2], msgs, is_video=True)["imgs_w"]
        work = None
        if world > 1 and mode == "overlap":
            work = gather(gath_imgs, out, async_op=True)        # NCCL stream, ordered after embed(); detect() runs beside it
        preds = model.detect(out, is_video=True)["preds"]
        if world > 1:
            gather(gath_log, preds)
            if mode == "serial":
                gather(gath_imgs, out)
            if work is not None:
                work.wait()
        return out, preds

    def timed(fn, n):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms / n

    # sub-sharded variant: every rank owns TWO ranges (videoseal_b200.dist.subshard_bounds); the all-gather of the first half of the
    # clip runs on NCCL's stream while the ranks embed their second range, the second one while they detect
    sub = None
    if world > 1 and frames % (world * 2 * step_size) == 0:
        sb = vdist.subshard_bounds(frames, world, step_size, 2)[rank]
        n_sub = sb[0][1] - sb[0][0]
        seg = frames // 2

        def step_sub(i):
            x = local[i % 2]
            outs, works = [], []
            for sidx in range(2):
                o = model.embed(x[sidx * n_sub:(sidx + 1) * n_sub], msgs, is_video=True)["imgs_w"]
                works.append(dist.all_gather_into_tensor(gath_imgs[sidx * seg:(sidx + 1) * seg], o, async_op=True))
                outs.append(o)
            preds = model.detect(torch.cat(outs, dim=0), is_video=True)["preds"]
            gather(gath_log, preds)
            for w in works:
                w.wait()
            return preds
        sub = step_sub

    res = {"frames": frames, "size": size, "frames_per_rank": n_loc, "step_size": step_size, "chunk_size": int(model.chunk_size),
           "scaling": "strong", "unit": "frames/s"}
    modes = ["none"] if world == 1 else ["none", "serial", "overlap"]
    for mode in modes:
        for i in range(3):
            step(i, mode)
        ms = timed(lambda i: step(i, mode), steps)
        res[{"none": "sharded_outputs", "serial": "gather_serial", "overlap": "gather_overlapped"}[mode]] = {
            "ms_per_step": ms, "value": frames / (ms / 1000.0)}
    if world > 1:
        out, _ = step(0, "none")
        for i in range(2):
            gather(gath_imgs, out)
        ms = timed(lambda i: gather(gath_imgs, out), 5)
        by = (world - 1) * n_loc * 3 * size * size * 4
        res["all_gather_imgs_w"] = {"collective": "ncclAllGather (torch.distributed all_gather_into_tensor)" if equal else "all_gather (ragged, padded)",
                                    "ms": ms, "bytes_received_per_rank": by, "bus_gbs": by / (ms * 1e-3) / 1e9,
                                    "limit": "inbound NVLink of every GPU: (N-1)/N of the clip's output per rank"}
        best = "gather_overlapped"
        if sub is not None:
            for i in range(3):
                sub(i)
            ms = timed(sub, steps)
            res["gather_overlapped_2_subshards"] = {"ms_per_step": ms, "value": frames / (ms / 1000.0),
                                                    "note": "rank r owns frame ranges r and world+r of 2*world; gather of half 0 under embed of half 1, of half 1 under detect"}
            if ms < res["gather_overlapped"]["ms_per_step"]:
                best = "gather_overlapped_2_subshards"
        res["value"] = res[best]["value"]
        res["ms_per_step"] = res[best]["ms_per_step"]
        res["value_mode"] = best
    else:
        res["value"] = res["sharded_outputs"]["value"]
        res["ms_per_step"] = res["sharded_outputs"]["ms_per_step"]
    del local, gath_imgs
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    fps, times, threads, sample = cpu_oracle_fps(args.card, args.size, args.steps, budget_s=150.0)
    line = {
        "impl": "reference", "metric": "embed+detect frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sum(times) / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.card} embed+detect, image mode, 3x{args.size}x{args.size}, CPU sample of {sample} frames/step",
                   "card": args.card, "batch_per_step": sample, "size": args.size},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} frames per step; oracle/restate.py (bit-exact restatement of the reference modules)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import ctypes as C
    import videoseal_b200
    from videoseal_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout must carry exactly ONE JSON line: libraries (e.g. the NCCL version banner) write to fd 1 directly, so
    # everything except the final print goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        # NCCL_DEBUG is left alone: fd 1 already points at stderr, so NCCL's INFO lines (rank / channel proof) land there and
        # stdout still carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    cpath, card = build_card_on_disk(args.card, seed=0)
    from pathlib import Path
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        model = videoseal_b200.load(Path(cpath)).eval().to(dev)
    B, S, K = args.batch, args.size, model.spec["nbits"]
    NB = 4  # rotating input batches: NB * B*3*S*S*4 bytes (201 MB at the default shape) > 126 MB L2
    g = torch.Generator().manual_seed(1000 + rank)
    imgs = [torch.rand(B, 3, S, S, generator=g).to(dev) for _ in range(NB)]
    msgs = torch.randint(0, 2, (B, K), generator=g).to(dev)
    gathered = [torch.empty(B, 1 + K, device=dev) for _ in range(world)] if world > 1 else None

    vid = bool(args.video)
    msgs_v = msgs[:1]
    n_keys = (B + model.step_size - 1) // model.step_size if vid else B   # frames that go through the U-Net per step

    def step_local(i):
        out = model.embed(imgs[i % NB], msgs_v if vid else msgs, is_video=vid)
        return {**out, **model.detect(out["imgs_w"], is_video=vid)}

    def step(i):
        outs = step_local(i)
        if world > 1:
            dist.all_gather(gathered, outs["preds"])   # reassemble the detection output on every rank ([B,1+K] per rank)
        return outs

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # sampled while the GPU is under this workload (warm-up + timed steps)
        time.sleep(0.3)          # let nvidia-smi come up so that samples fall inside the loaded region
    for i in range(max(3, args.warmup)):
        step(i)
    sync_all()
    L.vsb_launch_count(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    ev0.record()
    for i in range(args.steps - 1):
        step(i)
    last = step(args.steps - 1)
    ev1.record()
    sync_all()
    ms = ev0.elapsed_time(ev1)
    launches = int(L.vsb_launch_count(0))
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    fps = world * B * args.steps / (ms / 1000.0)
    dumped = dump_outputs(last, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    del last

    # ---- end-to-end through the C ABI with HOST buffers (pinned): H2D + embed + D2H, H2D + detect + D2H, every step
    e2e = None
    if not args.no_e2e:
        CD = model.spec["unet"]["out_channels"]
        h_in = [torch.rand(B, 3, S, S, generator=g).pin_memory() for _ in range(2)]
        h_msgs = torch.randint(0, 2, (B, K), generator=g).to(torch.uint8).pin_memory()
        h_out = torch.empty(B, 3, S, S).pin_memory()
        h_log = torch.empty(B, 1 + K).pin_memory()
        flags = _lib.FLAG_CLAMP
        h = model._handle()

        def e2e_step(i):
            _lib.check(L.vsb_embed_detect_host(h, h_in[i % 2].data_ptr(), h_msgs.data_ptr(), B, h_out.data_ptr(), h_log.data_ptr(), B, S, S,
                                               1, 0, int(model.chunk_size), float(model.blender.scaling_i), float(model.blender.scaling_w), flags))

        for i in range(3):
            e2e_step(i)
        sync_all()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n_e2e = max(5, args.steps // 2)
        for i in range(n_e2e):
            e2e_step(i)
        e1.record()
        sync_all()
        e_ms = (time.perf_counter() - t0) * 1000.0   # the calls are synchronous and use the library's own streams
        if world > 1:
            t = torch.tensor([e_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e_ms = t.item()
        e2e = {"value": world * B * n_e2e / (e_ms / 1000.0), "unit": "frames/s",
               "h2d_bytes_per_step": B * 3 * S * S * 4 + B * K, "d2h_bytes_per_step": B * 3 * S * S * 4 + B * (1 + K) * 4,
               "path": "vsb_embed_detect_host: pinned host frames in, watermarked frames + logits out; H2D in slices (16 frames, then 48), "
                       "embed per slice, D2H of a slice under the following compute, detect per 64 accumulated frames (3 streams); timed by "
                       "host wall clock around the synchronous calls"}
        # the streaming caller's RGB24 form of the same call (SURVEY 8(f)1, inference_streaming.py): uint8 HWC frames over PCIe,
        # conversions on the GPU; the detector sees the re-quantised frames.  Reported next to the fp32-API number, not instead.
        u_in = [torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8, generator=g).pin_memory() for _ in range(2)]
        u_out = torch.empty(B, S, S, 3, dtype=torch.uint8).pin_memory()

        def u8_step(i):
            _lib.check(L.vsb_frames_host_u8(h, u_in[i % 2].data_ptr(), h_msgs.data_ptr(), B, u_out.data_ptr(), h_log.data_ptr(), B, S, S,
                                            1, 0, int(model.chunk_size), float(model.blender.scaling_i), float(model.blender.scaling_w), flags))

        for i in range(3):
            u8_step(i)
        sync_all()
        t0 = time.perf_counter()
        for i in range(n_e2e):
            u8_step(i)
        sync_all()
        u_ms = (time.perf_counter() - t0) * 1000.0
        if world > 1:
            t = torch.tensor([u_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            u_ms = t.item()
        e2e["u8_frames"] = {"value": world * B * n_e2e / (u_ms / 1000.0), "unit": "frames/s",
                            "h2d_bytes_per_step": B * 3 * S * S + B * K, "d2h_bytes_per_step": B * 3 * S * S + B * (1 + K) * 4,
                            "path": "vsb_frames_host_u8: RGB24 frames in and out, uint8<->float on the GPU"}

    # ---- per-kernel profile (CUDA events around every plan step) -> roofline of the dominant kernel
    roofline, table = None, []
    if rank == 0:
        L.vsb_profile_enable(1)
        for i in range(3):
            step_local(i)      # rank 0 only: no collective inside
        torch.cuda.synchronize()
        n = L.vsb_profile_read(None, 0)
        buf = C.create_string_buffer(int(n) + 16)
        L.vsb_profile_read(buf, len(buf))
        L.vsb_profile_enable(0)
        tot = 0.0
        for line in buf.value.decode().splitlines():
            name, tms, cnt = line.split("\t")
            tms, cnt = float(tms), int(cnt)
            fl = conv_flops(name, B, n_keys)
            table.append({"name": name, "ms_per_step": tms / 3, "launches_per_step": cnt // 3, "avg_us": 1000 * tms / cnt,
                          "tflops": (fl / (tms / cnt * 1e-3) / 1e12) if fl else None})
            tot += tms / 3
        table.sort(key=lambda r: -r["ms_per_step"])
        for r in table:
            r["share"] = r["ms_per_step"] / tot if tot else 0
        peaks = load_peaks()
        dom = next((r for r in table if r["tflops"]), None)
        if dom:
            # the kernel is event-timed launch by launch at full clock (clocks line: 1965 MHz, no power cap inside these 3 steps),
            # so the denominator is the BURST cuBLAS figure; the sustained one is reported next to it
            # finalize_op (conv_gemm_host.cuh) sends 3x3 TMA convs with >= 24 K blocks (C_in >= 192) on whole-row tiles to the CTA-pair kernel
            mm = re.match(r"unet\.conv3x3\.(\d+)-", dom["name"])
            pair = bool(mm) and int(mm.group(1)) >= 192 and not os.environ.get("VSB_NO_PAIR")
            roofline = {"bound": "tensor", "kernel": ("conv_pair_kernel (tcgen05 cta_group::2) " if pair else "conv_gemm_kernel<LD_TMA> ") + dom["name"],
                        "achieved": dom["tflops"],
                        "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": dom["tflops"] / peaks["tf_burst"],
                        "peak_source": peaks["src"] + " bf16 cuBLAS, burst (kernel event-timed per launch at full clock)",
                        "frac_of_sustained_peak": dom["tflops"] / peaks["tf_sustained"],
                        "share_of_step": dom["share"], "avg_launch_us": dom["avg_us"],
                        "traffic": ncu_traffic(f"{args.card}:{dom['name']}@b{B}"),
                        "traffic_source": "dram__bytes_read+write per launch from the committed ncu --set full capture (profiles/ncu_traffic.json)",
                        "step_ms_under_events": tot}
        if args.profile_out:
            json.dump({"batch": B, "card": args.card, "table": table}, open(args.profile_out, "w"), indent=1)

    # ---- HBM-bound half of the path (SURVEY 8(d): "report both"): the full-resolution stage (resize, JND / blend) only shows at
    #      inputs larger than the processing size, so rank 0 also runs a few steps of the same model on 3x768x768 frames with the
    #      per-launch event profile on and reports achieved GB/s of those kernels against the measured copy bandwidth
    roofline_hbm = None
    if rank == 0 and not args.no_hbm_leg:
        HS, HB = (768, 32) if S != 768 else (S, B)
        gi = [torch.rand(HB, 3, HS, HS, generator=g).to(dev) for _ in range(2)]     # 2 x 226 MB > 126 MB L2
        hm = msgs[:HB] if not vid else msgs_v

        def hbm_step(i):
            o = model.embed(gi[i % 2], hm if not vid else msgs_v, is_video=vid)
            model.detect(o["imgs_w"], is_video=vid)

        for i in range(3):
            hbm_step(i)
        torch.cuda.synchronize()
        L.vsb_profile_enable(1)
        for i in range(3):
            hbm_step(i)
        torch.cuda.synchronize()
        n = L.vsb_profile_read(None, 0)
        buf = C.create_string_buffer(int(n) + 16)
        L.vsb_profile_read(buf, len(buf))
        L.vsb_profile_enable(0)
        peaks = load_peaks()
        rows, tot_b, tot_ms, all_ms = [], 0.0, 0.0, 0.0
        for line in buf.value.decode().splitlines():
            name, tms, cnt = line.split("\t")
            tms, cnt = float(tms), int(cnt)
            all_ms += tms / 3
            if not name.startswith("pw."):
                continue
            by = pointwise_bytes(name, model.spec["img_size"])
            gbs = by / (tms / cnt * 1e-3) / 1e9 if by else None
            rows.append({"name": name, "avg_us": 1000 * tms / cnt, "launches_per_step": cnt // 3, "algorithmic_bytes": by,
                         "gbs": gbs, "frac": gbs / peaks["hbm_gbs"] if gbs else None,
                         "traffic": ncu_traffic(f"{args.card}:{name}")})
            tot_b += by * cnt / 3
            tot_ms += tms / 3
        rows.sort(key=lambda r: -r["avg_us"] * r["launches_per_step"])
        if rows:
            top = rows[0]
            roofline_hbm = {"bound": "hbm", "kernel": top["name"], "achieved": top["gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": top["frac"], "peak_source": peaks["src"] + " copy bandwidth",
                            "traffic": ncu_traffic(f"{args.card}:{top['name']}"),
                            "workload": f"{args.card} embed+detect, {'video' if vid else 'image'} mode, {HB} x 3x{HS}x{HS}",
                            "stage_gbs": tot_b / (tot_ms * 1e-3) / 1e9 if tot_ms else None,
                            "stage_frac": (tot_b / (tot_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if tot_ms else None,
                            "stage_ms_per_step": tot_ms, "step_ms_under_events": all_ms, "kernels": rows}
        del gi

    # ---- BASELINE configs[2]: the 512-frame 3x768x768 clip sharded over the ranks with the NCCL all-gather of the outputs
    clip = None
    if not args.no_clip_leg:
        clip = clip_leg(model, dev, world, rank, args.clip_frames, 768, max(3, args.steps // 4))

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        v, times, threads, sample = cpu_oracle_fps(args.card, S, 3, budget_s=25.0)
        cpu = {"value": v, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"{sample} frames embed+detect per run, 1 warm-up + 3 runs ({sum(times):.1f} s), oracle/restate.py"}

    if rank == 0:
        fe, fd = FLOPS_PER_FRAME.get(args.card, (0, 0))
        line = {
            "metric": "embed+detect frames/sec", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16 operands, f32 accumulate (API tensors f32)", "data": "synthetic",
            "config": {"workload": f"{args.card} {K}-bit embed+detect, {'video (step ' + str(model.step_size) + ')' if vid else 'image'} mode, "
                                   f"batch {B} x 3x{S}x{S} per GPU" + (" (BASELINE configs[1])" if (B, S, vid, args.card) == (64, 256, False, "videoseal_1.0") else ""),
                       "card": args.card, "batch_per_gpu": B, "size": S, "parallelism": f"dp{world} (frames sharded, weak scaling)",
                       "l2": f"{NB} rotating input batches ({NB * B * 3 * S * S * 4 / 1e6:.0f} MB > 126 MB L2); activations per step >> L2"},
            "step_tflops": (fe * n_keys + fd * B) * world * args.steps / (ms / 1000.0) / 1e12,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "roofline_hbm": roofline_hbm, "clip": clip, "cpu_baseline": cpu,
            "dumped_outputs": dumped,
            "top_kernels": [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()} for r in table[:8]],
        }
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
