#!/usr/bin/env python
"""bench.py — Msamples/s (and Mrays/s) of the rendering hot path on N B200s, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--spp S] [--impl ours|reference]

A "step" is one full render of the workload.  Default workload = BASELINE.json configs[4], the heaviest one and the one
north_star shards: examples/part2_all.rs at 3840x2160, with a FIXED total of `--spp` samples per pixel (default 512; the
config names 4096, which is 20 s per step on one GPU — one 32 Mi-path batch is already 4 spp at 4K, so throughput is
spp-invariant from a few dozen spp on and 512 keeps the driver's 25 + 20 steps inside its time limit; pass --spp 4096 for
the literal config).  STRONG scaling: the sample range is split over the ranks (`shard_range`), every rank renders ALL
pixels for its slice (RNG keyed by the global sample index), one NCCL reduce(SUM) of the 99.5 MB fp32 sum buffers to
rank 0, resolve on rank 0.  The other six BASELINE.json configs are measured in the same run at their own full sizes and
reported under `per_config`.

  value    : whole-job Msamples/s, scene already resident in HBM, device-timed (CUDA events on the launching stream,
             max over ranks)
  e2e      : same metric through the public call with HOST buffers each step: YAML text + host texels ->
             fw_scene_from_yaml -> fw_scene_commit (BVH build, H2D) -> render -> u8 image in host memory (D2H)
  roofline : extend kernels (closest-hit traversal), algorithmic FP32 flops per ray (SURVEY.md §8d formula with per-ray
             test counts measured by the oracle's counters) / CUDA-event time of the extend launches (measured in a
             separate profiled step, not inside the timed region), against the FP32 FMA peak measured on this GPU in this
             run; issue-slot view (IPC/4 x lanes/32) and DRAM traffic from the committed ncu capture of the same config
  reduce   : CUDA-event time of the NCCL reduce per step (N > 1)
  cpu_baseline : the C++ oracle ("port" — the Rust reference cannot be built here) on all host cores, bounded sample
  --impl reference : the same CPU port as the reference arm (rank 0 only); every step is a bounded sample of the workload
             and the line reports the times it measured.
  --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step of the headline workload returned —
             the resolved image and the fp32 sample sums — as DIR/image.npy and DIR/sum.npy (float32; of an image above
             DUMP_PIXELS pixels, a fixed seeded sample of pixels, listed in DIR/pixel_index.npy).  Inputs are fixed
             (committed scene, seed 1), so two builds run with the same arguments can be compared array for array.
"""
import argparse
import gzip
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

from firework_b200.assets import load_asset  # noqa: E402
from firework_b200.scenes import CONFIGS, SCENE_DIR  # noqa: E402

ASSETS = os.path.join(SCENE_DIR, "assets")
DEFAULT_WORKLOAD = "part2_all"   # BASELINE.json configs[4]: the config north_star shards over 1/2/4/8 GPUs
DEFAULT_SPP = {"part2_all": 512}  # total spp of the default run (see the docstring); other workloads: the config's own
BASELINE_CONFIGS = ["random_spheres", "cornell_box", "suzanne", "teapot", "hdri_test", "earth", "part2_all"]
PROFILE_TAG = "r02"              # profiles/<tag>_extend_traffic_<workload>.json (tools/ncu_traffic.py)

# SURVEY.md §8(d): static per-test operation / byte counts of the reference's routines
F_NODE, F_SPHERE, F_RECT, F_TRI, F_CONIC, F_XROT, F_XTRANS, F_SHADE = 27, 40, 12, 60, 50, 33, 3, 45
B_NODE, B_SPHERE, B_RECT, B_TRI, B_CONIC, B_XROT, B_XTRANS, B_RAY = 32, 16, 32, 48, 16, 112, 16, 64
HBM_BYTES_PER_RAY = 176  # wavefront streams per extend + shade round (queues carry the records, all coalesced):
                         # extend: ray 32 r + hit record 48 w;  shade: hit record 48 r + next ray 32 w + attenuation 16 w
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # 148 SMs x 128 lanes x 2 flop x 1.965 GHz = 74.4
DUMP_PIXELS = 1 << 20            # --dump-outputs keeps at most this many pixels: 2 x 12 MiB of float32 + 8 MiB of indices


def read_scene_text(cfg):
    p = cfg.path()
    with (gzip.open(p, "rt") if p.endswith(".gz") else open(p)) as f:
        return f.read()


def predecode_assets(text):
    """Decode every asset the document names once, into host memory (the e2e loop then only copies)."""
    from firework_b200.serde_yaml import loads
    doc = loads(text)
    out = {}

    def walk(n):
        if isinstance(n, dict):
            if n.get("texture") == "ImageTexture":
                out[n["value"]] = load_asset(n["value"], "image", ASSETS)
            if n.get("environment") == "HdrEnvironment":
                out[n["value"]] = load_asset(n["value"], "hdr", ASSETS)
            for v in n.values():
                walk(v)
        elif isinstance(n, list):
            for v in n:
                walk(v)

    walk({"materials": doc["materials"], "environment": doc["environment"]})
    return doc, out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_scene_for(doc, cfg, assets):
    from oracle.oracle import OracleScene
    return OracleScene(doc, cfg.use_bvh, asset_loader=lambda p, k: assets[p], fast=True)


def per_ray_work(st):
    """Algorithmic flops / bytes per ray from the oracle's counters (reference traversal semantics)."""
    r = max(st["rays"], 1)
    flops = (st["aabb_tests"] * F_NODE + st["sphere"] * F_SPHERE + st["rect"] * F_RECT + st["tri"] * F_TRI +
             st["conic"] * F_CONIC + st["xform_rot"] * F_XROT + st["xform_trans"] * F_XTRANS) / r + F_SHADE
    byts = (st["aabb_tests"] * B_NODE + st["sphere"] * B_SPHERE + st["rect"] * B_RECT + st["tri"] * B_TRI +
            st["conic"] * B_CONIC + st["xform_rot"] * B_XROT + st["xform_trans"] * B_XTRANS) / r + B_RAY
    return flops, byts, {"node_tests_per_ray": st["aabb_tests"] / r, "prim_tests_per_ray": st["prim_tests"] / r}


class CpuPort:
    """The C++ port of the reference's CPU path (oracle/, fast build) on all host cores of this box, over bounded
    samples of a workload: same scene, same resolution, reduced spp."""

    def __init__(self, cfg, doc, assets, width, height, spp):
        self.orc = oracle_scene_for(doc, cfg, assets)
        self.cfg, self.width, self.height, self.spp = cfg, width, height, spp
        self.threads = len(os.sched_getaffinity(0))   # all host cores (torchrun exports OMP_NUM_THREADS=1: override it)

    def run(self, n_spp, seed):
        r = self.cfg.renderer(width=self.width, height=self.height, samples=self.spp, seed=seed)
        _, _, st = self.orc.render(r.params(sample_begin=0, sample_count=n_spp), want_rgb=False, threads=self.threads)
        return st

    def spp_for(self, probe_stats, target_seconds):
        rate = probe_stats["samples"] / max(probe_stats["seconds"], 1e-6)
        return int(max(1, min(self.spp, target_seconds * rate / (self.width * self.height))))

    def describe(self, n):
        return f"{self.width}x{self.height} x {n} of {self.spp} spp"


def run_cpu(cfg, doc, assets, width, height, spp, target_seconds, seed):
    """One bounded sample.  Returns (Msamples/s, Mrays/s, stats of the timed pass, sample description, per-ray work)."""
    port = CpuPort(cfg, doc, assets, width, height, spp)
    st = port.run(1, seed)
    work = per_ray_work(st)
    n = port.spp_for(st, target_seconds)
    if n > 1 or st["seconds"] < 0.2:          # otherwise the 1-spp probe already is the bounded sample
        st = port.run(n, seed)
    return st["samples"] / st["seconds"] / 1e6, st["rays"] / st["seconds"] / 1e6, st, port.describe(n), work


def dump_outputs(out_dir, rgb, sums):
    """Writes a render's u8 image and fp32 sums (both (H, W, 3)) as out_dir/image.npy and out_dir/sum.npy in float32.  An
    image of more than DUMP_PIXELS pixels is reduced to the same fixed, seeded sample of pixels in both files, (n, 3) each,
    whose flat pixel indices (y * W + x) go to out_dir/pixel_index.npy (float64, exact)."""
    os.makedirs(out_dir, exist_ok=True)
    rgb, sums = rgb.astype(np.float32), sums.astype(np.float32)
    npix = rgb.shape[0] * rgb.shape[1]
    if npix > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(npix, DUMP_PIXELS, replace=False))
        rgb, sums = rgb.reshape(-1, 3)[idx], sums.reshape(-1, 3)[idx]
        np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "image.npy"), rgb)
    np.save(os.path.join(out_dir, "sum.npy"), sums)


def committed_profile(name, width, height, cfg):
    """ncu-derived facts of the extend kernels for this workload, from the committed capture (None if absent or if the
    run is not at the captured size): DRAM bytes per launch, busy lanes per instruction, IPC."""
    try:
        tj = json.load(open(os.path.join(REPO, "profiles", f"{PROFILE_TAG}_extend_traffic_{name}.json")))
    except Exception:
        return None
    if (width, height) != (cfg.width, cfg.height):
        return None
    return tj


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(CONFIGS))
    ap.add_argument("--spp", type=int, default=0, help="TOTAL samples per pixel, split over the ranks (default: see DEFAULT_SPP / the config)")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-config", action="store_true", help="skip the table of the other BASELINE.json configs")
    ap.add_argument("--per-config-steps", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the image and fp32 sums of the last timed step to DIR/*.npy (see the docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    cfg = CONFIGS[args.workload]
    width, height = args.width or cfg.width, args.height or cfg.height
    spp_total = args.spp or DEFAULT_SPP.get(cfg.name, cfg.samples)
    text = read_scene_text(cfg)
    doc, assets = predecode_assets(text)
    config = {"workload": f"{cfg.name} ({cfg.cite})", "width": width, "height": height, "spp_total": spp_total,
              "spp_of_named_config": cfg.samples, "use_bvh": cfg.use_bvh,
              "sharding": f"sample range [0, {spp_total}) split over {world} rank(s), every rank renders all pixels",
              "l2": "256 MiB device write between timed steps; per-batch path state (>1 GB) exceeds L2"}
    base = {"metric": "Msamples/s", "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (reference example scene restated; seeded generator where the example is random)",
            "config": config}

    # ------------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        # The reference is Rust and cannot be built in this image: the arm times the C++ port of its CPU path (oracle/),
        # all host threads, each step a bounded sample of the same workload (a few spp at the full resolution).  What is
        # printed is what was measured: `ms_per_step` is the mean wall time of those bounded steps, `value` their rate.
        port = CpuPort(cfg, doc, assets, width, height, spp_total)
        n_spp = port.spp_for(port.run(1, seed=12345), max(1.0, min(6.0, args.cpu_seconds / 4)))   # ~3 s of CPU work per step
        sample = port.describe(n_spp)
        samples = rays_n = secs_sum = 0.0
        secs, st = [], None
        for i in range(args.warmup + args.steps):
            st = port.run(n_spp, seed=i)
            if i >= args.warmup:
                samples += st["samples"]; rays_n += st["rays"]; secs_sum += st["seconds"]; secs.append(st["seconds"])
        v = samples / secs_sum / 1e6             # samples / seconds over the timed steps
        line = dict(base)
        line.update({"impl": "reference", "value": v, "mrays_per_s": rays_n / secs_sum / 1e6,
                     "ms_per_step": 1e3 * float(np.mean(secs)), "step_is": f"one bounded sample: {sample}",
                     "n_gpus": world, "cpu_scaling": "the CPU arm runs on rank 0's host cores only; it does not scale with --gpus",
                     "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": st["threads"], "kind": "port", "sample": sample},
                     "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "gpu_launches": 0})
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    from firework_b200.distributed import GpuShardRenderer
    from firework_b200.engine import NativeScene, measure_peaks

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allreduce(vals, op):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=op)
        return [float(x) for x in t]

    peaks = measure_peaks(local_rank)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    try:
        hbm_peak = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        hbm_peak = 6650.0

    def measure(c, w, h, spp, steps, warm, text_c, doc_c, assets_c, e2e_steps, cpu_seconds, sample_clocks, dump_dir=None):
        """Device-resident throughput, a separately profiled step, e2e through the host-buffer API, CPU port beside it."""
        ns = NativeScene(text_c, device=local_rank, assets=assets_c)
        renderer = c.renderer(width=w, height=h, samples=spp, seed=1)
        shard = GpuShardRenderer(ns, renderer, local_rank)
        npix = w * h
        tot = {"rays": 0, "launches": 0}

        def step(timed_reduce=None):
            img, total = shard.render(spp, rank, world, reduce_events=timed_reduce)
            st = shard.last_stats
            if st:
                tot["rays"] += st["rays"]; tot["launches"] += st["launches"]
            tot["launches"] += 1 if rank == 0 else 0   # resolve
            return img, total

        sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks) else None
        for _ in range(warm):
            step()
        barrier()
        tot["rays"] = tot["launches"] = 0
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        red = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)] if world > 1 else None
        t_wall0 = time.time()
        for i, (e0, e1) in enumerate(evs):
            # the previous step's buffers go back to the allocator first, so that every step reuses the same sum buffer:
            # with two buffers in turn, part2_all steps measured 0.4 % slower (B200, 1000 W power limit)
            outs = None
            flush_buf.fill_(1)          # evict L2 between timed steps (not timed)
            barrier()
            e0.record(shard.stream)     # every kernel of the step is launched on shard.stream
            outs = step(red[i] if red else None)
            e1.record(shard.stream)
        barrier()
        t_wall1 = time.time()
        clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
        ms_total = sum(e0.elapsed_time(e1) for e0, e1 in evs)
        ms_reduce = sum(a.elapsed_time(b) for a, b in red) if red else 0.0
        ms_total, ms_reduce = allreduce([ms_total, ms_reduce], dist.ReduceOp.MAX if world > 1 else None)
        rays_all, launches_all = allreduce([float(tot["rays"]), float(tot["launches"])], dist.ReduceOp.SUM if world > 1 else None)
        samples_all = float(npix) * spp * steps
        out = {"width": w, "height": h, "spp_total": spp, "value": samples_all / (ms_total * 1e-3) / 1e6,
               "mrays_per_s": rays_all / (ms_total * 1e-3) / 1e6, "ms_per_step": ms_total / steps,
               "rays_per_sample": rays_all / samples_all, "gpu_launches": int(launches_all), "steps": steps, "clocks": clocks}
        if world > 1:
            out["reduce"] = {"ms_per_step": ms_reduce / steps, "bytes": npix * 12, "what": "ncclReduce(SUM, fp32) of the sum buffers to rank 0 (torch.distributed), CUDA events around it, max over ranks"}
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, outs[0], outs[1].cpu().numpy().reshape(h, w, 3))
        outs = None

        # ---- one extra step with per-launch events around the extend kernels (never inside the timed region) -----
        ns.set_profiling(True)
        tot["rays"] = 0
        step()
        torch.cuda.synchronize()
        st = shard.last_stats or {"ms_extend": 0.0, "extend_launches": 0, "ms_device": 0.0, "rays": 0}
        ns.set_profiling(False)
        prof = {"ms_extend": st["ms_extend"], "extend_launches": st["extend_launches"], "rays": st["rays"], "ms_device": st["ms_device"]}

        # ---- e2e: host YAML text + host texels in, host u8 image out, every step ------------------------------
        def e2e_step():
            s = NativeScene(text_c, device=local_rank, assets=assets_c)      # parse, BVH build, flatten, H2D
            r2 = c.renderer(width=w, height=h, samples=spp, seed=1)
            if world == 1:
                rgb, _, _ = s.render(r2.params(), want_sum=False)            # render + D2H into a host buffer
                d2h = rgb.nbytes
            else:
                sh = GpuShardRenderer(s, r2, local_rank)
                rgb, _ = sh.render(spp, rank, world)
                d2h = rgb.nbytes if rgb is not None else 0
            h2d = s.device_bytes()
            s.close()
            return h2d, d2h

        def e2e_loop():
            e2e_step()
            barrier()
            t0 = time.perf_counter()
            h2d = d2h = 0
            for _ in range(e2e_steps):
                a, b = e2e_step()
                h2d, d2h = a, max(d2h, b)
            barrier()
            (e2e_s,) = allreduce([time.perf_counter() - t0], dist.ReduceOp.MAX if world > 1 else None)
            return float(npix) * spp * e2e_steps / e2e_s / 1e6, h2d, d2h

        e2e_v, h2d, d2h = e2e_loop()
        out["e2e"] = {"value": e2e_v, "unit": "Msamples/s",
                      "h2d_bytes_per_step": int(h2d) + len(text_c), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                      "what": "YAML text + host texels -> fw_scene_from_yaml + commit (BVH build, H2D) + render -> host u8 image (D2H)"}
        if assets_c:
            # the texture store shares a resident array with a scene that is handed the same texels again (every step here);
            # the same loop with the store off copies and uploads the texels every step
            os.environ["FW_TEXTURE_CACHE"] = "0"
            try:
                cold_v, cold_h2d, _ = e2e_loop()
            finally:
                del os.environ["FW_TEXTURE_CACHE"]
            out["e2e"]["texture_store"] = "on: texels already resident are shared, not uploaded (h2d_bytes_per_step counts what was copied)"
            out["e2e"]["texture_store_off"] = {"value": cold_v, "h2d_bytes_per_step": int(cold_h2d) + len(text_c)}
        ns.close()

        # ---- rank 0: per-ray algorithmic work from the oracle's counters (+ the CPU port's speed at N = 1) -----
        if rank == 0:
            tgt = cpu_seconds if (world == 1 and not args.no_cpu_baseline) else 0.0
            ms_cpu, mr_cpu, cst, sample, (flops_ray, bytes_ray, per_ray) = run_cpu(c, doc_c, assets_c, w, h, spp, tgt, seed=1)
            ext_s = max(prof["ms_extend"], 1e-9) * 1e-3
            ach = flops_ray * prof["rays"] / ext_s / 1e12
            nl = max(prof["extend_launches"], 1)
            pj = committed_profile(c.name, w, h, c)
            roof = {"bound": "fp32", "kernel": "extend kernels (closest hit)", "achieved": ach, "peak": peaks["fp32_tflops"],
                    "unit": "TFLOP/s", "frac": ach / peaks["fp32_tflops"], "frac_of_nominal_74.4": ach / FP32_NOMINAL_TFLOPS,
                    "traffic": pj["traffic_bytes_per_launch"] if pj else None,
                    "peak_source": "FP32 FMA microbenchmark on this GPU in this run (fw_measure_peaks); MEASURED_PEAKS.json has no FP32 figure; "
                                   "the path may not contract a*b+c (Rust semantics), so half of this is the reachable ceiling",
                    "flops_per_ray": flops_ray, "rays_per_launch": prof["rays"] / nl, "avg_launch_ms": prof["ms_extend"] / nl,
                    "extend_share_of_step": prof["ms_extend"] / max(prof["ms_device"], 1e-9),
                    "measured_in": "a separate profiled step after the timed region (per-launch CUDA events)", **per_ray}
            if pj:
                lanes, ipc = pj.get("threads_per_inst_time_weighted"), pj.get("ipc_per_sm_time_weighted")
                roof["issue_slots"] = {"lanes_of_32": lanes, "ipc_of_4": ipc, "useful_frac": (ipc / 4.0) * (lanes / 32.0) if lanes and ipc else None,
                                       "fma_pipe_pct": pj.get("fma_pipe_pct_time_weighted"), "alu_pipe_pct": pj.get("alu_pipe_pct_time_weighted"),
                                       "l1_hit_pct": pj.get("l1_hit_pct_time_weighted"), "registers": pj.get("registers"),
                                       "source": f"profiles/{PROFILE_TAG}_extend_traffic_{c.name}.json (ncu --set full of the extend launches of one batch)"}
            out["roofline"] = roof
            l2 = {"bound": "l2", "achieved": bytes_ray * prof["rays"] / ext_s / 1e9, "peak": peaks["l2_gbs"], "unit": "GB/s",
                  "bytes_per_ray": bytes_ray, "peak_source": "L2-resident 48 MiB streaming read on this GPU in this run"}
            if c.use_bvh:
                l2["frac"] = l2["achieved"] / l2["peak"]
            else:   # LinProgram scenes read their scene words from the constant bank, not L2: a ratio, not a fraction
                l2["ratio_not_a_fraction"] = l2["achieved"] / l2["peak"]
            out["roofline_l2"] = l2
            hb = HBM_BYTES_PER_RAY * rays_all / (ms_total * 1e-3) / 1e9 / world
            out["roofline_hbm"] = {"bound": "hbm", "achieved": hb, "peak": hbm_peak, "unit": "GB/s", "frac": hb / hbm_peak,
                                   "bytes_per_ray": HBM_BYTES_PER_RAY, "note": "wavefront state/queue streams; scene data is L2-resident"}
            if tgt > 0:
                out["cpu_baseline"] = {"value": ms_cpu, "unit": "Msamples/s", "mrays_per_s": mr_cpu, "cores": cst["threads"],
                                       "kind": "port", "sample": sample}
        return out

    main_res = measure(cfg, width, height, spp_total, args.steps, warmup, text, doc, assets, args.steps, args.cpu_seconds, True,
                       args.dump_outputs)

    per_config = {}
    if not args.no_per_config:
        for name in BASELINE_CONFIGS:
            c = CONFIGS[name]
            if name == cfg.name and (width, height, spp_total) == (c.width, c.height, DEFAULT_SPP.get(name, c.samples)):
                continue   # the headline line already is this config
            t_c = read_scene_text(c)
            d_c, a_c = predecode_assets(t_c)
            spp_c = DEFAULT_SPP.get(name, c.samples)
            r = measure(c, c.width, c.height, spp_c, args.per_config_steps, 3, t_c, d_c, a_c, args.per_config_steps,
                        min(4.0, args.cpu_seconds), False)
            if rank == 0:
                roof = r.get("roofline", {})
                per_config[name] = {
                    "res_spp": f"{c.width}x{c.height}x{spp_c}", "value": r["value"], "mrays_per_s": r["mrays_per_s"],
                    "ms_per_step": r["ms_per_step"], "e2e": r["e2e"]["value"], "e2e_over_value": r["e2e"]["value"] / r["value"],
                    "e2e_texture_store_off": (r["e2e"].get("texture_store_off") or {}).get("value"), "roofline_frac": roof.get("frac"),
                    "traffic": roof.get("traffic"), "lanes": (roof.get("issue_slots") or {}).get("lanes_of_32"),
                    "issue_useful_frac": (roof.get("issue_slots") or {}).get("useful_frac"),
                    "flops_per_ray": roof.get("flops_per_ray"), "extend_share_of_step": roof.get("extend_share_of_step"),
                    "cpu_port": (r.get("cpu_baseline") or {}).get("value"), "cpu_sample": (r.get("cpu_baseline") or {}).get("sample"),
                    "reduce_ms": (r.get("reduce") or {}).get("ms_per_step"), "gpu_launches": r["gpu_launches"]}

    if rank == 0:
        line = dict(base)
        for k in ("width", "height", "spp_total", "steps"):
            main_res.pop(k, None)
        line.update(main_res)
        roof = line.get("roofline", {})
        per_config[cfg.name] = {
            "res_spp": f"{width}x{height}x{spp_total}", "value": line["value"], "mrays_per_s": line["mrays_per_s"],
            "ms_per_step": line["ms_per_step"], "e2e": line["e2e"]["value"], "e2e_over_value": line["e2e"]["value"] / line["value"],
            "e2e_texture_store_off": (line["e2e"].get("texture_store_off") or {}).get("value"), "roofline_frac": roof.get("frac"),
            "traffic": roof.get("traffic"), "lanes": (roof.get("issue_slots") or {}).get("lanes_of_32"),
            "issue_useful_frac": (roof.get("issue_slots") or {}).get("useful_frac"), "flops_per_ray": roof.get("flops_per_ray"),
            "extend_share_of_step": roof.get("extend_share_of_step"), "cpu_port": (line.get("cpu_baseline") or {}).get("value"),
            "cpu_sample": (line.get("cpu_baseline") or {}).get("sample"), "reduce_ms": (line.get("reduce") or {}).get("ms_per_step"),
            "gpu_launches": line["gpu_launches"]}
        line["per_config"] = per_config
        line["peaks_measured"] = peaks
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
