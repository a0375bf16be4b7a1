#!/usr/bin/env python
"""bench.py -- frame-pairs aligned/s (640x480, 4-level pyramid) on N B200s, with roofline, CPU baseline and end-to-end figures.

Headline workload (BASELINE.json configs[1]): a batch of synthetic 640x480 RGB-D frame pairs per GPU, NEAREST 4-level
pyramid, Canny + exact EDT + packed distance texels (now frame), Canny + edge back-projection (reference frame),
Gauss-Newton on H = J^T W J / g = J^T W eps, 10 iterations per level, levels 3 -> 0.  One "step" = one pass of the whole hot
path over the batch.  Inputs are resident in HBM before the timed region (`value`); the `e2e` figure runs the same batch
through dvo_align_batch with pinned HOST buffers (H2D of the images and D2H of the poses inside the timed region).
Multi-GPU: frame pairs are partitioned across ranks (no data-path collective); NCCL all-gathers the 12-double pose records
once per step.

The other BASELINE configs are measured in the same run and reported under `other_configs`, each with its own value, e2e,
roofline, cpu_baseline and parity sample:
    config3  dense photometric estimator (Huber + LM), 1024 pairs 640x480              (dvo_photo_*)
    config4  1280x720, 5 levels, sub-gradient solver, consecutive-pair sequences         (dvo_run_sequences_mem)
    config5  16384 pairs partitioned across the ranks, NCCL pose gather (N > 1 only)     (strong scaling)

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--pairs P] [--solver gn|subgrad|lm]
                    [--dump-outputs DIR]

--steps sets the number of timed steps behind every config's `value` (the e2e legs time their own 2 to 5 passes).
--dump-outputs DIR writes what the headline path returned in its last timed step as DIR/<name>.npy: poses.npy (pairs x 12
float64: R row-major, then T; every rank's pairs in rank order) and the PairInfo fields of rank 0's pairs (status, npts,
best_index, iterations_run as float64; best_energy, visible_ratio, laplacian_b as the float32 the library returns).  With
--impl reference it writes the poses and status of the oracle's last step.  The inputs depend only on the arguments (seeded
synthetic pairs), so two builds can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np

W, H, LEVELS = 640, 480, 4
K = (525.0, 525.0, 319.5, 239.5)
PIX = sum((W >> l) * (H >> l) for l in range(LEVELS))        # 408000 px per frame
METRIC = "frame-pairs aligned/s (640x480, 4-lvl)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=1024, help="frame pairs per GPU per step")
    ap.add_argument("--solver", default="gn", choices=["gn", "subgrad", "lm"])
    ap.add_argument("--iters", type=int, default=None, help="iterations per level (default 10 for gn/lm, 50 for subgrad)")
    ap.add_argument("--arith", default="exact", choices=["exact", "fast"])
    ap.add_argument("--cpu-sample", type=int, default=48, help="pairs in the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="measure the headline config only")
    ap.add_argument("--total-pairs", type=int, default=16384, help="config5: pairs partitioned across all ranks")
    ap.add_argument("--sequences", type=int, default=148, help="config4: sequences per GPU")
    ap.add_argument("--seq-frames", type=int, default=8, help="config4: frames per sequence")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirpath, arrays):
    """Each array as dirpath/<name>.npy in float64 (float32 arrays stay float32)."""
    arrays = {k: np.asarray(v, np.float32 if np.asarray(v).dtype == np.float32 else np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(dirpath, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirpath, name + ".npy"), a)


def pair_info_arrays(info):
    """PairInfo records -> one array per field (per-level fields cut to the LEVELS levels in use)."""
    out = {"status": [inf.status for inf in info], "laplacian_b": np.array([inf.laplacian_b for inf in info], np.float32)}
    for f in ("npts", "best_index", "iterations_run"):
        out[f] = [list(getattr(inf, f))[:LEVELS] for inf in info]
    for f in ("best_energy", "visible_ratio"):
        out[f] = np.array([list(getattr(inf, f))[:LEVELS] for inf in info], np.float32)
    return out


def solver_setup(args):
    import oracle_lib as O
    it = args.iters or (50 if args.solver == "subgrad" else 10)
    iters = (it,) * LEVELS
    code = {"gn": 1, "subgrad": 0, "lm": 2}[args.solver]
    return iters, code, O.cfg(solver=code)


def rot_angle(Ra, Rb):
    return float(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1) / 2, -1, 1)))


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons while a timed region runs (NVML every 5 ms; nvidia-smi fallback)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples = index, False, []
        self.nvml = self._init_nvml()        # before the timed region: nvmlInit can take longer than a short timed region lasts

    def _init_nvml(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM); get_reasons(h)
            return pynvml, h, mx, get_reasons
        except Exception:
            return None

    def _sample_nvml(self):
        pynvml, h, mx, get_reasons = self.nvml
        bits = (0x8, 0x40, 0x20, 0x4)      # hw_slowdown, hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap
        try:
            r = int(get_reasons(h))
            self.samples.append([str(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), str(mx)] + ["Active" if r & b else "Not Active" for b in bits])
        except Exception:
            pass

    def run(self):
        if self.nvml is not None:
            while not self.stop_flag:
                self._sample_nvml()
                time.sleep(0.005)
            return
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def finish(self):
        self.stop_flag = True
        self.join(timeout=2)
        if not self.samples:                 # region shorter than one sampling period: one reading right behind it
            if self.nvml is not None:
                self._sample_nvml()
            else:
                try:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.samples.append([x.strip() for x in out.split(",")])
                except Exception:
                    pass
        return self.summary()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
            except Exception:
                continue
            for n, v in zip(names, s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(key):
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        return float(t[key]) if key in t else None
    except Exception:
        return None


def config_dict(args, iters, sample_note=None):
    c = {"workload": f"batched edge alignment: {args.pairs} synthetic 640x480 frame pairs per GPU, 4-level NEAREST pyramid, "
                     f"{args.solver} solver, {iters[0]} iterations/level (BASELINE configs[1])",
         "pairs_per_gpu": args.pairs, "width": W, "height": H, "levels": LEVELS, "solver": args.solver, "iters_per_level": iters[0],
         "arithmetic": args.arith, "l2": "inputs (1.2 MB/pair) larger than L2, no explicit flush",
         "schedule": "dvo_process: two staggered half batches on internal streams, steps issued back to back"}
    if sample_note:
        c["sample"] = sample_note
    return c


# ====================================================================================================== reference arm
def run_reference(args):
    """The reference arm: the CPU restatement of the reference's own path (it cannot be compiled here -- SURVEY 8c) on all
    host threads, same metric / config.  Each step is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib as O
    iters, code, ocfg = solver_setup(args)
    nthreads = os.cpu_count() or 1
    sample = max(nthreads, min(args.cpu_sample, 4 * nthreads))
    d = O.synth_batch(0, sample, W, H, K, nthreads=nthreads)
    times = []
    for s in range(args.warmup + args.steps):
        poses, status, secs = O.align_batch(d["ref_gray"], d["ref_depth"], d["now_gray"], LEVELS, iters, K, ocfg, nthreads=nthreads)
        if s >= args.warmup:
            times.append(secs)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"poses": poses, "status": status})
    per_step = float(np.mean(times))
    v = sample / per_step
    line = {"metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64",
            "data": "synthetic", "impl": "reference",
            "config": config_dict(args, iters, sample_note=f"each step = {sample} pairs (bounded sample of the {args.pairs}-pair batch)"),
            "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": nthreads, "kind": "port",
                             "sample": f"{sample} synthetic pairs per step, oracle port of SolveDVO (reference not compilable here)"},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ====================================================================================================== our arm
class Env:
    """Per-process distributed / stream plumbing shared by every config."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.numa = bind_to_gpu_numa_node(self.local) if self.world > 1 else None    # host buffers of the e2e legs next to this rank's GPU
        if self.world > 1:
            # NCCL prints its version banner on stdout when the communicator is created; stdout carries the one JSON line, so
            # file descriptor 1 points at stderr while the process group and its communicator come up
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
                dist.all_reduce(torch.zeros(1, device="cuda"))
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
        # a dedicated non-default stream shared by torch (events, NCCL) and the C-ABI contexts, so that the CUDA events are
        # recorded on the stream the kernels are launched on
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        self.nthreads = max(1, (os.cpu_count() or 1) // max(1, self.world))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        t = self.torch.tensor([ms], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, n, finish=None):
        """n calls of fn between two CUDA events on the launching stream, barrier + synchronize on both sides; ms per call, max over ranks."""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        for _ in range(n):
            fn()
        if finish:
            finish()
        e1.record(self.stream)
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1) / n)

    def pinned_h2d_peak_gbs(self, mbytes=512):
        """Measured pinned-host -> device copy rate of this rank (all ranks copy at the same time): the ceiling of every e2e leg."""
        torch = self.torch
        src = torch.empty(mbytes << 20, dtype=torch.uint8).pin_memory()
        dst = torch.empty(mbytes << 20, dtype=torch.uint8, device="cuda")
        dst.copy_(src, non_blocking=True)
        best = None
        for _ in range(3):
            ms = self.timed(lambda: dst.copy_(src, non_blocking=True), 1)
            best = ms if best is None else min(best, ms)
        return (mbytes << 20) / (best * 1e-3) / 1e9


def e2e_block(env, value, ms, h2d_bytes, d2h_bytes, pcie_peak, note=None):
    gbs = h2d_bytes / (ms * 1e-3) / 1e9
    out = {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes), "ms_per_step": ms,
           "h2d_gbs_per_gpu": gbs, "h2d_gbs_all_gpus": gbs * env.world, "pinned_copy_peak_gbs_per_gpu": pcie_peak,
           "pcie_frac": gbs / pcie_peak if pcie_peak else None}
    if note:
        out["note"] = note
    return out


def bench_config2(env, args):
    import oracle_lib as O            # synthetic renderer + the checker legs only (cpu_baseline, parity sample)
    import rgbd_odometry_b200 as dvo
    torch, dist = env.torch, env.dist
    rank, world, stream = env.rank, env.world, env.stream
    iters, code, ocfg = solver_setup(args)
    B = args.pairs
    t0 = time.time()
    data = O.synth_batch(rank * B, B, W, H, K, nthreads=env.nthreads)       # this rank's contiguous block of seeds
    t_synth = time.time() - t0
    al = dvo.BatchAligner(W, H, LEVELS, max_batch=B, device=env.local, intrinsics=K)
    al.set_stream(stream.cuda_stream)
    params = dvo.solver_params(solver=code, arithmetic=1 if args.arith == "fast" else 0, iters=iters)
    # inputs resident in HBM (the context's level-0 regions) before any timed region
    al.set_frames(dvo.FRAME_REF, data["ref_gray"], data["ref_depth"])
    al.set_frames(dvo.FRAME_NOW, data["now_gray"], None)
    # dvo_process runs the batch as two staggered half batches on internal streams and copies the poses into a device buffer
    # without joining, so back-to-back steps overlap.  The pose buffers alternate per step; the NCCL gather of step k runs on
    # its own stream after that step's work and step k+2 (which overwrites the same buffer) first waits for it.
    poses_buf = [torch.empty((B, 12), dtype=torch.float64, device="cuda") for _ in range(2)]
    gathered = torch.empty((world * B, 12), dtype=torch.float64, device="cuda") if world > 1 else None
    comm = torch.cuda.Stream() if world > 1 else None
    gather_done = [None, None]
    step_no = [0]

    def step():
        k = step_no[0] % 2
        step_no[0] += 1
        if gather_done[k] is not None:
            stream.wait_event(gather_done[k])
        al.process(B, params, poses_out=poses_buf[k].data_ptr())
        if world > 1:
            al.join_stream(comm.cuda_stream)
            with torch.cuda.stream(comm):
                dist.all_gather_into_tensor(gathered, poses_buf[k])
                ev = torch.cuda.Event()
                ev.record(comm)
            gather_done[k] = ev

    def finish_steps():
        al.join()
        if comm is not None:
            stream.wait_stream(comm)

    for _ in range(args.warmup):
        step()
    env.barrier()
    sampler = ClockSampler(env.local)
    sampler.start()
    l0 = al.launch_count()
    ms_max = env.timed(step, args.steps, finish_steps)
    launches = (al.launch_count() - l0)
    clocks = sampler.finish()
    value = world * B / (ms_max * 1e-3)

    # ---- parity of the timed batch: a fixed sample of its poses against the CPU oracle (the checker, not the thing measured)
    poses, info = al.get_poses(B)
    if args.dump_outputs and rank == 0:
        last = gathered if world > 1 else poses_buf[(step_no[0] - 1) % 2]
        dump_outputs(args.dump_outputs, {"poses": last.cpu().numpy(), **pair_info_arrays(info)})
    sample_idx = sorted(set([0, 1, B // 3, (2 * B) // 3, B - 1]))
    max_drad = max_dm = 0.0
    for i in sample_idx:
        o = O.align_pair(data["ref_gray"][i], data["ref_depth"][i], data["now_gray"][i], LEVELS, iters, K, scfg=ocfg)
        max_drad = max(max_drad, rot_angle(poses[i, :9].reshape(3, 3), o["R"]))
        max_dm = max(max_dm, float(np.linalg.norm(poses[i, 9:] - o["T"])))
    parity = {"n": len(sample_idx), "pairs": sample_idx, "max_drad": max_drad, "max_dm": max_dm, "tolerance": "1e-5 rad / 1e-5 m (north_star)",
              "ok": bool(max_drad < 1e-5 and max_dm < 1e-5)}

    # ---- per-stage device time (CUDA events on the launching stream), for the roofline of the dominant kernel
    al.enable_timing(True)
    nstage = 3
    for _ in range(nstage):
        al.build_pyramids(B); al.prepare(B); al.run(B, params)
    stage = {k: v / nstage for k, v in al.stage_ms().items()}
    al.enable_timing(False)
    stage["texels"] = stage.pop("normgrad")              # slot of the old normalise+gradient pass: pack_texel_kernel when it runs on its own
    fused = stage["texels"] == 0.0                       # 640x480: EDT rows and texel packing are one kernel, timed in the edt_rows slot
    if fused:
        stage["edt_rows+texels"] = stage.pop("edt_rows"); stage.pop("texels")
    npts = np.array([[inf.npts[l] for l in range(LEVELS)] for inf in info], dtype=np.int64)
    itrun = np.array([[inf.iterations_run[l] for l in range(LEVELS)] for inf in info], dtype=np.int64)
    n_total = int(npts.sum())
    iter_pts = int((npts * itrun).sum())
    # algorithmic bytes (SURVEY 8d): S1 pyramid 4P, S2 canny 4P, S3 EDT 5P, S4 distance texels 16P (survey figure for DTn+gx+gy;
    # the packed path moves 12), S5 points 3P + 12N, S6 24 * sum(I_L N_L)
    alg = {"pyramid": 4 * PIX * B, "canny": (4 + 3) * PIX * B + 12 * n_total, "edt_rows": 5 * PIX * B, "texels": 16 * PIX * B,
           "solve": 24 * iter_pts}
    if fused:
        alg["edt_rows+texels"] = alg.pop("edt_rows") + alg.pop("texels")
    bytes_pair = (32 * PIX * B + 12 * n_total + 24 * iter_pts) / B
    peak, peak_src = peaks()
    dom = "solve"
    dom_gbs = alg[dom] / (stage[dom] * 1e-3) / 1e9
    tr = ncu_traffic(f"solve_kernel_{args.solver}{iters[0]}_bytes_per_pair")
    roofline = {"bound": "hbm", "kernel": "solve_kernel", "achieved": dom_gbs, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                "frac": dom_gbs / peak, "traffic": tr * B if tr else None,
                "timing": "CUDA events around each stage on the launching stream, 3 staged steps run right after the timed region "
                          "(inside it the two half batches overlap on internal streams, so a kernel cannot be bracketed there)",
                "algorithmic_bytes_per_launch": alg[dom], "kernel_ms": stage[dom],
                "whole_path": {"bytes_per_pair": bytes_pair, "achieved_gbs": bytes_pair * B / (ms_max * 1e-3) / 1e9,
                               "frac": bytes_pair * B / (ms_max * 1e-3) / 1e9 / peak},
                "stages_ms": stage,
                "stages_gbs": {k: alg[k] / (stage[k] * 1e-3) / 1e9 for k in alg if stage.get(k, 0) > 0},
                "mean_points_per_pair": n_total / B, "mean_point_iterations_per_pair": iter_pts / B}

    # ---- end to end through the public C-ABI with pinned HOST buffers
    e2e = None
    pcie_peak = None
    if not args.no_e2e:
        pcie_peak = env.pinned_h2d_peak_gbs()
        pin = {k: torch.from_numpy(data[k]).pin_memory() for k in ("ref_gray", "ref_depth", "now_gray")}
        hp = {k: v.numpy() for k, v in pin.items()}
        al.align_batch(hp["ref_gray"], hp["ref_depth"], hp["now_gray"], params, want_info=False)
        n_e2e = max(2, min(args.steps, 5))
        ems = env.timed(lambda: al.align_batch(hp["ref_gray"], hp["ref_depth"], hp["now_gray"], params, want_info=False), n_e2e)
        e2e = e2e_block(env, world * B / (ems * 1e-3), ems, B * W * H * 4, B * 96, pcie_peak,
                        note="uploads in 128-pair chunks on a copy stream, chunk k+1's copy overlaps chunk k's kernels; the pass is bound by the host link")
        del pin, hp

    # ---- CPU baseline beside it (rank 0, N=1 only): the oracle port on the box's host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        nth = os.cpu_count() or 1
        sample = max(nth, min(args.cpu_sample, 4 * nth))

        def cpu_rate(n, threads):
            d = O.synth_batch(0, n, W, H, K, nthreads=threads)
            best = None
            for _ in range(3):
                _, _, secs = O.align_batch(d["ref_gray"], d["ref_depth"], d["now_gray"], LEVELS, iters, K, ocfg, nthreads=threads)
                best = secs if best is None else min(best, secs)
            return n / best
        cpu = {"value": cpu_rate(sample, nth), "unit": "pairs/s", "cores": nth, "kind": "port",
               "sample": f"{sample} synthetic pairs, best of 3, oracle port of SolveDVO built -O3 -march=native (reference not compilable here)",
               "single_core_pairs_per_s": cpu_rate(max(4, sample // max(1, nth)), 1)}
    status_nonzero = int(sum(1 for inf in info if inf.status != 0))
    al.close()
    del data
    return {"value": value, "ms_per_step": ms_max, "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "e2e": e2e, "parity_sample": parity, "synth_seconds": t_synth, "status_nonzero_pairs": status_nonzero, "iters": iters,
            "pcie_peak": pcie_peak}


def bench_config3(env, args, pcie_peak):
    """BASELINE configs[2]: dense photometric estimator (EPoseEstimator path, corrected formulation with Huber weights and LM
    damping), 1024 pairs 640x480, INTER_AREA pyramid levels 4 -> 0 x 6 iterations.  A step = BGR2GRAY + pyramids of both frames
    from device-resident BGR / depth, reference Jacobian normal matrix, the coarse-to-fine estimate."""
    import oracle_lib as O
    import rgbd_odometry_b200 as dvo
    torch = env.torch
    B, L3, iters3, hk, lam = args.pairs, 5, 6, 10.0, 1e-3
    d = O.synth_batch(100000 + env.rank * B, B, W, H, K, nthreads=env.nthreads, bgr=True)
    est = dvo.PhotoEstimator(W, H, L3, max_batch=B, device=env.local, intrinsics=K)
    est.set_stream(env.stream.cuda_stream)
    pin = {k: torch.from_numpy(d[k]).pin_memory() for k in ("ref_bgr", "now_bgr")}
    pin["ref_depth"] = torch.from_numpy(d["ref_depth"].view(np.int16)).pin_memory()
    dev = {k: v.cuda() for k, v in pin.items()}
    torch.cuda.synchronize()

    def solve():
        est.prepare_ref(B, compat=False)
        est.set_pose(B, None)
        for l in (4, 3, 2, 1, 0):
            est.estimate(B, l, iters=iters3, compat=False, huber_k=hk, lambda0=lam)

    def step_dev():
        est.set_frames(dvo.FRAME_REF, dev["ref_bgr"].data_ptr(), dev["ref_depth"].data_ptr(), count=B, device=True)
        est.set_frames(dvo.FRAME_NOW, dev["now_bgr"].data_ptr(), None, count=B, device=True)
        solve()

    # end to end: pinned host buffers, uploaded in 128-pair chunks on a copy stream into two staging sets so that chunk k+1 travels
    # while chunk k is converted and solved; poses read back at the end of the pass
    CH = min(128, B)          # 64 / 128 / 256 pairs per stage: 81.1 / 74.7 / 76.3 ms per pass
    copy_stream = torch.cuda.Stream()
    stage_buf = [{k: torch.empty((CH,) + tuple(v.shape[1:]), dtype=v.dtype, device="cuda") for k, v in pin.items()} for _ in range(2)]
    ev_up = [torch.cuda.Event() for _ in range(2)]
    ev_used = [None, None]

    def step_host():
        chunks = list(range(0, B, CH))

        def upload(i):
            c0 = chunks[i]; n = min(CH, B - c0); k = i & 1
            if ev_used[k] is not None:
                copy_stream.wait_event(ev_used[k])
            with torch.cuda.stream(copy_stream):
                for key in pin:
                    stage_buf[k][key][:n].copy_(pin[key][c0:c0 + n], non_blocking=True)
                ev_up[k].record(copy_stream)
        copy_stream.wait_stream(env.stream)
        upload(0)
        for i, c0 in enumerate(chunks):
            n = min(CH, B - c0); k = i & 1
            if i + 1 < len(chunks):
                upload(i + 1)
            env.stream.wait_event(ev_up[k])
            est.set_frames(dvo.FRAME_REF, stage_buf[k]["ref_bgr"].data_ptr(), stage_buf[k]["ref_depth"].data_ptr(), first=c0, count=n, device=True)
            est.set_frames(dvo.FRAME_NOW, stage_buf[k]["now_bgr"].data_ptr(), None, first=c0, count=n, device=True)
            ev_used[k] = torch.cuda.Event(); ev_used[k].record(env.stream)
            est.prepare_ref(n, first=c0, compat=False)
            est.set_pose(n, None, first=c0)
            for l in (4, 3, 2, 1, 0):
                est.estimate(n, l, iters=iters3, first=c0, compat=False, huber_k=hk, lambda0=lam)
        return est.get_poses(B)

    for _ in range(max(1, args.warmup - 1)):
        step_dev()
    sampler = ClockSampler(env.local); sampler.start()
    l0 = est.launch_count()
    nsteps = args.steps
    ms = env.timed(step_dev, nsteps)
    launches = est.launch_count() - l0
    clocks = sampler.finish()
    value = env.world * B / (ms * 1e-3)
    poses, info = est.get_poses(B)
    # dominant launches: the level-0 estimate (splat + accumulate per iteration); 28 B per pixel and iteration (SURVEY 8d photometric S6)
    est.prepare_ref(B, compat=False); est.set_pose(B, None)
    for l in (4, 3, 2, 1):
        est.estimate(B, l, iters=iters3, compat=False, huber_k=hk, lambda0=lam)
    ms_l0 = env.timed(lambda: est.estimate(B, 0, iters=iters3, compat=False, huber_k=hk, lambda0=lam), 1)
    it_run = float(np.mean([inf.iters_run for inf in est.get_poses(B)[1]]))
    alg = 28.0 * W * H * it_run * B
    peak, peak_src = peaks()
    roofline = {"bound": "hbm", "kernel": "ph_splat_kernel + ph_accum_kernel, level 0 (fp64 per-pixel warp, Jacobian row and 27 accumulations)",
                "achieved": alg / (ms_l0 * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": alg / (ms_l0 * 1e-3) / 1e9 / peak,
                "traffic": None, "algorithmic_bytes_per_launch": alg, "kernel_ms": ms_l0, "mean_iterations_level0": it_run,
                "note": "fp64-issue bound, not HBM bound: every pixel and iteration costs ~10 IEEE fp64 divisions kept for bit-parity with the oracle"}
    e2e = None
    if not args.no_e2e:
        step_host()
        ems = env.timed(step_host, 2)
        e2e = e2e_block(env, env.world * B / (ems * 1e-3), ems, B * W * H * (3 + 3 + 2), B * 12 * 8, pcie_peak)
    # CPU baseline + parity sample: the oracle's coarse-to-fine loop on the first pairs of this rank (single thread: the oracle keeps
    # the reference level in a global)
    cpu = parity = None
    if env.rank == 0 and not args.no_cpu_baseline:
        ns = 2
        t0 = time.time()
        max_drad = max_dm = 0.0
        for i in range(ns):
            Ro, To = np.eye(3), np.zeros(3)
            for l in (4, 3, 2, 1, 0):
                O.photo_build_ref_level(d["ref_bgr"][i], d["ref_depth"][i], l, K, compat=False)
                o = O.photo_estimate(O.photo_now_level(d["now_bgr"][i], l), Ro, To, iters3, K, compat=False, huber_k=hk, lambda0=lam)
                Ro, To = o["R"], o["T"]
            max_drad = max(max_drad, rot_angle(poses[i, :9].reshape(3, 3), Ro)); max_dm = max(max_dm, float(np.linalg.norm(poses[i, 9:] - To)))
        secs = time.time() - t0
        cpu = {"value": ns / secs, "unit": "pairs/s", "cores": 1, "kind": "port", "sample": f"{ns} pairs, levels 4..0 x {iters3} iterations, oracle port of the corrected EPoseEstimator"}
        parity = {"n": ns, "max_drad": max_drad, "max_dm": max_dm, "tolerance": "1e-5 rad / 1e-5 m", "ok": bool(max_drad < 1e-5 and max_dm < 1e-5)}
    err0 = float(np.mean(np.linalg.norm(d["T"], axis=1))); err1 = float(np.mean(np.linalg.norm(poses[:, 9:] - d["T"], axis=1)))
    est.close()
    return {"metric": "frame-pairs aligned/s (640x480, photometric Huber+LM, 5-lvl x 6 it)", "value": value, "unit": "pairs/s", "ms_per_step": ms,
            "steps": nsteps, "scaling": "weak", "dtype": "f64",
            "config": {"workload": f"dense photometric alignment (EPoseEstimator corrected formulation, Huber k={hk}, LM lambda0={lam}): {B} synthetic 640x480 BGR-D pairs per GPU, "
                                   f"INTER_AREA levels 4..0 x {iters3} iterations (BASELINE configs[2])", "pairs_per_gpu": B},
            "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu, "parity_sample": parity,
            "mean_translation_error_m": {"before": err0, "after": err1}}


def bench_config4(env, args, pcie_peak):
    """BASELINE configs[3]: 1280x720, 5-level pyramid, the shipped sub-gradient solver (50 iterations per level), consecutive-pair
    odometry with a key frame every 5 frames, batched over sequences (slot = sequence)."""
    import oracle_lib as O
    import rgbd_odometry_b200 as dvo
    torch = env.torch
    W4, H4, L4, K4 = 1280, 720, 5, O.K1280
    nseq, nframes = args.sequences, args.seq_frames
    iters4 = (50,) * L4
    t0 = time.time()
    with ThreadPoolExecutor(env.nthreads) as ex:
        seqs = list(ex.map(lambda s: O.synth_sequence(700000 + env.rank * nseq + s, nframes, W4, H4, K4, max_angle_deg=0.4, max_trans_m=0.008), range(nseq)))
    t_synth = time.time() - t0
    gray = torch.from_numpy(np.stack([s[0] for s in seqs])).pin_memory()
    depth = torch.from_numpy(np.stack([s[1] for s in seqs]).view(np.int16)).pin_memory()
    dgray, ddepth = gray.cuda(), depth.cuda()
    al = dvo.BatchAligner(W4, H4, L4, max_batch=nseq, device=env.local, keep_now_depth=True, intrinsics=K4)
    al.set_stream(env.stream.cuda_stream)
    prm = dvo.solver_params(iters=iters4)
    pol = dvo.keyframe_policy()
    run_dev = lambda: al.run_sequences_mem(dgray.data_ptr(), ddepth.data_ptr(), nseq, nframes, prm, pol, device=True)
    run_host = lambda: al.run_sequences_mem(gray.data_ptr(), depth.data_ptr(), nseq, nframes, prm, pol)
    rel, kind, reason, glob = run_dev()
    sampler = ClockSampler(env.local); sampler.start()
    l0 = al.launch_count()
    nrun = args.steps
    ms = env.timed(run_dev, nrun)
    launches = (al.launch_count() - l0) // nrun
    clocks = sampler.finish()
    fp = nseq * (nframes - 1)
    value = env.world * fp / (ms * 1e-3)
    e2e = None
    if not args.no_e2e:
        run_host()
        ems = env.timed(run_host, 2)
        e2e = e2e_block(env, env.world * fp / (ems * 1e-3), ems, nseq * nframes * W4 * H4 * 3, nseq * nframes * (12 + 19) * 8 + nseq * nframes * 8, pcie_peak,
                        note="frame t+1 of every sequence is uploaded on a copy stream while frame t is solved; every frame travels once (it is now, previous and reference in turn)")
        e2e["unit"] = "frame-pairs/s"
    # roofline of the solve on the data the sequence run left in the context (last frame against its key frame)
    al.set_initial_pose(nseq, None)
    al.run(nseq, prm)
    al.enable_timing(True)
    for _ in range(3):
        al.run(nseq, prm)
    st = al.stage_ms()["solve"] / 3
    al.enable_timing(False)
    _, info = al.get_poses(nseq)
    iter_pts = int(sum(info[i].npts[l] * info[i].iterations_run[l] for i in range(nseq) for l in range(L4)))
    peak, peak_src = peaks()
    tr = ncu_traffic("solve_kernel_1280x720_subgrad50_bytes_per_pair")
    roofline = {"bound": "hbm", "kernel": "solve_kernel (sub-gradient, 8 fp64 accumulators)", "achieved": 24.0 * iter_pts / (st * 1e-3) / 1e9, "peak": peak,
                "peak_source": peak_src, "unit": "GB/s", "frac": 24.0 * iter_pts / (st * 1e-3) / 1e9 / peak, "traffic": tr * nseq if tr else None,
                "algorithmic_bytes_per_launch": 24.0 * iter_pts, "kernel_ms": st, "mean_point_iterations_per_pair": iter_pts / nseq,
                "solver_threads_per_pair": 512 if nseq <= 148 else 256}
    # CPU baseline + parity: the oracle-driven loop over the first frames of a few sequences, one thread per sequence
    cpu = parity = None
    if env.rank == 0 and not args.no_cpu_baseline:
        ns, nf = min(nseq, max(2, min(8, os.cpu_count() or 1))), min(nframes, 3)
        g_np, d_np = gray.numpy(), depth.numpy().view(np.uint16)

        def one(s):
            R, T = np.eye(3), np.zeros(3)
            out = []
            for t in range(1, nf):
                o = O.align_pair(g_np[s, 0], d_np[s, 0], g_np[s, t], L4, iters4, K4, R0=R, T0=T)
                R, T = o["R"], o["T"]
                out.append((R, T))
            return out
        t0 = time.time()
        with ThreadPoolExecutor(ns) as ex:
            res = list(ex.map(one, range(ns)))
        secs = time.time() - t0
        max_drad = max_dm = 0.0
        for s in range(ns):
            for t in range(1, nf):
                R, T = res[s][t - 1]
                max_drad = max(max_drad, rot_angle(rel[s, t, :9].reshape(3, 3), R)); max_dm = max(max_dm, float(np.linalg.norm(rel[s, t, 9:] - T)))
        cpu = {"value": ns * (nf - 1) / secs, "unit": "frame-pairs/s", "cores": ns, "kind": "port",
               "sample": f"{ns} sequences x {nf - 1} frame pairs, one thread per sequence, oracle port of SolveDVO::loop"}
        parity = {"n": ns * (nf - 1), "max_drad": max_drad, "max_dm": max_dm, "tolerance": "1e-5 rad / 1e-5 m", "ok": bool(max_drad < 1e-5 and max_dm < 1e-5)}
    Tw = np.stack([s[3] for s in seqs])
    err = float(np.linalg.norm(glob[:, -1, 9:12] - Tw[:, -1], axis=1).mean())
    al.close()
    return {"metric": "frame-pairs aligned/s (1280x720, 5-lvl, sub-gradient 50 it/lvl, sequences)", "value": value, "unit": "frame-pairs/s", "ms_per_step": ms,
            "steps": nrun, "scaling": "weak", "dtype": "f32+f64",
            "config": {"workload": f"{nseq} synthetic sequences x {nframes} frames of 1280x720 per GPU, 5-level NEAREST pyramid, SUBGRAD_REF 50 iterations/level, "
                                   "key frame every 5 frames = previous frame, pose reset + re-solve (BASELINE configs[3])",
                       "sequences_per_gpu": nseq, "frames": nframes, "intrinsics": list(K4), "keyframes_per_sequence": int((kind[0] == 2).sum()) + 1},
            "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu, "parity_sample": parity,
            "final_position_error_m_mean": err, "path_length_m_mean": float(np.linalg.norm(Tw[:, -1], axis=1).mean()), "synth_seconds": t_synth}


def bench_config5(env, args, pcie_peak):
    """BASELINE configs[4]: 16384 synthetic pairs = seeds 0..16383, contiguous block partition across the ranks (strong scaling), poses
    gathered with NCCL.  A rank keeps its block's level-0 images resident in HBM and streams them through a 2048-pair context."""
    import oracle_lib as O
    import rgbd_odometry_b200 as dvo
    from rgbd_odometry_b200 import shard
    torch, dist = env.torch, env.dist
    iters, code, ocfg = solver_setup(args)
    total = args.total_pairs
    start, count = shard.partition(total, env.world, env.rank)
    CH = min(2048, count)
    t0 = time.time()
    dev = {"ref_gray": torch.empty((count, H, W), dtype=torch.uint8, device="cuda"), "ref_depth": torch.empty((count, H, W), dtype=torch.int16, device="cuda"),
           "now_gray": torch.empty((count, H, W), dtype=torch.uint8, device="cuda")}
    first_block = None
    for c0 in range(0, count, 1024):                       # synthesise in blocks, keep only the device copy
        n = min(1024, count - c0)
        d = O.synth_batch(start + c0, n, W, H, K, nthreads=env.nthreads)
        if c0 == 0:
            first_block = {k: d[k][:2].copy() for k in ("ref_gray", "ref_depth", "now_gray")}
        dev["ref_gray"][c0:c0 + n] = torch.from_numpy(d["ref_gray"]).cuda()
        dev["ref_depth"][c0:c0 + n] = torch.from_numpy(d["ref_depth"].view(np.int16)).cuda()
        dev["now_gray"][c0:c0 + n] = torch.from_numpy(d["now_gray"]).cuda()
    t_synth = time.time() - t0
    al = dvo.BatchAligner(W, H, LEVELS, max_batch=CH, device=env.local, intrinsics=K)
    al.set_stream(env.stream.cuda_stream)
    params = dvo.solver_params(solver=code, iters=iters)
    poses_dev = torch.empty((count, 12), dtype=torch.float64, device="cuda")
    mx = max(shard.partition(total, env.world, r)[1] for r in range(env.world))
    pad = torch.zeros((mx, 12), dtype=torch.float64, device="cuda")
    gathered = torch.empty((env.world * mx, 12), dtype=torch.float64, device="cuda")
    P0 = W * H

    def step():
        for c0 in range(0, count, CH):
            n = min(CH, count - c0)
            al.set_frames(dvo.FRAME_REF, dev["ref_gray"].data_ptr() + c0 * P0, dev["ref_depth"].data_ptr() + c0 * P0 * 2, count=n, device=True)
            al.set_frames(dvo.FRAME_NOW, dev["now_gray"].data_ptr() + c0 * P0, None, count=n, device=True)
            al.process(n, params, poses_out=poses_dev.data_ptr() + c0 * 96)
        al.join()
        pad[:count] = poses_dev
        if env.world > 1:
            dist.all_gather_into_tensor(gathered, pad)

    step()
    sampler = ClockSampler(env.local); sampler.start()
    nsteps = args.steps
    ms = env.timed(step, nsteps)
    clocks = sampler.finish()
    parity = None
    if env.rank == 0:
        p = poses_dev[:2].cpu().numpy()
        max_drad = max_dm = 0.0
        for i in range(2):
            o = O.align_pair(first_block["ref_gray"][i], first_block["ref_depth"][i], first_block["now_gray"][i], LEVELS, iters, K, scfg=ocfg)
            max_drad = max(max_drad, rot_angle(p[i, :9].reshape(3, 3), o["R"])); max_dm = max(max_dm, float(np.linalg.norm(p[i, 9:] - o["T"])))
        parity = {"n": 2, "max_drad": max_drad, "max_dm": max_dm, "tolerance": "1e-5 rad / 1e-5 m", "ok": bool(max_drad < 1e-5 and max_dm < 1e-5)}
    al.close()
    return {"metric": METRIC, "value": total / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms, "steps": nsteps, "scaling": "strong", "dtype": "f32+f64",
            "config": {"workload": f"{total} synthetic 640x480 frame pairs (seeds 0..{total - 1}) partitioned in contiguous blocks across {env.world} ranks, "
                                   f"{args.solver} {iters[0]} iterations/level, NCCL all-gather of the poses (BASELINE configs[4])",
                       "pairs_this_rank": count, "context_pairs": CH, "inputs": "level-0 images of the whole block resident in HBM, device-to-device into the context per 2048-pair chunk"},
            "clocks": clocks, "parity_sample": parity, "synth_seconds": t_synth}


def run_ours(args):
    env = Env()
    torch, dist = env.torch, env.dist
    h = bench_config2(env, args)
    other = {}
    if not args.no_other_configs:
        for name, fn in (("config3_photometric_huber_lm", bench_config3), ("config4_sequences_1280x720", bench_config4)):
            try:
                other[name] = fn(env, args, h["pcie_peak"])
            except Exception as e:                                  # a failing extra leg must not take the headline line with it
                other[name] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()
        if env.world > 1:
            try:
                other["config5_partitioned_16384"] = bench_config5(env, args, h["pcie_peak"])
            except Exception as e:
                other["config5_partitioned_16384"] = {"error": f"{type(e).__name__}: {e}"}
    if env.rank == 0:
        line = {"metric": METRIC, "value": h["value"], "unit": "pairs/s", "n_gpus": env.world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64",
                "data": "synthetic", "config": config_dict(args, h["iters"]), "clocks": h["clocks"], "gpu_launches": h["gpu_launches"],
                "roofline": h["roofline"], "cpu_baseline": h["cpu_baseline"], "e2e": h["e2e"], "parity_sample": h["parity_sample"], "numa": env.numa,
                "synth_seconds": h["synth_seconds"], "status_nonzero_pairs": h["status_nonzero_pairs"], "other_configs": other}
        print(json.dumps(line))
    if env.world > 1:
        dist.destroy_process_group()


def bind_to_gpu_numa_node(local):
    """Pin this rank's threads (and so the first touch of its pinned host buffers) to the NUMA node its GPU hangs off:
    with 8 ranks uploading 1.26 GB per step each, buffers on the far socket halve the aggregate H2D rate.  Best effort:
    returns None when the topology is not visible (containers without /sys NUMA info)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bdf = bus.lower()
        if len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception:
        return None


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
