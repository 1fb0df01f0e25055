#!/usr/bin/env python
"""bench.py -- EPro-PnP hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config fused|lm_only|amis|dense|train]   # our arm
    python bench.py --impl reference [--gpus N] [--steps K] [--config ...]                          # CPU arm
    python bench.py ... --dump-outputs DIR     # also write what the last timed step returned, DIR/<name>.npy

Default = the headline metric: PnP objects/sec at (B = 4096 per GPU, N = 512, M = 512), BASELINE.json configs #3 / #5's
shape.  One "step" = one pass of the hot path over one batch of synthetic correspondence sets through ONE C-ABI call
(epnp_lm_amis_fused_f32: the warp-per-object LM kernel, then the CTA-per-object AMIS kernel, same stream), followed,
for N > 1, by the single gather of poses + log-weights.  Prints ONE JSON line (rank 0).  The other configs are
BASELINE.json's #2 (LM only, B = 1024), #3 (B = 1024), #4 (dense 64 x 64 coordinate map, B = 256) and the training step
(forward + backward through the drop-in classes); each prints the same line layout.

  value      objects/s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        the same through the host-buffer call (pinned host tensors; H2D of the inputs and D2H of the results inside
             the timed region), min / median / max over the timed steps as well
  roofline   the dominant kernel (amis_kernel; lm_warp_kernel for lm_only): algorithmic HBM bytes per launch / its
             launch time (CUDA events around that kernel alone, measured in this run) against MEASURED_PEAKS.json.
             The path is FP32-pipe bound, not HBM bound (DESIGN.md section 4): `issue` reports the kernel's executed
             warp-instructions (profiles/kernel_stats.json, from the committed ncu capture of the SAME SASS -- refused
             when the kernel's SASS fingerprint has changed since) per second against 148 SM x 4 schedulers x clock.
  cpu_baseline   the UNMODIFIED reference layer (oracle/_ref staged by oracle/stage_ref.py + oracle/pyro_shim) -- or the
             oracle port when it has not been staged -- on all host cores (one worker process per 4 cores, the objects
             are independent), bounded sample; rank 0, N = 1 only.

--dump-outputs DIR writes, after the timed steps, the arrays the last timed step returned as DIR/<name>.npy (float32;
at most DUMP_MAX_BYTES, else a fixed, seeded sample of objects); the training config adds dL/dx2d and dL/dw2d, which
the step leaves in the leaves' .grad.  Inputs and seeds depend only on the arguments, so two builds can be compared
output for output.  With N > 1 only rank 0's own objects are written, not the gathered full batch: a deliberate limit
(the gathered pose_opt / logw rows of rank 0 hold the same values).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "epro-pnp_b200"))

import torch  # noqa: E402

# name -> workload.  kind: "lm_amis" = epnp_lm_amis_fused_f32, "lm" = epnp_lm_solve_f32, "train" = forward + backward
CONFIGS = {
    "fused": dict(B=4096, N=512, M=512, I=4, lm_iter=10, fast=0, z_min=0.1, rel_delta=0.5, grid2d=False, kind="lm_amis",
                  metric="PnP objects/sec (B=4096,N=512,M=512)",
                  what="fused EProPnP6DoF.monte_carlo_forward: LM(10) + cov + AMIS(4x128)"),
    "lm_only": dict(B=1024, N=512, M=0, I=0, lm_iter=10, fast=0, z_min=0.1, rel_delta=0.5, grid2d=False, kind="lm",
                    metric="PnP objects/sec (B=1024,N=512,LM only)", what="BASELINE #2: LMSolver 10 iterations + covariance, no MC"),
    "amis": dict(B=1024, N=512, M=512, I=4, lm_iter=10, fast=0, z_min=0.1, rel_delta=0.5, grid2d=False, kind="lm_amis",
                 metric="PnP objects/sec (B=1024,N=512,M=512)", what="BASELINE #3: LM(10) init + AMIS(4x128)"),
    "dense": dict(B=256, N=4096, M=512, I=4, lm_iter=3, fast=1, z_min=0.01, rel_delta=0.1, grid2d=True, kind="lm_amis",
                  metric="PnP objects/sec (B=256,N=4096,M=512)",
                  what="BASELINE #4: dense 64x64 coordinate map, AdaptiveHuber(0.1), GN(3) + AMIS(4x128) (lib/test.py:148-229)"),
    "train": dict(B=4096, N=512, M=512, I=4, lm_iter=10, fast=0, z_min=0.1, rel_delta=0.5, grid2d=False, kind="train",
                  metric="PnP training objects/sec (B=4096,N=512,M=512)",
                  what="training step through the drop-in classes: set_param, monte_carlo_forward (pose_init given), "
                       "MonteCarloPoseLoss, backward to x3d / x2d / w2d"),
}
E2E_CHUNKS = int(os.environ.get("EPNP_E2E_CHUNKS", "8"))   # object chunks of the host-buffer pipeline (0 = whole waves)
# host-buffer calls in flight: consecutive steps rotate over this many (stream, workspace, pinned result set) triples, so
# step i+1's upload runs under step i's solve and step i-1's download.  3 calls x 8 chunks was the configuration with the
# smallest box-to-box spread (2.0 M objects/s on both boxes measured; profiles/r2_e2e_sweep*.txt -- the upload bandwidth
# of pinned memory varies between 20 and 55 GB/s from box to box and size to size, which is what e2e mostly measures)
E2E_LANES = max(1, int(os.environ.get("EPNP_E2E_LANES", "3")))
WARM_SECONDS = 0.5            # minimum duration of back-to-back warm-up launches before the timed region
# allocate the pinned host buffers while the thread is bound to the CPUs NVML reports as local to the GPU (first touch
# puts the pages on the GPU's NUMA node; a remote node costs upload bandwidth)
E2E_NUMA = os.environ.get("EPNP_E2E_NUMA", "1") == "1"
L2_BYTES = 126e6
DUMP_MAX_BYTES = 64_000_000   # --dump-outputs writes at most this many bytes, .npy headers included


class gpu_local_cpus:
    """Context manager: bind the calling thread to the GPU's CPU affinity mask (NVML), restore on exit.  Best effort:
    any failure (no NVML, restricted cpuset) leaves the affinity untouched; `.applied` says what happened."""

    def __init__(self, index, enabled):
        self.index, self.enabled, self.applied, self.saved = index, enabled, None, None

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
            self.saved = os.sched_getaffinity(0)
            cpus &= self.saved
            if cpus:
                os.sched_setaffinity(0, cpus)
                self.applied = len(cpus)
        except Exception as exc:                           # noqa: BLE001 -- measurement aid only
            self.applied = f"unavailable: {type(exc).__name__}"
        return self

    def __exit__(self, *exc):
        if self.saved is not None:
            try:
                os.sched_setaffinity(0, self.saved)
            except OSError:
                pass
        return False



def algorithmic_bytes_per_object(cfg, kernel):
    """SURVEY.md section 8(d).  amis_kernel: read 28 N (correspondences) + 36 (K) + 4 (delta) + 28 (pose) + 144 (cov),
    write 28 M (samples) + 4 M (log-weights).  lm_warp_kernel: read 28 N + 36 + 4 + 28 (pose_init), write 28 (pose) + 144
    (cov) + 4 (cost).  The fused call = both (the correspondences are read once by each kernel)."""
    n, m = cfg["N"], cfg["M"]
    lm = 28 * n + 36 + 4 + 28 + 28 + 144 + 4
    amis = 28 * n + 36 + 4 + 28 + 144 + 28 * m + 4 * m
    return dict(lm_warp_kernel=lm, amis_kernel=amis)[kernel]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def kernel_stats(kernel, cfg_name):
    """Per-launch numbers of `kernel` from the committed ncu capture (profiles/kernel_stats.json, written by
    tools/ncu_summary.py): executed warp-instructions and DRAM bytes -- ONLY if the kernel's SASS in the library that
    is about to be timed is bit-identical to the SASS that was profiled.  Otherwise (None, why)."""
    path = os.path.join(ROOT, "profiles", "kernel_stats.json")
    if not os.path.exists(path):
        return None, "no profiles/kernel_stats.json"
    try:
        rec = json.load(open(path)).get(f"{kernel}@{cfg_name}")
        if rec is None:
            return None, f"no capture of {kernel} at config {cfg_name}"
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import sass_identity
        have = sass_identity.fingerprints(sass_identity.DEFAULT_LIB)
        sha = {k: v["sha1"] for k, v in have.items() if rec["sass_symbol"] in k}
        if rec["sass_sha1"] not in sha.values():
            return None, "stale: the kernel's SASS changed since the capture (re-profile, tools/ncu_summary.py)"
        return rec, "profiles/kernel_stats.json (same SASS fingerprint)"
    except Exception as ex:                                # noqa: BLE001
        return None, f"unavailable: {type(ex).__name__}: {ex}"


class ClockSampler:
    """nvidia-smi sampled every 50 ms in the background; only samples whose timestamp falls inside the
    timed region [t0, t1] (host wall clock) are summarised."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def wait_ready(self, timeout=8.0):
        """Block until the first sample has been written: nvidia-smi's start-up (it attaches to every GPU of the
        box) takes 0.1-2 s and stalls running kernels for tens of ms -- that must be over before anything is timed."""
        if self.proc is None:
            return
        t0 = time.time()
        while time.time() - t0 < timeout:
            try:
                if os.path.getsize(self.path) > 0:
                    return
            except OSError:
                return
            time.sleep(0.02)

    def stop(self, t0, t1):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            time.sleep(0.12)
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [[c.strip() for c in r.split(",")] for r in open(self.path).read().strip().splitlines() if r.strip()]
            inside = []
            for r in rows:
                try:
                    ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except Exception:
                    continue
                if t0 - 0.03 <= ts <= t1 + 0.03:
                    inside.append(r)
            use = inside if inside else rows
            sm = [float(r[1]) for r in use]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = sorted({names[i] for r in use for i in range(4)
                              if len(r) >= 8 and "Active" in r[4 + i] and "Not" not in r[4 + i]})
            if sm:
                out = {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": float(use[0][2]),
                       "reasons": reasons, "samples": len(sm), "samples_in_timed_region": len(inside),
                       "power_w_max": max(float(r[3]) for r in use)}
        except Exception as ex:   # noqa: BLE001
            out["error"] = repr(ex)
        finally:
            try:
                os.unlink(self.path)
            except Exception:
                pass
        return out



# ------------------------------------------------------------------------------------------------ CPU arm
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_reference_rates(cfg, steps, warmup, seconds_per_step, threads_per_worker=4):
    """objects/s of the reference's own CPU path on ALL host cores, per step.  One worker process per
    `threads_per_worker` cores (oracle/ref_worker.py; the objects are independent, and the reference's batched torch ops
    stop scaling long before 128 threads in one process); every worker runs `warmup + steps` slices of `seconds_per_step`
    on its own bounded sample and reports objects / seconds per slice; a step's rate is the sum over the workers."""
    cores = host_cores()
    nproc = max(1, cores // threads_per_worker)
    per = 16 if cfg["N"] <= 1024 else 2          # objects per pass and worker
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_worker.py"), "--objects", str(per), "--threads",
           str(threads_per_worker), "--points", str(cfg["N"]), "--samples", str(max(cfg["M"], cfg["I"] or 1)),
           "--mc-iter", str(cfg["I"] or 1), "--lm-iter", str(cfg["lm_iter"]), "--config",
           "lm_only" if cfg["kind"] == "lm" else "fused", "--slices", str(steps + warmup), "--seconds", str(seconds_per_step)]
    if cfg["fast"]:
        cmd += ["--fast-mode", "--z-min", str(cfg["z_min"]), "--rel-delta", str(cfg["rel_delta"]), "--grid2d"]
    env = dict(os.environ, OMP_NUM_THREADS=str(threads_per_worker), MKL_NUM_THREADS=str(threads_per_worker), CUDA_VISIBLE_DEVICES="")
    procs = [subprocess.Popen(cmd + ["--seed", str(5 + i)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
             for i in range(nproc)]
    outs = []
    for p in procs:
        so, se = p.communicate()
        line = [l for l in so.splitlines() if l.startswith("{")]
        if p.returncode == 0 and line:
            outs.append(json.loads(line[-1]))
    if not outs:
        raise RuntimeError("no CPU worker finished: " + (se or "")[-400:])
    rates = [sum(o["slices"][s][0] / o["slices"][s][1] for o in outs) for s in range(warmup, warmup + steps)]
    kind = outs[0]["kind"]
    sample = (f"{len(outs)} worker processes x {threads_per_worker} threads = {len(outs) * threads_per_worker} of {cores} host cores; "
              f"each worker: passes of {per} objects (N={cfg['N']}, M={cfg['M']}, LM {cfg['lm_iter']}"
              f"{' + AMIS ' + str(cfg['I']) + 'x' + str(cfg['M'] // cfg['I']) if cfg['M'] else ''}) for {seconds_per_step:.1f} s per step, fp32; "
              f"{'EProPnP6DoF.monte_carlo_forward of the unmodified reference (oracle/_ref) + pyro shim' if kind == 'reference+shim' else 'oracle port (reference not staged)'}")
    return rates, len(outs) * threads_per_worker, kind, sample


def rotating_sets(cfg):
    """(number of rotating input sets, bytes of one set): enough that consecutive steps cannot be served from the L2."""
    set_bytes = 28 * cfg["N"] * cfg["B"]
    return max(2, min(16, int(math.ceil(1.15 * L2_BYTES / set_bytes)) + 1)), set_bytes


def npy_bytes(a):
    """Size of the .npy file np.save writes for `a`: header + data."""
    import io
    import numpy as np
    buf = io.BytesIO()
    np.lib.format.write_array_header_1_0(buf, np.lib.format.header_data_from_array_1_0(a))
    return buf.tell() + a.nbytes


def host_outputs(out, n_obj):
    """--dump-outputs: the arrays of one step's result dict (absent ones skipped) as float32 / float64 numpy arrays.
    When their .npy files would come to more than DUMP_MAX_BYTES, every per-object array (leading dimension n_obj) keeps
    the same fixed, seeded sample of objects, in object order: the largest sample that fits."""
    import numpy as np
    arrs = {}
    for name, t in out.items():
        if t is not None:
            a = t.detach().cpu().numpy()
            arrs[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float32)
    per_obj = [name for name, a in arrs.items() if a.ndim and a.shape[0] == n_obj]
    total = sum(npy_bytes(a) for a in arrs.values())     # a sample's headers are no longer than these
    if total > DUMP_MAX_BYTES:
        obj_bytes = sum(arrs[name].nbytes for name in per_obj) // n_obj
        keep = (DUMP_MAX_BYTES - (total - obj_bytes * n_obj)) // obj_bytes
        idx = np.sort(np.random.default_rng(0).choice(n_obj, size=keep, replace=False))
        for name in per_obj:
            arrs[name] = arrs[name][idx]
    return arrs


def config_block(args, cfg, world):
    """The `config` object of the JSON line -- the SAME for both arms (`--impl ours` / `--impl reference`): it names the
    workload; what is specific to how the CPU arm samples it goes into that arm's `cpu_baseline.sample`."""
    n_sets, set_bytes = rotating_sets(cfg)
    Bg, M = cfg["B"], cfg["M"]
    gather = ""
    if world > 1 and cfg["kind"] == "lm_amis":
        gather = (f", gather(pose,logw) only ({args.gather}"
                  + (f", NCCL_MAX_CTAS={args.nccl_max_ctas}" if args.nccl_max_ctas else "") + ")"
                  + ("" if args.gather == "push" else ", gather of batch i overlapped with solve of batch i+1"))
    return {"workload": f"{cfg['what']}, B={Bg}/GPU, N={cfg['N']}, M={M}" + (", in-kernel Philox" if M else ""),
            "name": args.config, "global_batch": Bg * world, "parallelism": f"batch-split x{world}{gather}",
            "batches_in_flight": args.streams,
            "l2": f"rotating {n_sets} input sets ({n_sets * set_bytes / 1e6:.0f} MB > 126 MB L2)"}


def run_reference_arm(args, cfg, rank):
    if rank != 0:
        return
    # exactly K timed steps; the arm aims at about 2.5 minutes whatever K and W are, so a step's slice shrinks as K grows
    # (a worker's slice still runs at least one whole pass, so at large K the arm takes K + W passes)
    per_step = min(20.0, 140.0 / (args.steps + args.warmup))
    t0 = time.perf_counter()
    rates, cores, kind, sample = cpu_reference_rates(cfg, args.steps, args.warmup, per_step)
    el = time.perf_counter() - t0
    value = statistics.mean(rates)
    line = {"impl": "reference", "metric": cfg["metric"], "value": value, "unit": "objects/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(args, cfg, int(os.environ.get("WORLD_SIZE", "1"))),
            "cpu_baseline": {"value": value, "unit": "objects/s", "cores": cores, "kind": kind, "sample": sample,
                             "per_step_min_max": [min(rates), max(rates)], "wall_s": el},
            "e2e": {"value": value, "unit": "objects/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="fused", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--gather", default="push", choices=["nccl", "push"],
                    help="N > 1: 'push' = the AMIS kernel stores finished rows into every rank's result buffer over "
                         "NVLink (no gather kernel); 'nccl' = overlapped all_gather_into_tensor (the baseline it is measured against)")
    ap.add_argument("--nccl-max-ctas", type=int, default=0,
                    help="N > 1, --gather nccl: cap the CTAs NCCL may use per collective (0 = NCCL's default)")
    ap.add_argument("--streams", type=int, default=2,
                    help="batches in flight: consecutive (independent) batches are issued round-robin on this many CUDA streams, "
                         "so the next batch's LM kernel and first AMIS CTAs fill the SMs the previous batch's last, partial wave "
                         "of CTAs leaves idle (measured +4.4 %% at one GPU); 1 = strictly one batch at a time")
    ap.add_argument("--batch", type=int, default=0, help="objects per GPU (default: the config's)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the arrays the last timed step returned as DIR/<name>.npy, so that "
                         "two builds can be compared output for output on identical inputs (N > 1: rank 0's own objects only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    if args.batch > 0:
        cfg["B"] = args.batch
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return

    import torch.distributed as dist
    from epropnp_b200 import native
    from epropnp_b200.sharded import PushGather, gather_results_async
    from epropnp_b200.synth import make_problem

    torch.cuda.set_device(local_rank)
    # EPNP_BENCH_DEVICE exists for tests/test_bench_dryrun_cpu.py, which drives this loop on the SIMT-emulated library;
    # with the real library anything but "cuda" is refused by the native layer (no CPU path)
    dev = torch.device(os.environ.get("EPNP_BENCH_DEVICE", "cuda"), local_rank)
    saved_stdout = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if args.nccl_max_ctas > 0:
            os.environ["NCCL_MAX_CTAS"] = str(args.nccl_max_ctas)
        # NCCL prints its version banner on stdout at communicator creation; keep stdout = the one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    Bg, N_PTS, M, I = cfg["B"], cfg["N"], cfg["M"], cfg["I"]
    B_total = Bg * world
    kind = cfg["kind"]
    gathering = world > 1 and kind == "lm_amis"

    # ---- synthetic inputs of this rank's shard (global object index keys the RNG, rank keys the data seed); enough
    # rotating input sets that consecutive steps cannot be served from the 126 MB L2
    n_sets, set_bytes = rotating_sets(cfg)
    pc = make_problem(Bg, N_PTS, seed=1000 + rank, grid2d=cfg["grid2d"])
    sets = []
    for r in range(n_sets):
        shift = (r * Bg) // n_sets
        d = {k: torch.roll(v, shifts=shift, dims=0).to(dev).contiguous() for k, v in pc.items()}
        d["delta"] = native.adaptive_delta(d["x2d"], d["w2d"], cfg["rel_delta"])
        d["prob"] = native.Problem(d["x3d"], d["x2d"], d["w2d"], d["cam_mats"], None, None, d["delta"])
        sets.append(d)
    params = native.default_params(6, lm_iter=cfg["lm_iter"], fast_mode=cfg["fast"], z_min=cfg["z_min"],
                                   **({"mc_samples": M, "mc_iter": I} if M else {}))
    launches_per_step = {"lm_amis": 2, "lm": 1, "train": 5}[kind]

    train = None
    if kind == "train":
        from epropnp.camera import PerspectiveCamera
        from epropnp.cost_fun import AdaptiveHuberPnPCost
        from epropnp.epropnp import EProPnP6DoF
        from epropnp.levenberg_marquardt import LMSolver
        from epropnp.monte_carlo_pose_loss import MonteCarloPoseLoss
        layer = EProPnP6DoF(mc_samples=M, num_iter=I, solver=LMSolver(dof=6, num_iter=cfg["lm_iter"]))
        loss_fn = MonteCarloPoseLoss().to(dev)
        for d in sets:
            d["leaf"] = tuple(d[k].clone().requires_grad_(True) for k in ("x3d", "x2d", "w2d"))
            d["camera"] = PerspectiveCamera(cam_mats=d["cam_mats"], z_min=cfg["z_min"])

        def train(i):
            """One training step of the 6DoF flavour (EPro-PnP-6DoF/lib/train.py:170-200): adaptive delta from the
            weights, Monte-Carlo forward with the ground-truth pose as pose_init, MC pose loss, backward."""
            d = sets[i % n_sets]
            x3d, x2d, w2d = d["leaf"]
            x3d.grad = x2d.grad = w2d.grad = None
            cost_fun = AdaptiveHuberPnPCost(relative_delta=cfg["rel_delta"])
            cost_fun.set_param(x2d.detach(), w2d)
            # the AMIS seed follows the step index, as in solve(): without it each call draws one from torch's generator,
            # and the time-bounded warm-up would leave the timed steps on different seeds from run to run
            _, _, _, _, logw, cost_tgt = layer.monte_carlo_forward(x3d, x2d, w2d, d["camera"], cost_fun,
                                                                   pose_init=d["pose_gt"], force_init_solve=False,
                                                                   amis_seed=1234 + i)
            loss = loss_fn(logw, cost_tgt, 1.0)
            loss.backward()
            return {"loss": loss.detach(), "gx3d": x3d.grad}

    def solve(i):
        s = sets[i % n_sets]
        if kind == "lm":
            return native.lm_solve(s["prob"], s["pose_init"], params, want_cov=True, want_cost=True)
        if kind == "train":
            return train(i)
        return native.lm_amis_fused(s["prob"], s["pose_init"], params, seed=1234 + i, obj_offset=rank * Bg,
                                    want_cost=True, want_cost_init=False)

    pending = None
    push_gather = None
    lanes = [torch.cuda.Stream(dev) for _ in range(args.streams)] if args.streams > 1 else None
    k_ev = {}                       # step -> (event before, event after) around the solve's launches, timed region only
    timing = [False]

    def mark(i, which):
        if timing[0] and lanes is None and i < 64:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            k_ev.setdefault(i, [None, None])[which] = e

    def step(i):
        """One batch on its lane (stream i mod S) -- or on the current stream when S = 1."""
        if lanes is None:
            return step_on_current_stream(i)
        with torch.cuda.stream(lanes[i % len(lanes)]):
            return step_on_current_stream(i)

    def fork_lanes():
        if lanes is not None:
            for s in lanes:
                s.wait_stream(torch.cuda.current_stream(dev))

    def join_lanes():
        if lanes is not None:
            for s in lanes:
                torch.cuda.current_stream(dev).wait_stream(s)

    def step_on_current_stream(i):
        """One batch: the solve, then (N > 1) the gather of (pose_opt, logw).  The gather is asynchronous and the previous
        batch's is awaited only after this batch's solve is enqueued, so exchange i overlaps solve i+1 (batches are
        independent); every gather completes inside the timed region (drain() before t_end)."""
        nonlocal pending, push_gather
        if gathering and args.gather == "push":
            # solve + gather in one: the AMIS kernel stores every finished object's rows into all ranks' result buffers
            if push_gather is None:
                push_gather = PushGather(B_total, M, 7, dev)
            s = sets[i % n_sets]
            mark(i, 0)
            out, nxt = push_gather.solve(s["prob"], s["pose_init"], params, seed=1234 + i, want_cost=True, want_cov=True)
            mark(i, 1)
            if pending is not None:
                pending.wait()
            pending = nxt
            return out
        mark(i, 0)
        out = solve(i)
        mark(i, 1)
        if gathering:
            if pending is not None:
                pending.wait()
            pending = gather_results_async(out, B_total, keys=("pose_opt", "logw"))
        return out

    def drain():
        nonlocal pending
        if pending is not None:
            pending.wait()
            pending = None

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # clock sampler first: the nvidia-smi process takes 0.1-0.3 s to initialise and stalls the GPU while it does;
    # that must land in the warm-up, not in the timed region (samples are filtered by timestamp afterwards)
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("EPNP_NO_SAMPLER"):
        sampler.start()
        sampler.wait_ready()
    # warm-up: at least W steps AND at least ~0.5 s of back-to-back launches -- the first ~100 ms after an idle
    # period run measurably slower (power-state ramp), which W = 3 steps of 1 ms do not cover
    t_warm = None                # the 0.5 s start counting after the first chunk: it holds the one-off costs (module load,
    n_warm = 0                   # NCCL communicator / IPC set-up -- seconds at N > 1), which are not back-to-back launches
    out = None
    while True:
        out = step(n_warm)       # same liveness pattern as the timed loop (previous outputs alive while the next are
        n_warm += 1              # allocated), so torch's caching allocator is primed and never calls cudaMalloc later
        if n_warm % 16 == 0:
            torch.cuda.synchronize()
            # the stop decision must be COLLECTIVE: every rank has to run the same number of steps (= the same number
            # of gathers); ranks deciding on their own wall clocks deadlock the next collective
            if t_warm is None:
                t_warm = time.time()
            flag = torch.tensor([1.0 if (n_warm >= args.warmup and time.time() - t_warm >= WARM_SECONDS) else 0.0], device=dev)
            if world > 1:
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() > 0.5:
                break
    drain()
    fence()
    if saved_stdout is not None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    # ---- timed region: exactly K steps, one event pair around all of them
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    wall0 = time.time()
    timing[0] = True
    t_begin.record()
    fork_lanes()                   # lanes start after t_begin ...
    for i in range(args.steps):
        out = step(i)
    drain()
    join_lanes()                   # ... and t_end waits for every lane: all K batches complete inside the region
    t_end.record()
    fence()
    wall1 = time.time()
    timing[0] = False
    total_ms = t_begin.elapsed_time(t_end)
    dump = None
    if args.dump_outputs and rank == 0:
        last = out
        if kind == "train":
            # a caller of the training step receives all three gradients; train() returns only the loss and dL/dx3d,
            # which is what the end-to-end section downloads
            _, x2d, w2d = sets[(args.steps - 1) % n_sets]["leaf"]
            last = dict(out, gx2d=x2d.grad, gw2d=w2d.grad)
        dump = host_outputs(last, Bg)
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    # the solve's launches inside the loop (first 64 steps): their own duration, and the gap to the next step's launches
    in_loop = None
    if k_ev:
        ks = sorted(k for k, v in k_ev.items() if v[0] is not None and v[1] is not None)
        dur = [k_ev[k][0].elapsed_time(k_ev[k][1]) for k in ks]
        gap = [k_ev[a][1].elapsed_time(k_ev[b][0]) for a, b in zip(ks[:-1], ks[1:]) if b == a + 1]
        in_loop = {"solve_ms": statistics.mean(dur), "gap_ms": statistics.mean(gap) if gap else 0.0, "steps": len(ks)}

    # ---- the kernels on their own (roofline): CUDA events around each kernel's launch, same rotating inputs
    def kernel_time(fn, iters):
        for j in range(3):
            fn(j)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for j, (a, b) in enumerate(ev):
            a.record()
            fn(j)
            b.record()
        torch.cuda.synchronize()
        return statistics.mean(a.elapsed_time(b) for a, b in ev)

    n_k = max(3, min(args.steps, 50))
    lm_ms = kernel_time(lambda j: native.lm_solve(sets[j % n_sets]["prob"], sets[j % n_sets]["pose_init"], params,
                                                  want_cov=True, want_cost=True), n_k)
    amis_ms = None
    if M:
        lm0 = native.lm_solve(sets[0]["prob"], sets[0]["pose_init"], params, want_cov=True)
        amis_ms = kernel_time(lambda j: native.amis(sets[j % n_sets]["prob"], lm0["pose_opt"], lm0["pose_cov"], params, seed=j), n_k)
    t = torch.tensor([total_ms, lm_ms, amis_ms or 0.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, lm_ms, amis_ms = t.tolist()

    # ---- end to end: HOST (pinned) buffers, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        with gpu_local_cpus(local_rank, E2E_NUMA) as numa:
            host = {k: pc[k].contiguous().pin_memory() for k in ("x3d", "x2d", "w2d", "cam_mats", "pose_init")}
            host["delta"] = sets[0]["delta"].cpu().pin_memory()
        e_steps = max(3, min(args.steps, 60))
        n_lanes = E2E_LANES
        e_lanes = [torch.cuda.Stream(dev) for _ in range(n_lanes)]
        ress = [None] * n_lanes
        if kind == "lm_amis":
            # the C ABI's host-buffer entry point: chunked copy-in / LM + AMIS / copy-out pipeline on helper streams
            wss = [torch.empty(native.fused_workspace_bytes(Bg, N_PTS, params), dtype=torch.uint8, device=dev) for _ in range(n_lanes)]
            path = "epnp_lm_amis_fused_host_f32 (pinned host buffers, chunked copy / solve overlap)"

            def e2e_step(i, seed):
                k = i % n_lanes
                with torch.cuda.stream(e_lanes[k]):
                    ress[k] = native.lm_amis_fused_host(host, params, wss[k], n_chunks=E2E_CHUNKS, seed=seed + i,
                                                        obj_offset=rank * Bg, out=ress[k])
                return ress[k]
        else:
            # the call a user of the drop-in makes with host tensors: upload, solve, download
            path = ("pinned host tensors -> .to(device) -> " + ("epnp_lm_solve_f32" if kind == "lm" else "training step (drop-in classes)")
                    + " -> pinned host results")
            pins = [None] * n_lanes

            def e2e_step(i, seed):
                k = i % n_lanes
                with torch.cuda.stream(e_lanes[k]):
                    dv = {n: t.to(dev, non_blocking=True) for n, t in host.items()}
                    if kind == "lm":
                        prob = native.Problem(dv["x3d"], dv["x2d"], dv["w2d"], dv["cam_mats"], None, None, dv["delta"])
                        r = native.lm_solve(prob, dv["pose_init"], params, want_cov=True, want_cost=True)
                        r = {n: v for n, v in r.items() if v is not None}
                    else:
                        sets[0]["leaf"][0].data.copy_(dv["x3d"]); sets[0]["leaf"][1].data.copy_(dv["x2d"]); sets[0]["leaf"][2].data.copy_(dv["w2d"])
                        r = train(0)
                    if pins[k] is None:
                        pins[k] = {n: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for n, v in r.items()}
                    for n, v in r.items():
                        pins[k][n].copy_(v, non_blocking=True)
                    ress[k] = pins[k]
                return ress[k]
        for i in range(2 * n_lanes):
            res = e2e_step(i, 77)
        fence()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(e_steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in e_lanes:
            s.wait_stream(torch.cuda.current_stream(dev))
        for i in range(e_steps):
            ev[i][0].record(e_lanes[i % n_lanes])
            res = e2e_step(i, 99)
            ev[i][1].record(e_lanes[i % n_lanes])
        for s in e_lanes:
            torch.cuda.current_stream(dev).wait_stream(s)
        e1.record()
        fence()
        te = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        # per-step completion intervals (end of step i-1 -> end of step i on the host clock of the events): their spread
        # is the run-to-run stability of the pipeline
        ends = [e0.elapsed_time(b) for _, b in ev]
        gaps = sorted(b - a for a, b in zip([0.0] + ends[:-1], ends))[1:] if len(ends) > 2 else [te.item() / e_steps]
        h2d = sum(host[k].numel() * 4 for k in host)
        d2h = sum(v.numel() * v.element_size() for v in res.values() if v is not None)
        e2e = {"value": B_total * e_steps / (te.item() * 1e-3), "unit": "objects/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": e_steps, "chunks": E2E_CHUNKS if kind == "lm_amis" else None,
               "calls_in_flight": n_lanes, "host_buffers_on_gpu_numa_node": numa.applied,
               "ms_per_step": te.item() / e_steps,
               "step_interval_ms": {"min": gaps[0], "median": statistics.median(gaps), "max": gaps[-1]},
               "path": path}

    if rank == 0:
        peak, peak_src, sm_max = load_peaks()
        value = B_total * args.steps / (total_ms * 1e-3)
        dom = "amis_kernel" if M else "lm_warp_kernel"
        dom_ms = amis_ms if M else lm_ms
        per_launch_bytes = algorithmic_bytes_per_object(cfg, dom) * Bg
        achieved = per_launch_bytes / (dom_ms * 1e-3) / 1e9
        clk = (clocks or {}).get("sm_mhz") or sm_max
        stats, stats_src = kernel_stats(dom, args.config)
        issue = None
        if stats is not None:
            scale = Bg / float(stats["objects_per_launch"])
            issue_peak = 148 * 4 * clk * 1e6                      # one warp-instruction per SM sub-partition per cycle
            issue_rate = stats["warp_instr_per_launch"] * scale / (dom_ms * 1e-3)
            issue = {"bound": "warp-instruction issue / FP32 pipe (the binding resource, DESIGN.md section 4)",
                     "kernel": dom, "warp_instr_per_object": stats["warp_instr_per_launch"] / stats["objects_per_launch"],
                     "achieved_warp_instr_per_s": issue_rate, "peak_warp_instr_per_s": issue_peak, "frac": issue_rate / issue_peak,
                     "sm_mhz_used": clk, "ncu": {k: stats.get(k) for k in ("issue_active_pct", "fma_pipe_pct", "xu_pipe_pct", "duration_ms")}}
        line = {
            "metric": cfg["metric"], "value": value, "unit": "objects/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "warmup_steps_run": n_warm, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(args, cfg, world),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (stats["dram_bytes_per_launch"] * Bg / float(stats["objects_per_launch"])) if stats else None,
                         "traffic_source": stats_src, "peak_source": peak_src,
                         "bytes_per_object": algorithmic_bytes_per_object(cfg, dom), "kernel_ms": dom_ms,
                         "note": "issue / FP32-pipe bound, not HBM bound: see the issue block"},
            "kernels_ms": {"lm_warp_kernel": lm_ms, "amis_kernel": amis_ms if M else None,
                           "note": "each kernel launched alone, CUDA events on its stream, mean over the rotating input sets"},
            "in_loop": in_loop,
            "clocks": clocks, "gpu_launches": args.steps * world * launches_per_step,
            "kernel": ("lm_warp_kernel<6,staged> + amis_kernel<6>" + (", in-kernel push to the peers" if (gathering and args.gather == "push") else "")
                       if kind != "lm" else "lm_warp_kernel<6,staged>") + " (libepropnp_b200.so)",
        }
        if issue is not None:
            line["issue"] = issue
        if e2e is not None:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline and kind != "train":
            try:
                rates, cores, ckind, sample = cpu_reference_rates(cfg, 1, 0, 12.0)
                line["cpu_baseline"] = {"value": rates[0], "unit": "objects/s", "cores": cores, "kind": ckind, "sample": sample}
            except Exception as ex:                            # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "error": repr(ex)}
        if dump is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
