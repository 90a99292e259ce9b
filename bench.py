#!/usr/bin/env python
"""bench.py -- scans/sec of the PFSlam2D hot path at 256 particles x 1080 beams (BASELINE.json metric).

A "step" is one PFSlam2D::update() of one synthetic 1080-beam scan (predict -> scan matching of every particle ->
normalise / resample -> ray-cast + distance-map update of every particle).  Synthetic data, fp64 arithmetic over
packed u32 map cells.  N GPUs: particles shard over ranks (the SAME 256-particle filter is split, so `scaling` is "strong"); a multi-GPU line also carries
`weak_scaling`: the same scans with 256 particles PER GPU (P = 256 x N), which is what the partitioning is for (skip with --no-weak).

  python bench.py --gpus 1 --steps K --warmup W            # this framework
  python bench.py --impl reference --steps K --warmup W    # the CPU restatement of the reference on the host cores

What the line reports (N = 1):
  value          K timed scans of the revisit regime (the filter has seen `prebuild` scans), scans staged in HBM; every step has its
                 own CUDA event pair on the launching stream: value = K / (sum of the steps), plus median / p99 / max per step
  e2e            the same K scans through lama_pf_update with HOST buffers, timed with the host clock around the K calls
  regimes        explore (scans 6-45 of a fresh map), revisit (= value), resample_forced (measurement gain lowered until the filter
                 resamples every few dozen scans: copy-on-write detaches inside the window), full_loop (all 5 000 scans of
                 BASELINE config 4's loop, every step timed) -- each with its own CPU-arm figure where that is affordable
  parity_checked after the timed passes the GPU filter and the CPU arm (same scans, same options) are compared: particle states
                 <= 1e-9, weights, resampling history (count + hash), work counters, every cell of three particles
  cpu_baseline   the oracle's thread pool on this host's cores: logical CPUs, affinity and cgroup quota are printed; the thread count is
                 chosen on steady-state scans; both the best and the all-cores figure are given

--dump-outputs DIR writes, after all timed passes, what the `value` pass's filter holds after its last timed step (see dump_outputs) as
DIR/<name>.npy.  Scans and seeds are fixed, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PARTICLES = 256
BEAMS = 1080
WORLD = "loop"   # 30 m x 30 m room with four pillars, rounded-square loop (BASELINE.json configs[3] world family)
METRIC = "scans/sec at 256 particles x 1080 beams"
WORKLOAD = f"PFSlam2D {PARTICLES} particles x {BEAMS} beams, 0.05 m grid, l2_max 0.5, GN+Cauchy(0.15), synthetic 30 m loop room"
FORCED_GAIN = 0.0008   # meas_sigma_gain of the `resample_forced` regime (default 3: the filter never resamples on this world)
DUMP_MAP_PARTICLES = 4       # particles whose maps --dump-outputs writes, drawn with a fixed seed from rank 0's shard
DUMP_BUDGET = 64 << 20       # bytes --dump-outputs may write in all


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)["hbm_gbs"], "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe), sampled every 20 ms.  Started BEFORE the
    barrier that opens the timed region: nothing is spawned between the barrier and the first event."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.t_open = self.t_close = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            t0 = time.perf_counter()
            while not self.rows and time.perf_counter() - t0 < 3.0:   # first sample in hand before the timed region opens
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def window(self, t_open, t_close):
        self.t_open, self.t_close = t_open, t_close

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, sm_all, mx, reasons = [], [], None, set()
        for ts, r in self.rows:
            try:
                inside = self.t_open is None or (self.t_open - 0.02 <= ts <= self.t_close + 0.02)
                sm_all.append(float(r[0])); mx = float(r[1])
                if inside:
                    sm.append(float(r[0]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            except Exception:
                pass
        use = sm if sm else sm_all
        return {"sm_mhz": float(np.median(use)) if use else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "samples_total": len(sm_all)}


def make_data(n_scans):
    from iris_lama_b200 import synth
    return synth.make_dataset(WORLD, n_scans, n_beams=BEAMS)


def pf_options_kwargs(**over):
    # reference defaults (pf_slam2d.h:132-185) except the gates so that every scan updates, and a fixed seed
    kw = dict(trans_thresh=0.05, rot_thresh=0.05, seed=42)
    kw.update(over)
    return kw


def host_facts():
    """What this host gives the CPU arm.  The 1-GPU lease of this pool shows 128 logical CPUs but runs under a cgroup quota of 16
    (cpu.max = 1600000 100000), the 8-GPU node has all 128: the same code reads 24 scans/s on one and 82 on the other."""
    f = {"logical_cpus": os.cpu_count(), "affinity": len(os.sched_getaffinity(0)), "cgroup_quota_cpus": None}
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        f["cgroup_quota_cpus"] = None if q == "max" else int(q) / int(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            f["cgroup_quota_cpus"] = None if q <= 0 else q / per
        except Exception:
            pass
    usable = f["affinity"]
    if f["cgroup_quota_cpus"]:
        usable = max(1, min(usable, int(round(f["cgroup_quota_cpus"]))))
    f["usable_cpus"] = usable
    return f


def fnv_history():
    """the same digest as lama_pf_get_resample_digest: FNV-1a over (accepted-scan number, indices) of every resampling"""
    state = {"n": 0, "h": 1469598103934665603}

    def mix(v):
        h = state["h"]
        for k in range(8):
            h ^= (v >> (8 * k)) & 0xFF
            h = (h * 1099511628211) & 0xFFFFFFFFFFFFFFFF
        state["h"] = h

    def note(scan_no, idx):
        state["n"] += 1
        mix(scan_no)
        for i in idx:
            mix(int(i) & 0xFFFFFFFF)
    return state, note


# --------------------------------------------------------------------------------------------------------
# CPU arm: the oracle restatement of the reference's thread-pool path (the reference cannot be built: no Eigen)
# --------------------------------------------------------------------------------------------------------
class CpuArm:
    def __init__(self, ds, facts, **opts):
        from oracle import pyoracle as po
        self.po, self.ds, self.facts = po, ds, facts
        self.o = po.PFSlam2D(po.PFOptions.defaults(PARTICLES, threads=facts["usable_cpus"], **pf_options_kwargs(**opts)))
        self.o.set_prior(*ds.truth[0])
        self.t = 0
        self.accepted = 0
        self.hist, self._note = fnv_history()

    def step(self):
        did = self.o.update(self.ds.scans[self.t], self.ds.odom[self.t])
        if did and self.t > 0:
            self.accepted += 1
            idx = self.o.last_resample()
            if len(idx):
                self._note(self.accepted, idx)
        self.t += 1
        return did

    def run_to(self, t_end):
        while self.t < t_end:
            self.step()

    def timed(self, n):
        t0 = time.perf_counter()
        k = 0
        for _ in range(n):
            k += int(self.step())
        dt = time.perf_counter() - t0
        return k / dt, dt

    def pick_threads(self, probe=6):
        """thread count chosen on steady-state scans (the regime of the timed window): usable CPUs (affinity capped by the cgroup quota), half
        and twice that, and every logical CPU ("all cores")"""
        f = self.facts
        cands = sorted({max(2, f["usable_cpus"] // 2), f["usable_cpus"], min(f["affinity"], 2 * f["usable_cpus"]), f["affinity"]})
        res = {}
        for th in cands:
            self.o.set_threads(th)
            res[th] = self.timed(probe)[0]
        best = max(res, key=res.get)
        self.o.set_threads(best)
        return best, res


def cpu_measure(ds, facts, first, steps, end, **opts):
    """runs the CPU arm over scans [0, end): untimed up to `first` (thread probe on the last scans before it), `steps` timed scans from
    `first`, untimed to `end`.  Returns (arm, info)."""
    arm = CpuArm(ds, facts, **opts)
    probe = 6
    n_cand = 4
    arm.run_to(max(1, first - probe * n_cand))
    best, probes = arm.pick_threads(probe) if first - arm.t >= probe * n_cand else (facts["usable_cpus"], {})
    arm.run_to(first)
    buckets0 = arm.o.times()
    val, dt = arm.timed(steps)
    buckets1 = arm.o.times()
    arm.run_to(end)
    info = {"value": val, "unit": "scans/s", "cores": best, "kind": "port",
            "threads_probed_scans_per_s": {str(k): round(v, 2) for k, v in probes.items()},
            "all_cores_scans_per_s": round(probes.get(facts["affinity"], float("nan")), 2) if probes else None,
            "host": facts,
            "summary_ms_per_scan": {k: 1000.0 * (buckets1[k] - buckets0[k]) / max(steps, 1) for k in buckets1},
            "sample": f"{steps} scans from scan {first} of the same workload (same scans as the GPU's timed region), oracle restatement of the reference "
                      f"(it needs Eigen, absent), g++ -O3 -march=x86-64-v3, thread pool of {best} = best of {sorted(probes)} on steady-state scans"}
    return arm, info


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup, pre = args.steps, args.warmup, args.prebuild
    ds = make_data(max(8, 1 + pre + warmup + steps))
    facts = host_facts()
    first = 1 + pre + warmup
    _, info = cpu_measure(ds, facts, first, steps, first + steps)
    val = info["value"]
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "scans/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": 1000.0 / val if val else None, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": WORKLOAD, "particles": PARTICLES, "beams": BEAMS, "prebuild_scans": pre},
            "cpu_baseline": info,
            "e2e": {"value": val, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------
def step_stats(ms):
    a = np.asarray(ms, float)
    return {"median_ms": float(np.median(a)), "mean_ms": float(a.mean()), "p99_ms": float(np.percentile(a, 99)), "max_ms": float(a.max()),
            "min_ms": float(a.min())}


def gpu_arm(args):
    import torch
    from iris_lama_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if api.device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: the lama_b200 hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        from iris_lama_b200.distributed import ShardedPFSlam2D
        dist.init_process_group("nccl", device_id=dev)   # the bench's own plumbing: barriers, max over ranks, handing out the NCCL id

    steps, warmup, pre = args.steps, args.warmup, args.prebuild
    # scan 0 initialises the maps, scans 1 .. pre build them (untimed), then W warm-up and K timed scans; every pass replays the SAME scans
    first = 1 + pre + warmup
    n_scans = max(8, first + steps)
    ds = make_data(n_scans)
    stream = torch.cuda.Stream(device=dev)   # the engine launches on this stream, so torch CUDA events see its kernels

    def new_pf(timing=False, particles=PARTICLES, **opts):
        o = api.PFSlam2D.Options(particles, device=local_rank, timing=int(timing), shard_rank=rank, shard_count=world,
                                 stream=stream.cuda_stream, **pf_options_kwargs(**opts))
        pf = api.PFSlam2D(o)
        pf.setPrior(*ds.truth[0])
        return pf

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_pass(data, t_first, k_steps, staged, timing=False, sample_clocks=False, particles=PARTICLES, **opts):
        """one fresh filter over scans 0 .. t_first + k_steps of `data`; the last k_steps are timed, each with its own event pair"""
        pf = new_pf(timing, particles, **opts)
        sh = None
        if world > 1 and args.sharded_impl == "python":
            sh = ShardedPFSlam2D(pf, particles, device=dev)   # round-1 orchestration: torch.distributed collectives driven from Python
        elif world > 1:
            import torch.distributed as dist                   # the sharded step inside the library (NCCL from C++, shard_comm.cpp)
            box = [api.shard_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            pf.shardConnect(box[0])
        if staged and sh is None:
            pf.stageScans(data.scans[:t_first + k_steps])
            step = lambda t: pf.updateStaged(t, data.odom[t])
        elif sh is not None:
            step = lambda t: sh.update(data.scans[t], data.odom[t])
        else:
            step = lambda t: pf.update(data.scans[t], data.odom[t])   # the public call with HOST buffers
        for t in range(t_first):
            step(t)
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()            # before the barrier: nothing is spawned inside the timed region
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(k_steps + 1)]
        barrier()
        pf.traffic(reset=True)
        _, tot0 = pf.counters()
        sum0 = pf.summary()
        ms0, _ = pf.kernelTimes()
        w0 = time.perf_counter()
        ev[0].record(stream)
        n_upd = 0
        for i in range(k_steps):
            n_upd += int(step(t_first + i))
            ev[i + 1].record(stream)
        torch.cuda.synchronize()
        w1 = time.perf_counter()
        barrier()
        if sampler:
            sampler.window(w0, w1)
        per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(k_steps)]
        dt = max_over_ranks(sum(per_step) * 1e-3)          # device timeline of the launching stream, max over ranks
        wall = max_over_ranks(w1 - w0)
        _, tot1 = pf.counters()
        sum1 = pf.summary()
        ms1, ln = pf.kernelTimes()
        h2d, d2h = pf.traffic()
        return dict(dt=dt, wall=wall, pf=pf, clocks=sampler.stop() if sampler else None, n_upd=n_upd, per_step=per_step,
                    work={k: tot1[k] - tot0[k] for k in tot1}, summary={k: (sum1[k] - sum0[k]) / k_steps for k in sum1},
                    kernel_ms={k: (ms1[k] - ms0[k]) / k_steps for k in ms1}, launches=ln, h2d=h2d, d2h=d2h)

    # ---- pass 1: `value` -- scans resident in HBM (single GPU: staged scans; sharded: host scans, see config) ----
    r1 = timed_pass(ds, first, steps, staged=True, sample_clocks=(rank == 0))
    dt_value, clocks, n_upd = r1["dt"], r1["clocks"], r1["n_upd"]
    gpu_launches = int(sum(r1["launches"].values()))
    work, stats_value, summary_value = r1["work"], step_stats(r1["per_step"]), r1["summary"]
    pf_value = r1["pf"]
    wall_value = r1["wall"]

    # ---- pass 2: `e2e` -- same metric, same scans, through the public API with host buffers, host clock -----------------------
    r2 = timed_pass(ds, first, steps, staged=False)
    e2e_val = steps / r2["wall"]
    h2d, d2h = r2["h2d"], r2["d2h"]
    stats_e2e = step_stats(r2["per_step"])
    del r2

    # ---- weak scaling (N > 1): the filter grows with the node, 256 particles per GPU stay; same scans, same public call ------------
    weak = None
    if world > 1 and not args.no_weak:
        rw = timed_pass(ds, first, steps, staged=False, particles=PARTICLES * world)
        weak = {"particles": PARTICLES * world, "particles_per_gpu": PARTICLES, "scans_per_s": steps / rw["dt"], "e2e_scans_per_s": steps / rw["wall"],
                "particle_scans_per_s": PARTICLES * world * steps / rw["dt"], "resamples": rw["work"]["resampled"], **step_stats(rw["per_step"]),
                "note": "P = 256 x N: per-GPU work fixed; efficiency = scans_per_s here / the N = 1 line's value (256 particles on one GPU)"}
        del rw

    # ---- N > 1: a window with resampling scans, i.e. with map migration between ranks (the measurement gain is lowered like in the N = 1 regime) --------
    shard_resample = None
    if world > 1 and not args.no_weak and args.sharded_impl == "native":
        kf, pf_first = 80, 60
        rs = timed_pass(ds, pf_first, kf, staged=False, meas_sigma_gain=FORCED_GAIN)
        st = rs["pf"].shardStats()
        shard_resample = {"scans_per_s": kf / rs["dt"], "first_scan": pf_first, "steps": kf, **step_stats(rs["per_step"]), "meas_sigma_gain": FORCED_GAIN,
                          "resamples": rs["work"]["resampled"], "shard_stats_rank0": st}
        del rs

    # ---- pass 3: per-kernel CUDA-event durations for the roofline (timing mode adds event records and host syncs) ------------
    roofline, kernel_ms = None, None
    if world == 1 or args.sharded_impl == "native":
        # N > 1: the sharded step records its kernel events without host synchronisation (Engine::step_enqueue); the figures are RANK 0's shard
        r3 = timed_pass(ds, first, steps, staged=(world == 1), timing=True)
        d, tm = r3["work"], r3["kernel_ms"]
        peak, peak_kind = load_peaks()
        # algorithmic bytes (SURVEY 8(d)): match E*N*(4 cells x 2 B); ray C*(4 B read + 4 B write); brushfire W*(5x8 B read + 4x8 B write);
        # copy D * 2 * 1024 * 12 B.  On a sharded handle the evaluations are counted over all ranks (they travel with the all-gather), cells and pops locally.
        by = {"k_match": d["evals"] / world * BEAMS * 8.0 / steps, "k_raycast": d["ray_cells"] * 8.0 / steps, "k_brushfire": d["dm_pops"] * 72.0 / steps}
        t = {"k_match": tm["match_ms"], "k_raycast": tm["raycast_ms"], "k_brushfire": tm["brushfire_ms"]}
        kernel_ms = dict(t)
        kernel_ms["map_device"] = tm["raycast_ms"] + tm["brushfire_ms"]
        dom = max(t, key=t.get)
        ach = by[dom] / (t[dom] * 1e-3) / 1e9 if t[dom] > 0 else 0.0
        traffic, traffic_src = None, None   # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of that kernel (per launch)
        for name in sorted(os.listdir(os.path.join(ROOT, "profiles")), reverse=True):
            if world == 1 and name.endswith("ncu_traffic.json"):
                with open(os.path.join(ROOT, "profiles", name)) as f:
                    tj = json.load(f)
                if dom in tj:
                    traffic, traffic_src = tj[dom].get("dram_bytes_per_launch"), name + (" @ " + tj["commit"] if "commit" in tj else "")
                    break
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                    "traffic_source": traffic_src, "peak_kind": peak_kind, "algorithmic_bytes_per_launch": by[dom], "avg_launch_ms": t[dom],
                    "all_kernels": {kk: {"GBps": (by[kk] / (t[kk] * 1e-3) / 1e9 if t[kk] > 0 else 0.0), "ms_per_step": t[kk], "bytes_per_step": by[kk],
                                         "frac": (by[kk] / (t[kk] * 1e-3) / 1e9 / peak if t[kk] > 0 else 0.0)} for kk in t},
                    "bytes_copy_per_step": d["detached"] * 2 * 1024 * 12.0 / steps}
        if world > 1:
            roofline["scope"] = "rank 0's shard: %d of %d particles (no ncu capture of a sharded run: traffic null)" % (PARTICLES // world, PARTICLES)
        del r3

    # ---- CPU baseline + parity (rank 0, N = 1 only): the same scans on the host cores, then GPU vs CPU state --------------------
    cpu, parity = None, None
    facts = host_facts()
    if world == 1 and not args.no_cpu:
        cpu_steps = max(1, min(steps, args.cpu_steps))   # never past scan first + steps: the dataset ends there
        arm, cpu = cpu_measure(ds, facts, first, cpu_steps, first + steps)
        parity = compare(pf_value, arm)
        del arm

    # ---- the other regimes of BASELINE config 4 (N = 1) --------------------------------------------------------------------------
    regimes = None
    if world == 1 and not args.no_regimes:
        regimes = {"revisit": {"scans_per_s": steps / dt_value, "first_scan": first, "steps": steps, **stats_value, "resamples": work["resampled"],
                               "cpu_scans_per_s": cpu["value"] if cpu else None}}
        ke = 40
        re_ = timed_pass(ds, 6, ke, staged=True)
        regimes["explore"] = {"scans_per_s": ke / re_["dt"], "first_scan": 6, "steps": ke, **step_stats(re_["per_step"]),
                              "dm_pops_per_scan": re_["work"]["dm_pops"] / ke}
        del re_
        kf, pf_first = 80, 60
        rf = timed_pass(ds, pf_first, kf, staged=True, meas_sigma_gain=FORCED_GAIN)
        regimes["resample_forced"] = {"scans_per_s": kf / rf["dt"], "first_scan": pf_first, "steps": kf, **step_stats(rf["per_step"]),
                                      "meas_sigma_gain": FORCED_GAIN, "resamples": rf["work"]["resampled"], "patches_detached_per_scan": rf["work"]["detached"] / kf,
                                      "bytes_copy_per_scan": rf["work"]["detached"] * 2 * 1024 * 12.0 / kf}
        pf_forced = rf["pf"]
        del rf
        if not args.no_cpu:
            t0 = time.perf_counter()
            armf, cf = cpu_measure(ds, facts, pf_first, kf, pf_first + kf, meas_sigma_gain=FORCED_GAIN)
            regimes["explore"]["cpu_note"] = "exploration scans are part of the CPU arm's run-in; its rate there is in cpu_baseline.threads_probed"
            regimes["resample_forced"]["cpu_scans_per_s"] = cf["value"]
            regimes["resample_forced"]["parity_checked"] = compare(pf_forced, armf)["ok"]
            regimes["resample_forced"]["cpu_seconds"] = time.perf_counter() - t0
            del armf
        del pf_forced
        if not args.no_full_loop:
            nfull = args.full_loop
            dsf = make_data(nfull)
            rl = timed_pass(dsf, 1, nfull - 1, staged=True)
            ps = np.asarray(rl["per_step"])
            regimes["full_loop"] = {"scans": nfull - 1, "scans_per_s": (nfull - 1) / rl["dt"], **step_stats(ps), "resamples": rl["work"]["resampled"],
                                    "explore_share_of_time_first_100": float(ps[:100].sum() / ps.sum()),
                                    "dm_pops_per_scan": rl["work"]["dm_pops"] / (nfull - 1), "ray_cells_per_scan": rl["work"]["ray_cells"] / (nfull - 1)}
            del rl, dsf

    if rank == 0:
        value = steps / dt_value
        line = {"metric": METRIC, "value": value, "unit": "scans/s", "n_gpus": world, "steps": steps, "warmup": warmup,
                "ms_per_step": 1000.0 * dt_value / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "particles": PARTICLES, "beams": BEAMS, "prebuild_scans": pre,
                           "parallelism": f"particles sharded over {world} GPU(s)",
                           "l2": "per-scan working set (~290 MB of touched map patches over 256 particles) exceeds the 126 MB L2; no explicit flush",
                           "value_inputs": "scans staged in HBM",
                           "sharded_step": None if world == 1 else ("inside liblama_b200.so (NCCL all-gather + send/recv from C++)" if args.sharded_impl == "native"
                                                                    else "torch.distributed collectives driven from Python"),
                           "updates_in_timed_region": n_upd,
                           "timer": "one CUDA event pair per step on the launching stream (a step enqueues match + map update at once; the event after "
                                    "it completes when that map update has); value = K / sum of the K steps; host wall clock of the same region: "
                                    "%.4f s" % wall_value},
                "step_ms": stats_value, "value_from_median": 1000.0 / stats_value["median_ms"],
                "clocks": clocks,
                "e2e": {"value": e2e_val, "unit": "scans/s", "h2d_bytes_per_step": h2d / steps, "d2h_bytes_per_step": d2h / steps,
                        "timer": "host clock around the K lama_pf_update calls with host buffers, device synchronised at both ends", "step_ms": stats_e2e},
                "gpu_launches": gpu_launches,
                "counters_per_step": {k: v / steps for k, v in work.items()},
                "summary_ms_per_step": {**summary_value, "map_device": kernel_ms["map_device"] if kernel_ms else None,
                                        "note": "reference Summary buckets (pf_slam2d.h:88-129): host wall clock of sampling / solve (enqueue + wait for the "
                                                "match) / normalise / resample; the map bucket runs asynchronously on the device"}}
        line["particle_scans_per_s"] = PARTICLES * value
        if weak:
            line["weak_scaling"] = weak
        if shard_resample:
            line["regimes"] = {"resample_forced": shard_resample}
        if roofline:
            line["roofline"] = roofline
            line["kernel_ms_per_step"] = kernel_ms
        if cpu:
            line["cpu_baseline"] = cpu
        if parity is not None:
            line["parity_checked"] = parity["ok"]
            line["parity"] = parity
        if regimes:
            line["regimes"] = regimes
        if args.dump_outputs:
            line["dump_outputs"] = {"dir": args.dump_outputs, "bytes": dump_outputs(pf_value, args.dump_outputs, PARTICLES // world)}
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def compare(pf, arm):
    """GPU filter vs CPU arm after the same scans: states, weights, resampling history, total counters, cells of three particles"""
    o = arm.o
    out = {"scans": arm.t}
    sg, wg = pf.getParticles()
    so, wo = o.particles()
    out["max_state_diff"] = float(np.abs(sg - so).max())
    out["max_weight_rel_diff"] = float(np.abs(wg - wo).max() / max(1.0, np.abs(wo).max()))
    n, h = pf.resampleDigest()
    out["resamples"] = [n, arm.hist["n"]]
    out["resample_history_equal"] = bool(n == arm.hist["n"] and h == arm.hist["h"])
    _, tg = pf.counters()
    _, to = o.counters()
    out["counters_equal"] = bool(all(tg[k] == to[k] for k in ("evals", "gn_iters", "ray_cells", "dm_pops")) or
                                 (n > 0 and all(tg[k] == to[k] for k in ("evals", "gn_iters"))))   # map work of resampling scans is booked before the copy
    cells_ok, n_cells = True, 0
    for p in (0, PARTICLES // 2 - 27, PARTICLES - 1):
        _, mn, mx = o.occ_bounds(p)
        w, hh = int(mx[0] - mn[0]), int(mx[1] - mn[1])
        a, b = pf.exportOccupancy(p, int(mn[0]), int(mn[1]), w, hh), o.export_occ(p, mn[0], mn[1], w, hh)
        cells_ok &= bool((a["occupied"] == b["occupied"]).all() and (a["visited"] == b["visited"]).all())
        _, mn, mx = o.dm_bounds(p)
        w, hh = int(mx[0] - mn[0]), int(mx[1] - mn[1])
        d1, d2 = pf.exportDistance(p, int(mn[0]), int(mn[1]), w, hh), o.export_dm(p, mn[0], mn[1], w, hh)
        cells_ok &= bool(all((d1[k] == d2[k]).all() for k in ("sqdist", "valid", "ox", "oy")))
        n_cells += w * hh
    out["cells_equal"], out["cells_compared"] = cells_ok, n_cells
    out["ok"] = bool(out["max_state_diff"] <= 1e-9 and out["max_weight_rel_diff"] <= 1e-6 and out["resample_history_equal"] and out["counters_equal"]
                     and cells_ok)
    return out


def dump_outputs(pf, out_dir, local_particles):
    """Writes what a caller of PFSlam2D receives after the last update as out_dir/<name>.npy: the pose, every particle's state and
    weights, neff, the best particle and its trajectory (float64), and the occupancy and distance maps of DUMP_MAP_PARTICLES particles
    drawn with a fixed seed from the first `local_particles` (float32, with their origin cell).  Stops adding maps at DUMP_BUDGET bytes."""
    st, w = pf.getParticles()
    best = pf.getBestParticleIdx()
    arrays = {"pose": pf.getPose(), "particle_states": st, "particle_weights": w, "neff": np.array([pf.getNeff()]),
              "best_particle": np.array([best], np.float64), "best_trajectory": pf.trajectory(best)}
    total = sum(a.nbytes for a in arrays.values())
    sample = np.random.default_rng(0).choice(local_particles, size=min(DUMP_MAP_PARTICLES, local_particles), replace=False)
    for p in sorted(int(i) for i in sample):
        maps = {}
        for kind, export, planes in ((0, pf.exportOccupancy, ("occupied", "visited")), (1, pf.exportDistance, ("sqdist", "valid", "ox", "oy"))):
            _, mn, mx = pf.mapBounds(p, kind)
            m = export(p, int(mn[0]), int(mn[1]), int(mx[0] - mn[0]), int(mx[1] - mn[1]))
            maps[f"map{p:03d}_{'occ' if kind == 0 else 'dm'}_origin"] = mn.astype(np.float64)
            maps.update({f"map{p:03d}_{k}": m[k].astype(np.float32) for k in planes})
        size = sum(a.nbytes for a in maps.values())
        if total + size > DUMP_BUDGET:
            break
        arrays.update(maps)
        total += size
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--cpu-steps", type=int, default=60)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-regimes", action="store_true")
    ap.add_argument("--no-full-loop", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling pass (P = 256 x N) of a multi-GPU run")
    ap.add_argument("--full-loop", type=int, default=5000, help="scans of the full-loop regime (BASELINE config 4: 5 000)")
    ap.add_argument("--sharded-impl", default="native", choices=["native", "python"])
    ap.add_argument("--prebuild", type=int, default=300, help="untimed scans that build the map before warm-up (both arms)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed filter's state after its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
