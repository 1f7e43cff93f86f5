#!/usr/bin/env python
"""bench.py -- agent observations per second of the step+render hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA engine through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  the reference arm: the CPU restatement (oracle/) on the box's
                                                           host cores -- the real reference cannot be built here
                                                           (Bullet 2.89 / Vulkan / EGL absent, DESIGN.md)
  python bench.py --config {2,3,4}                         headline another single-GPU BASELINE config

A "step" is one pass of the hot path over one batch.  The HEADLINE workload is BASELINE.json configs[3], Collect 1024 envs x
4 agents at 128x72 per GPU: 4096 agent views = 151 MB of RGBA8 observations per step -- the largest single-GPU config by
agent views (configs[2], ObstaclesHard 2048x1 RGB+depth, moves the same 151 MB with half the views).  The other single-GPU
configs are measured in the same run and reported under "configs" (value, e2e, roofline, cpu_baseline each); BASELINE
configs[4] (the eight Megaverse scenarios mixed, 1024 envs per GPU) is reported under "config5", under torchrun with and
without the NCCL gather of the observation tensor.  Weak scaling: the same workload on every GPU, no data-path collective.

  value  whole-job obs/s with the action masks already resident in HBM and the obs tensor left in HBM
  e2e    the same metric through the public host-buffer call (mv_set_actions + mv_step): H2D actions and D2H
         obs/rewards/dones inside the timed region

--steps K sets every timed loop to K steps.  --dump-outputs DIR writes, after the headline's timed steps, what its last step
handed the caller (see dump_outputs).  The inputs (env seeds, action stream) depend only on the arguments, so two builds can be
compared output for output.  The bench loads the native libraries already built in the tree (`python -m megaverse_b200._build`)
and writes nothing there.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the tree may be read-only; nothing is cached in it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("BOXOBAN_LEVELS", os.path.join(ROOT, "tests", "golden", "boxoban"))  # Sokoban (config 5) reads level files

W, H = 128, 72
OBS_BYTES = W * H * 4
METRIC, UNIT = "agent obs/sec (whole box)", "obs/s"
CONFIGS = {
    2: {"scenario": "TowerBuilding", "envs": 256, "agents": 1, "depth": False, "name": "TowerBuilding num_envs=256 num_agents_per_env=1 128x72 RGB"},
    3: {"scenario": "ObstaclesHard", "envs": 2048, "agents": 1, "depth": True, "name": "ObstaclesHard num_envs=2048 num_agents_per_env=1 128x72 RGB+depth"},
    4: {"scenario": "Collect", "envs": 1024, "agents": 4, "depth": False, "name": "Collect num_envs=1024 num_agents_per_env=4 128x72 RGB"},
}
HEADLINE = 4
MEGAVERSE8 = ["TowerBuilding", "ObstaclesEasy", "ObstaclesHard", "Collect", "Sokoban", "HexMemory", "HexExplore", "Rearrange"]  # megaverse_env.py:12-20
MIXED_ENVS_PER_GPU = 1024


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(cfg_id):
    """dram__bytes_read.sum + dram__bytes_write.sum of the raster kernel per launch, from the committed ncu capture of this config"""
    try:
        with open(os.path.join(ROOT, "profiles", "dram_traffic.json")) as f:
            rec = json.load(f)[str(cfg_id)]
        return float(rec["bytes_per_launch"]), rec.get("source")
    except Exception:  # noqa: BLE001
        return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region"""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:  # noqa: BLE001
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def bind_to_gpu_numa(gpu):
    """pin this process to the CPUs of the NUMA node the GPU hangs off BEFORE the engine allocates its pinned host slabs, so that the
    PCIe writes of the observation tensor land in local memory (GPUs 4-7 of an HGX box sit on node 1).  Returns a description."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(gpu).pci_bus_id if hasattr(torch.cuda.get_device_properties(gpu), "pci_bus_id") else None
        dom = torch.cuda.get_device_properties(gpu).pci_domain_id if bus is not None else None
        dev = torch.cuda.get_device_properties(gpu).pci_device_id if bus is not None else None
        if bus is None:
            return None
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as ex:  # noqa: BLE001
        return {"unavailable": str(ex)[:120]}


def action_stream(steps, n, seed):
    """the reference harness' distribution: one uniformly random action bit per agent per step (megaverse_test_app.cpp:140-147)"""
    rng = np.random.default_rng(seed)
    return (1 << rng.integers(0, 11, size=(steps, n))).astype(np.int32)


def run_cpu(cfg, threads, seconds, warmup=3, min_steps=3):
    """times the oracle (CPU restatement: step + software render of every view) on the host cores for about `seconds`; returns
    (obs/s, seconds, steps)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orc

    E, A = cfg["envs"], cfg["agents"]
    o = orc.Oracle(cfg["scenario"], E, A, W, H, threads=threads, depth=cfg["depth"])
    for e in range(E):
        o.seed_env(e, 42 + e)
    o.reset()
    acts = action_stream(64, E * A, 1)
    for t in range(warmup):
        o.step(acts[t % 64])
    n, t0 = 0, time.perf_counter()
    while n < min_steps or time.perf_counter() - t0 < seconds:
        o.step(acts[(warmup + n) % 64])
        n += 1
    dt = time.perf_counter() - t0
    o.close()
    return E * A * n / dt, dt, n


def run_reference_env_library(envs, agents, scenario, threads, seconds=4.0):
    """simulation-only rate of the REFERENCE's own env library where its build travelled with the snapshot (oracle/_ref/pyref: the
    reference's pybind module + env.cpp / agent.cpp / character controller / scenarios compiled in place on the Bullet stand-in, null
    renderer -- DESIGN.md section 6).  No rendering: the reference renders on the GPU.  Returns None when the module is not there."""
    try:
        d = os.path.join(ROOT, "oracle", "_ref", "pyref")
        if not os.path.isdir(d):
            return None
        sys.path.insert(0, d)
        import megaverse as ref_ext

        ref_ext.set_megaverse_log_level(2)
        g = ref_ext.MegaverseGym(scenario, W, H, envs, agents, threads, True, {})
        g.seed(42)
        g.reset()
        rng = np.random.default_rng(1)
        heads = rng.integers(0, [3, 3, 3, 2, 2, 3], size=(16, envs * agents, 6)).tolist()

        def one(t):
            row = heads[t % 16]
            for e in range(envs):
                for a in range(agents):
                    g.set_actions(e, a, row[e * agents + a])
            g.step()

        for t in range(3):
            one(t)
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            one(n)
            n += 1
        dt = time.perf_counter() - t0
        g.close()
        return {"value": envs * agents * n / dt, "unit": "agent steps/s (simulation only, no rendering)", "threads": threads, "steps": n,
                "note": "reference env library compiled in place on the Bullet stand-in (analytic narrow phase), driven through its own pybind module"}
    except Exception as ex:  # never let the context figure break the bench line
        return {"unavailable": str(ex)[:200]}


class Harness:
    """timing primitives shared by every measured config (CUDA events on the engine stream, max over ranks)"""

    def __init__(self, torch, dist, world, local_rank):
        self.torch, self.dist, self.world, self.local_rank = torch, dist, world, local_rank
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ms(self, ms):
        from megaverse_b200 import sharding

        _, ms, _ = sharding.aggregate_throughput(1, ms, self.dist if self.world > 1 else None)
        return ms

    def timed(self, stream, fn, steps, base):
        """K steps back to back (steady-state rollout, L2 warm)"""
        torch = self.torch
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record(stream)
        for t in range(steps):
            fn(base + t)
        ev1.record(stream)
        self.barrier()
        return self.max_ms(ev0.elapsed_time(ev1))

    def timed_flushed(self, stream, sync, fn, steps, base):
        """K steps, each preceded by an (untimed) L2 flush; per-step CUDA events on the engine stream, summed; max over ranks"""
        torch = self.torch
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        for t in range(steps):
            with torch.cuda.stream(stream):
                self.flush.zero_()
            evs[t][0].record(stream)
            fn(base + t)
            evs[t][1].record(stream)
        sync()
        self.barrier()
        return self.max_ms(float(sum(a.elapsed_time(b) for a, b in evs)))

    def timed_host_flushed(self, stream, fn, steps, base):
        """the host-buffer call blocks until the results are in host memory: wall clock around each call, L2 flushed (and the
        flush waited for) before it"""
        torch = self.torch
        total = 0.0
        self.barrier()
        for t in range(steps):
            with torch.cuda.stream(stream):
                self.flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(base + t)
            total += time.perf_counter() - t0
        self.barrier()
        return self.max_ms(total * 1e3)


DUMP_VIEWS = 256  # 256 views of RGBA as float32 are 38 MB: the dump stays under 64 MB with depth (9 MB) as well


def dump_outputs(eng, out_dir, depth):
    """what the device-resident step hands its caller, after its last step, as float32 / float64 .npy files: the rewards of every
    agent, the done flags of every env, and the RGBA (and depth) frames of a fixed, seeded sample of views (obs_views: their indices)
    -- the whole obs tensor would take four times its 151 MB as float32"""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    views = np.sort(np.random.default_rng(0).choice(eng.N, min(eng.N, DUMP_VIEWS), replace=False))
    idx = torch.from_numpy(views).cuda()

    def dev(what):
        return torch.as_tensor(eng.device_array(what), device="cuda")

    out = {"rewards": dev("rewards").float(), "dones": dev("dones").float(), "obs": dev("obs")[idx].float(), "obs_views": views.astype(np.float64)}
    if depth:
        out["depth"] = dev("depth")[idx].float()
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy() if torch.is_tensor(a) else a)


def measure_config(hz, cfg_id, K, Wm, rank, cores, sample_clocks=False, dump_dir=None):
    """one BASELINE single-GPU config on this rank's GPU: device-resident value, e2e through host buffers, roofline of the raster kernel"""
    from megaverse_b200 import capi, sharding

    torch, world, local_rank = hz.torch, hz.world, hz.local_rank
    cfg = CONFIGS[cfg_id]
    E, A, depth = cfg["envs"], cfg["agents"], cfg["depth"]
    N = E * A
    obs_bytes = N * OBS_BYTES * (2 if depth else 1)
    eng = capi.Engine(cfg["scenario"], E, A, W, H, num_threads=min(16, max(1, cores // max(world, 1))), device=local_rank, depth=depth)
    begin, end = sharding.shard_range(E * world, world, rank)  # weak scaling: E envs on every rank
    for e, seed in enumerate(sharding.env_seeds(begin, end)):
        eng.seed_env(e, seed)  # global env i is seeded 42 + i (megaverse_test_app.cpp:250-254)
    eng.reset()
    stream = torch.cuda.ExternalStream(eng.stream(), device=local_rank)
    acts_host = action_stream(K + Wm + 8, N, 1 + rank)
    acts_dev = torch.from_numpy(acts_host).cuda()
    torch.cuda.synchronize()
    ptr0, step_bytes = acts_dev.data_ptr(), N * 4

    def dev_step(t):
        eng.step_device(ptr0 + (t % len(acts_host)) * step_bytes)  # asynchronous: the timed region ends with a device synchronize

    def host_step(t):
        eng.step(acts_host[t % len(acts_host)])

    # ---- device-resident value (action masks resident in HBM, obs left in HBM)
    for t in range(Wm):
        dev_step(t)
    sampler = ClockSampler(local_rank) if sample_clocks else None
    if sampler:
        sampler.start()
    l0 = eng.kernel_launches()
    ms = hz.timed_flushed(stream, eng.sync, dev_step, K, Wm)
    launches = eng.kernel_launches() - l0
    if dump_dir:
        dump_outputs(eng, dump_dir, depth)
    ms_warm = hz.timed(stream, dev_step, K, Wm)
    eng.sync()
    clocks = sampler.stop() if sampler else None

    # ---- end-to-end through host buffers
    for t in range(3):
        host_step(t)
    ms_e = hz.timed_host_flushed(stream, host_step, K, Wm)
    ms_e_warm = hz.timed(stream, host_step, K, Wm)

    # ---- roofline of the dominant kernel (rasteriser): CUDA events around the kernel on the engine stream, L2 flushed before
    peak, peak_src = measured_peaks()
    eng.set_option("overlap", 0)  # kernels back to back so that each can be timed on its own
    ras, stp = [], []
    for t in range(4 + K):  # the first 4 are not counted
        with torch.cuda.stream(stream):
            hz.flush.zero_()
        dev_step(Wm + t)
        eng.sync()
        s_ms, r_ms = eng.last_kernel_ms()
        stp.append(s_ms); ras.append(r_ms)
    ras_ms, stp_ms = float(np.mean(ras[4:])), float(np.mean(stp[4:]))
    achieved = obs_bytes / (ras_ms / 1e3) / 1e9
    traffic, traffic_src = ncu_traffic(cfg_id)
    roofline = {"bound": "hbm", "kernel": "mvr::viewKernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": obs_bytes, "kernel_ms": ras_ms, "step_kernel_ms": stp_ms,
                "note": "obs(+depth) bytes written per launch / raster kernel duration (CUDA events, L2 flushed, kernels serialised); the kernel is "
                        "issue / latency bound (geometry, coverage and shading all run from shared memory), not HBM bound: DESIGN.md"}
    faults = eng.faults()
    rcfg = eng.raster_config()
    eng.close()
    return {"workload": cfg["name"] + " per GPU, random one-bit actions, resets included",
            "value": N * world * K / (ms / 1e3), "ms_per_step": ms / K, "value_l2_warm": N * world * K / (ms_warm / 1e3), "ms_per_step_l2_warm": ms_warm / K,
            "e2e": {"value": N * world * K / (ms_e / 1e3), "unit": UNIT, "h2d_bytes_per_step": N * 4, "d2h_bytes_per_step": obs_bytes + N * 8 + E, "steps": K,
                    "ms_per_step": ms_e / K, "value_l2_warm": N * world * K / (ms_e_warm / 1e3), "d2h_gbs": obs_bytes / (ms_e / K / 1e3) / 1e9},
            "roofline": roofline, "gpu_launches": int(launches), "faults": int(faults), "clocks": clocks, "raster": rcfg, "views_per_gpu": N}


def measure_mixed(hz, K, Wm, rank, cores, gather, overlap_gather=False, grid_share=False):
    """BASELINE configs[4]: the eight Megaverse scenarios mixed, MIXED_ENVS_PER_GPU envs per GPU (global env i runs scenario i % 8, so every
    GPU holds all eight).  One engine per scenario, each on its own stream, all rasterising into slices of ONE contiguous obs tensor (no
    staging copy); with `gather` the tensor is all-gathered over NCCL after every step, ordered by events (no host synchronisation).
    `overlap_gather`: the obs tensor is double-buffered (mv_set_obs_buffer switches every step), so the gather of step t runs while step
    t+1 is stepped and drawn -- the consumer sees step t one step later, as a double-buffered sampler does."""
    from megaverse_b200 import capi, sharding

    torch, dist, world, local_rank = hz.torch, hz.dist, hz.world, hz.local_rank
    begin, end = sharding.shard_range(MIXED_ENVS_PER_GPU * world, world, rank)
    per = (end - begin) // len(MEGAVERSE8)
    n_local = per * len(MEGAVERSE8)
    gathering = gather and world > 1
    nbuf = 2 if (gathering and overlap_gather) else 1
    obs_bufs = [torch.empty((n_local, H, W, 4), dtype=torch.uint8, device="cuda") for _ in range(nbuf)]
    engines, streams = [], []
    for k, scenario in enumerate(MEGAVERSE8):
        g = capi.Engine(scenario, per, 1, W, H, num_threads=max(1, min(16, cores // max(world, 1)) // 2), device=local_rank)
        g.set_obs_buffer(obs_bufs[0][k * per:(k + 1) * per].data_ptr())
        if grid_share:  # the eight engines' persistent raster grids side by side instead of queueing behind each other (measured: slower --
            # the maze scenarios then hold their eighth of the GPU long after the light ones have left theirs idle)
            g.set_option("raster_grid", max(8, g.raster_config()["grid"] // len(MEGAVERSE8)))
        for e in range(per):
            g.seed_env(e, 42 + begin + e * len(MEGAVERSE8) + k)  # global env i = begin + e*8 + k runs scenario k
        g.reset()
        engines.append(g)
        streams.append(torch.cuda.ExternalStream(g.stream(), device=local_rank))
    masks = torch.from_numpy(action_stream(64, n_local, 101 + rank)).cuda()
    gathered_bufs = [torch.empty((world * n_local, H, W, 4), dtype=torch.uint8, device="cuda") for _ in range(nbuf)] if gathering else None
    comm = torch.cuda.Stream(device=local_rank) if gathering else None
    read_done = [None] * nbuf  # per obs buffer: the gather that last read it
    torch.cuda.synchronize()

    def step(t):
        b = t % nbuf
        for k, g in enumerate(engines):
            if nbuf > 1:
                g.set_obs_buffer(obs_bufs[b][k * per:(k + 1) * per].data_ptr())
            if read_done[b] is not None:  # this step overwrites the send buffer of an earlier gather: wait for it, on the device
                streams[k].wait_event(read_done[b])
            g.step_device(masks.data_ptr() + ((t % 64) * n_local + k * per) * 4)
        if gathering:
            for s in streams:  # the gather waits for every engine's raster kernel, on the device
                comm.wait_event(s.record_event())
            with torch.cuda.stream(comm):
                dist.all_gather_into_tensor(gathered_bufs[b].view(-1), obs_bufs[b].view(-1))
            read_done[b] = comm.record_event()

    def sync():
        for g in engines:
            g.sync()
        torch.cuda.synchronize()

    for t in range(max(Wm, 4)):
        step(t)
    sync()
    hz.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    main = torch.cuda.current_stream()
    for s in streams:
        main.wait_event(s.record_event())
    ev0.record(main)
    for s in streams:
        s.wait_event(ev0)
    t0 = max(Wm, 4)
    for t in range(K):
        step(t0 + t)
    for s in streams + ([comm] if comm is not None else []):
        main.wait_event(s.record_event())
    ev1.record(main)
    sync()
    hz.barrier()
    ms = hz.max_ms(ev0.elapsed_time(ev1))
    faults = sum(g.faults() for g in engines)
    if gathering:  # the gathered tensor holds every rank's frames: block r equals what rank r rendered (checksums exchanged)
        last = (t0 + K - 1) % nbuf
        obs, gathered = obs_bufs[last], gathered_bufs[last]

        def checksum(t):
            v = t.reshape(-1).view(torch.int32).to(torch.int64)
            return torch.stack([v.sum(), (v * torch.arange(1, v.numel() + 1, device=v.device, dtype=torch.int64) % 1000003).sum()])

        mine = checksum(obs)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        ok = bool(torch.equal(gathered[rank * n_local:(rank + 1) * n_local], obs)) and all(
            bool(torch.equal(checksum(gathered[r * n_local:(r + 1) * n_local]), every[r])) for r in range(world))
    else:
        ok = None
    for g in engines:
        g.close()
    out = {"value": n_local * world * K / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / K, "envs_per_gpu": n_local, "faults": int(faults), "steps": K,
           "raster_grid_per_engine": "1/8 of the GPU's CTA slots (option raster_grid)" if grid_share else "all (the engines' grids queue behind each other)"}
    if gathering:
        recv = (world - 1) * n_local * OBS_BYTES  # bytes arriving at each GPU per step
        out.update({"gathered_bytes_per_step_per_gpu": recv, "nvlink_rx_gbs_per_gpu": recv / (ms / K / 1e3) / 1e9, "gathered_blocks_match_their_ranks": ok,
                    "obs_tensor": "double-buffered: the gather of step t runs under step t+1" if nbuf > 1 else "single: step t+1 waits for the gather of step t"})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=HEADLINE, choices=sorted(CONFIGS), help="BASELINE config to headline (default: the largest)")
    ap.add_argument("--only-headline", action="store_true", help="skip the other configs' sub-records")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline's outputs of its last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    rank, local_rank, world = dist_env()
    K, Wm = args.steps, max(args.warmup, 3)
    cores = os.cpu_count() or 1
    head = CONFIGS[args.config]
    config = {"workload": head["name"] + " per GPU (BASELINE.json configs[%d]), random one-bit actions, resets included" % (args.config - 1),
              "envs_per_gpu": head["envs"], "agents_per_env": head["agents"], "resolution": [W, H], "depth": head["depth"],
              "parallelism": "env-sharded x%d (no data-path collective)" % max(world, 1),
              "l2_policy": "L2 flushed (256 MB written) before EVERY timed step, untimed: each step is timed on its own with CUDA events on the "
                           "engine stream and the K step times are summed; value_l2_warm / e2e value_l2_warm are the same loops run back to back"}

    if args.impl == "reference":
        # the reference's own CPU path cannot be built here; the port (oracle) stands in.  Rank 0 only.
        if rank != 0:
            return
        v, dt, n = run_cpu(head, cores, seconds=max(6.0, min(60.0, 0.05 * K)), warmup=min(Wm, 3), min_steps=min(K, 50))
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": n, "warmup": min(Wm, 3),
                "ms_per_step": dt / n * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": "%d envs x %d agents x %d steps (step + software render of every view), all %d host threads, %.1f s" % (head["envs"], head["agents"], n, cores, dt)},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa(local_rank)  # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    hz = Harness(torch, dist, world, local_rank)

    main_rec = measure_config(hz, args.config, K, Wm, rank, cores, sample_clocks=True, dump_dir=args.dump_outputs if rank == 0 else None)
    others = {}
    if world == 1 and not args.only_headline:
        for cid in sorted(CONFIGS):
            if cid != args.config:
                others[str(cid)] = measure_config(hz, cid, K, Wm, rank, cores)
    config5 = None
    if not args.only_headline:
        config5 = {"workload": "Megaverse-8 mixed scenarios (%s), %d envs x 1 agent per GPU, 128x72 RGB (BASELINE.json configs[4])" % (", ".join(MEGAVERSE8), MIXED_ENVS_PER_GPU),
                   "no_gather": measure_mixed(hz, K, Wm, rank, cores, gather=False)}
        if world == 1:
            config5["no_gather_grid_shares"] = measure_mixed(hz, K, Wm, rank, cores, gather=False, grid_share=True)
        if world > 1:
            config5["nccl_all_gather"] = measure_mixed(hz, K, Wm, rank, cores, gather=True)
            config5["nccl_all_gather_overlapped"] = measure_mixed(hz, K, Wm, rank, cores, gather=True, overlap_gather=True)

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt, n = run_cpu(head, cores, seconds=12.0)
        main_rec["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "%d envs x %d agents x %d steps of the same workload (step + software render) on all %d host threads (%.1f s)" % (head["envs"], head["agents"], n, cores, dt),
                                    "reference_env_library": run_reference_env_library(head["envs"], head["agents"], head["scenario"], min(cores, 16))}
        for cid, rec in others.items():
            c = CONFIGS[int(cid)]
            v, dt, n = run_cpu(c, cores, seconds=4.0)
            rec["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": "%d envs x %d agents x %d steps on all host threads (%.1f s)" % (c["envs"], c["agents"], n, dt)}

    if rank == 0:
        line = {"metric": METRIC, "value": main_rec["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": main_rec["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "roofline": main_rec["roofline"], "cpu_baseline": main_rec.get("cpu_baseline"),
                "value_l2_warm": main_rec["value_l2_warm"], "ms_per_step_l2_warm": main_rec["ms_per_step_l2_warm"],
                "e2e": main_rec["e2e"], "clocks": main_rec["clocks"], "gpu_launches": main_rec["gpu_launches"], "faults": main_rec["faults"],
                "raster": main_rec["raster"], "numa": numa, "configs": others, "config5": config5}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
