#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched MiniWorld step path on B200 (and the CPU arm).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json): MiniWorld-FourRooms-v0, N_envs = 4096 per GPU, 80x60 RGB + depth,
uniformly random actions, next-step auto-reset, env i seeded 1000 + i.  One "step" = one
mwb_step call: K1 (physics / reward / device resets) + K2 (render RGB + depth) for every env.

  value  : whole-job env-steps/s with actions and outputs resident in HBM (torch CUDA tensors),
           timed with CUDA events over exactly K steps, barrier + synchronize on both sides,
           max over ranks.  Multi-GPU: envs shard 4096 per rank (weak scaling); every step the
           uint8 observations are gathered to rank 0 with NCCL (inside the timed region).
  e2e    : the same K steps through the public host API (BatchedMiniWorld.step_host): actions
           from pinned host memory, observations / rewards / flags back to pinned host memory,
           copies inside the timed region.
  roofline: K2's algorithmic bytes (framebuffer written once) / its CUDA-event time inside the
           timed region, against the measured HBM copy bandwidth (MEASURED_PEAKS.json).
  cpu_baseline: the oracle port (oracle/physics_port.py + oracle/softgl.c) on host cores.

--dump-outputs DIR: after the timed steps, what the last timed step returned (obs, reward, terminated, truncated and
the info arrays, e.g. depth) is written as DIR/<name>.npy in float32 (float64 where the step returns float64), for
a fixed, seeded sample of envs that keeps the files under 64 MB (DIR/env_index.npy lists it).  Actions and seeds
depend only on the arguments, so two builds run with the same arguments can be compared output for output.

--impl reference: the reference's own Pyglet/OpenGL path cannot run here (no pyglet, GL or
gymnasium in the image; /root/reference is absent on the GPU box), so this arm times the CPU
oracle port of the same workload on all host cores, one process per core.
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

LEVEL = "MiniWorld-FourRooms-v0"
N_ENVS = 4096
W, H = 80, 60
BYTES_RGB = W * H * 3
BYTES_DEPTH = W * H * 4
FALLBACK_HBM_GBS = 6650.0
DUMP_BYTES = 60 << 20               # --dump-outputs payload limit (64 MB with headroom for the .npy headers)
# BASELINE.json configs (index as in its `configs` list); envs = per GPU under weak scaling.  Config 3 is the one the
# metric is quoted on and the default; 4 and 5 are the two configs it states for 8 GPUs (8192 / 8 and 4096 / 8 envs per GPU).
CONFIGS = {
    2: dict(level="MiniWorld-OneRoom-v0", envs=1024, w=80, h=60, depth=False, dr=False),
    3: dict(level="MiniWorld-FourRooms-v0", envs=4096, w=80, h=60, depth=True, dr=False),
    4: dict(level="MiniWorld-MazeS8-v0", envs=1024, w=80, h=60, depth=False, dr=True),
    5: dict(level="MiniWorld-PickupObjects-v0", envs=512, w=160, h=120, depth=False, dr=False),
}


def bind_to_gpu_numa(local):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned host memory is allocated
    (first-touch then places the pinned pages on that node): with 8 ranks on a two-socket box the device->host
    copies otherwise cross the socket interconnect for half of the GPUs.  Returns (node, n_cpus) or None."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node, len(cpus)
    except Exception:
        return None


def measured_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons while the timed region runs (NVML every 10 ms; nvidia-smi
    as a fallback)."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False   # rows: (sm_mhz, max_mhz, [4 flags])

    def _nvml_loop(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        masks = [nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap]
        while not self.stop_flag:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.rows.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), mx, [bool(r & m) for m in masks]))
            time.sleep(0.01)

    def _smi_loop(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6 and parts[0].isdigit():
                    self.rows.append((int(parts[0]), int(parts[1]) if parts[1].isdigit() else None,
                                      [p.lower().startswith("active") for p in parts[2:6]]))
            except Exception:
                pass
            time.sleep(0.1)

    def run(self):
        try:
            self._nvml_loop()
        except Exception:
            self._smi_loop()

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(r[0] for r in self.rows)
        reasons = [n for k, n in enumerate(self.NAMES) if any(r[2][k] for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.rows[0][1], "reasons": reasons, "samples": len(self.rows)}


# --------------------------------------------------------------------------- CPU arm

def _port_worker(args):
    """One process: the oracle port of the workload on one core; `warm_s` untimed seconds, then
    `budget_s` timed seconds.  Returns (env-steps, seconds) of the timed part."""
    rank, warm_s, budget_s, seed0, cpu = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    if cpu is not None:
        try:
            os.sched_setaffinity(0, {cpu})      # one worker per PHYSICAL core, pinned: no migration, no sibling sharing
        except OSError:
            pass
    from miniworld_b200.assets import Texture
    from miniworld_b200.envs import LEVELS
    from oracle import softgl
    from oracle.physics_port import PortEnv
    port = PortEnv(LEVELS[LEVEL](device=None))
    port.reset(seed=seed0 + rank)
    ts = softgl.TextureSet([t.texels for t in Texture.registry])
    rng = np.random.default_rng(12345 + rank)
    tex_index = lambda tex: tex.tex_id
    n, done = 0, False
    t_start = time.perf_counter()
    t0 = None
    while True:
        now = time.perf_counter()
        if t0 is None and now - t_start >= warm_s:
            t0, n = now, 0
        if t0 is not None and now - t0 >= budget_s:
            break
        if done:
            port.reset()
            done = False
        else:
            _, te, tr, _ = port.step(int(rng.integers(0, 3)))
            done = te or tr
        softgl.render(port.env, ts, tex_index, W, H, 8)     # RGB + depth in one pass
        n += 1
    return n, time.perf_counter() - t0


def physical_cores():
    """One logical CPU per physical core (the first hyper-thread sibling of each), restricted to this process's
    affinity mask."""
    allowed = sorted(os.sched_getaffinity(0))
    seen, out = set(), []
    for c in allowed:
        try:
            with open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c) as f:
                sib = f.read().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            out.append(c)
    return out


def cpu_port_throughput(cores, warm_s, budget_s):
    """cores: 1, or a list of logical CPUs to pin one worker each to."""
    if cores == 1:
        n, dt = _port_worker((0, warm_s, budget_s, 1000, None))
        return n / dt, n
    import multiprocessing as mp
    with mp.get_context("spawn").Pool(len(cores)) as pool:
        res = pool.map(_port_worker, [(r, warm_s, budget_s, 1000, c) for r, c in enumerate(cores)])
    return sum(n / dt for n, dt in res), sum(n for n, _ in res)


def reference_physics_only(seconds=4.0):
    """BASELINE.md section 4 fallback 2a, where /root/reference exists (the build container, not the GPU box): the
    UNMODIFIED reference's step() with GL stubbed out (no rendering) on one core -- an upper bound of what the
    reference's own Python can do per core.  None when the reference is absent."""
    try:
        from oracle import ref_stub
        if not ref_stub.reference_available():
            return None
        env = ref_stub.make_reference_env(LEVEL, record=False)
        env.reset(seed=1000)
        rng = np.random.default_rng(12345)
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            _, _, te, tr, _ = env.step(int(rng.integers(0, 3)))
            if te or tr:
                env.reset()
            n += 1
        return {"value": n / (time.perf_counter() - t0), "unit": "env-steps/s", "cores": 1,
                "what": "reference MiniWorldEnv.step, GL calls ignored (no frame is produced)"}
    except Exception:
        return None


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import softgl
    softgl.build()
    # one worker pinned to every PHYSICAL core: measured on the 2 x 32-core box, 64 pinned workers deliver 7.3 k
    # env-steps/s, 128 (one per hyper-thread) only 5.0 k -- the port is cache / memory bound under full load
    cpus = physical_cores()
    cores = len(cpus)
    n_phys = cores
    # the K "steps" are K equal slices of one continuous run (each slice a bounded sample of
    # the workload); W warm-up slices are discarded.  Whole arm <= ~2 minutes.
    slice_s = min(1.0, 100.0 / max(1, args.steps + args.warmup))
    warm_s, budget = slice_s * args.warmup, slice_s * args.steps
    value, vals = cpu_port_throughput(cpus, warm_s, budget)
    ref_physics = reference_physics_only()
    line = {
        "impl": "reference", "metric": "env steps/sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64+f32", "data": "synthetic",
        "config": {"workload": "%s 80x60 RGB+depth, random actions, auto-reset" % LEVEL, "n_envs": cores,
                   "note": "reference Pyglet/GL path cannot run on this box (no pyglet/GL/gymnasium, no libEGL/libGL); "
                           "CPU oracle port timed instead, one env process pinned to each physical core "
                           "(its best configuration: one per hyper-thread is slower)",
                   "per_worker": value / cores, "physical_cores": n_phys, "per_physical_core": value / n_phys,
                   "reference_python_physics_only": ref_physics},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                         "sample": "%d env-steps total in %.0f s on %d pinned processes (one env each, one per physical core), "
                                   "%.0f per core" % (vals, budget, cores, value / n_phys)},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# --------------------------------------------------------------------------- GPU arm

def dump_outputs(path, step_out):
    """Write the arrays one BatchedMiniWorld.step returned (see --dump-outputs) to path/<name>.npy."""
    import torch
    obs, reward, terminated, truncated, info = step_out
    arrays = dict(obs=obs, reward=reward, terminated=terminated, truncated=truncated, **info)
    n = obs.shape[0]
    for k, v in arrays.items():
        assert v.shape[0] == n, "%s is not per env" % k
    wide = lambda v: torch.float64 if v.dtype == torch.float64 else torch.float32
    env_bytes = sum(v[0].numel() * (8 if wide(v) == torch.float64 else 4) for v in arrays.values())
    keep = min(n, DUMP_BYTES // env_bytes)
    rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False)) if keep < n else np.arange(n)
    idx = torch.as_tensor(rows, device=obs.device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), rows.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v.index_select(0, idx).to(wide(v)).cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from miniworld_b200.batched import BatchedMiniWorld

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = None if args.no_numa else bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cfg = CONFIGS[args.config]
    LEVEL, W, H = cfg["level"], cfg["w"], cfg["h"]
    BYTES_RGB, BYTES_DEPTH = W * H * 3, (W * H * 4 if cfg["depth"] else 0)
    env_kw = dict(obs_width=W, obs_height=H, want_depth=cfg["depth"], domain_rand=cfg["dr"])
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL's own banner / debug output ("NCCL version ...") goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, args.warmup
    N = args.envs if args.envs else cfg["envs"]
    if args.scaling == "strong":                 # fixed total work: `--envs` (default the config's) is the GLOBAL count
        assert N % world == 0, "strong scaling needs envs divisible by the number of GPUs"
        N //= world
    sharded, peer = None, False
    if world > 1:
        from miniworld_b200.dist import ShardedMiniWorld
        sharded = ShardedMiniWorld(LEVEL, world * N, dist=dist, device=local, **env_kw)
        env = sharded.local
        sharded.reset(1000)
        peer = (not args.nccl_gather) and sharded.enable_peer_obs()
    else:
        env = BatchedMiniWorld(LEVEL, N, device=local, **env_kw)
        env.reset(seed=1000)
    total = Wm + K
    gen = np.random.default_rng(12345 + rank)
    acts_np = gen.integers(0, env.action_space.n, size=(total, N), dtype=np.int32)
    acts = torch.as_tensor(acts_np, device=dev)
    gather_list = None
    if world > 1 and rank == 0 and not peer:
        gather_list = [torch.empty((N, H, W, 3), dtype=torch.uint8, device=dev) for _ in range(world)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(t):
        if peer:                          # K2 writes into rank 0's HBM over NVLink; one-way completion flags, no collective
            return sharded.step_peer(acts[t])
        out = env.step(acts[t])
        if world > 1:
            dist.gather(out[0], gather_list, dst=0)
        return out

    # ---- device-resident arm
    for t in range(Wm):
        one_step(t)
    barrier()
    env.engine.profile(True)
    env.engine.profile_read()
    launches0 = env.engine.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    done0 = int(env.get_state()["episodes_done"][0])
    e0.record()
    for t in range(Wm, total):
        last = one_step(t)
    e1.record()
    barrier()
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    k1_ms, k2_ms, n1, n2 = env.engine.profile_read()
    env.engine.profile(False)
    done_steps = int(env.get_state()["episodes_done"][0]) - done0
    launches = env.engine.launch_count() - launches0
    if args.dump_outputs:                  # before the end-to-end arm below steps the same buffers again
        dump_outputs(args.dump_outputs, last)
    if world > 1:
        tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    value = world * N * K / (ms * 1e-3)

    # ---- end-to-end arm: host buffers in, host buffers out
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
    out = dict(obs=pin((N, H, W, 3), torch.uint8), depth=pin((N, H, W, 1), torch.float32) if cfg["depth"] else None,
               reward=pin((N,), torch.float64), terminated=pin((N,), torch.uint8), truncated=pin((N,), torch.uint8))
    if peer:                               # the end-to-end leg renders into this rank's own buffer again
        env._bufs["obs"] = torch.zeros((N, H, W, 3), dtype=torch.uint8, device=dev)
    acts_pin = torch.as_tensor(acts_np).pin_memory().numpy()
    for t in range(min(Wm, 3)):
        env.step_host(acts_pin[t], out)
    barrier()
    t0 = time.perf_counter()
    for t in range(Wm, total):
        env.step_host(acts_pin[t], out)      # synchronous: returns when the host buffers are filled
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    d2h_bytes = N * (BYTES_RGB + BYTES_DEPTH + 8 + 1 + 1)
    my_d2h_gbs = d2h_bytes * K / e2e_s / 1e9
    rank_d2h = [my_d2h_gbs]
    if world > 1:
        tmax = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = float(tmax.item())
        allr = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(allr, torch.tensor([my_d2h_gbs], dtype=torch.float64, device=dev))
        rank_d2h = [float(x.item()) for x in allr]
    e2e_value = world * N * K / e2e_s
    sampler.join(timeout=2)

    if rank == 0:
        peak, peak_kind = measured_hbm()
        bytes_per_launch = N * (BYTES_RGB + BYTES_DEPTH)
        k2_avg_ms = k2_ms / max(1, n2)
        achieved = bytes_per_launch / (k2_avg_ms * 1e-3) / 1e9 if n2 else None
        cpu = {"value": None, "unit": "env-steps/s", "cores": 1, "kind": "port", "sample": "skipped"}
        if world == 1 and not args.no_cpu and args.config == 3:
            from oracle import softgl
            softgl.build()
            v, n = cpu_port_throughput(1, 1.0, 12.0)
            cpu = {"value": v, "unit": "env-steps/s", "cores": 1, "kind": "port",
                   "sample": "%d env-steps of 1 env in 12 s (oracle/physics_port.py + oracle/softgl.c)" % n}
        traffic, traffic_src = None, None
        try:   # DRAM bytes of one K2 launch: from the committed `ncu --set full` capture of THIS build and config
            with open(os.path.join(ROOT, "profiles", "k2_traffic.json")) as f:
                tj = json.load(f)
            if N == tj.get("n_envs") and args.config == tj.get("config", 3):
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                traffic_src = tj.get("source")
        except Exception:
            pass
        line = {
            "metric": "env steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64+f32", "data": "synthetic",
            "config": {"workload": "BASELINE.json configs[%d]: %s N_envs=%d per GPU, %dx%d RGB%s, 8x MSAA%s, random actions, "
                                   "next-step auto-reset on device" % (args.config, LEVEL, N, W, H, "+depth" if cfg["depth"] else "",
                                                                       ", domain_rand" if cfg["dr"] else ""),
                       "global_envs": world * N, "partition": "%d GPUs x %d envs (%s scaling)" % (world, N, args.scaling),
                       "obs_gather": ("none" if world == 1 else "K2 stores its frames straight into rank 0's buffer (CUDA IPC peer memory "
                                      "over NVLink), double-buffered, one-way stream-ordered completion flags (no per-step collective)" if peer else
                                      "NCCL gather of uint8 obs to rank 0"),
                       "numa": "rank 0 bound to NUMA node %d (%d CPUs)" % numa if numa else "not bound",
                       "l2": "per-step outputs %.1f MB > 126 MB L2; no explicit flush" % (bytes_per_launch / 1e6),
                       "episodes_finished_in_timed_region": done_steps},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if achieved else None, "traffic": traffic,
                         "kernel": "render_kernel<8>", "kernel_avg_ms": k2_avg_ms, "peak_kind": peak_kind,
                         "algorithmic_bytes_per_launch": bytes_per_launch,
                         "k1_avg_ms": k1_ms / max(1, n1), "kernel_share_of_step": k2_ms / ms if ms else None,
                         "non_kernel_ms_per_step": (ms - k1_ms - k2_ms) / K if ms else None,
                         "traffic_source": traffic_src},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": N * 4,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_s * 1e3 / K,
                    "scope": "per rank: every rank copies its own envs' outputs to its own pinned host buffers",
                    "d2h_gbs_per_rank": rank_d2h},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON result: whatever else a library writes to file descriptor 1
    (NCCL's "NCCL version ..." banner, for one) is sent to stderr for the rest of the run."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (weak) / in total (strong); default: the config's")
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS), help="BASELINE.json configs[] index (default 3)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-numa", action="store_true", help="do not bind the process to the GPU's NUMA node")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--nccl-gather", action="store_true", help="gather observations with NCCL instead of peer stores")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours in a single process")
    if args.warmup < 3:
        args.warmup = 3
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
