#!/usr/bin/env python
"""
bench.py -- env-steps/sec of the B200-native batched simulator (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload kuka|mobile] [--no-secondary] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

Headline workload = BASELINE.json configs[1]: KukaButtonGymEnv-v0, ground_truth, 4096 envs per GPU,
synthetic random discrete actions + N(0, 0.01) step noise.  One bench "step" = ONE fused rollout of
T = 128 env steps over the whole batch (the n_steps of the reference's PPO2 runner,
rl_baselines/rl_algorithm/ppo2.py:58-72): a single kernel launch, 4096 x 128 env-steps.

  value : env-steps/s, actions/noise already resident in HBM, outputs left in HBM (CUDA events, max over ranks)
  e2e   : the same metric through the host-facing C-ABI call (srl_sim_rollout_host): pinned HOST action/noise
          buffers in, pinned HOST obs/reward/done out, copies inside the timed region
  roofline     : what bounds the dominant kernel, computed from THIS run's launch time and the committed ncu capture of
                 the very same SASS (profiles/r02_*_ncu.json; the ncu-derived terms are withheld when the hash differs)
  cpu_baseline : the CPU oracle (double precision, oracle/liboracle_sim.so, kind "port") on the host cores
  secondary    : the other two measurable BASELINE.json configs, in the same line so that the driver's record carries them:
                 mobile_config4   = configs[3], MobileRobotGymEnv-v0, 8192 envs/GPU, T = 1024 fused rollouts, at every N
                 plumbing_config1 = configs[0], MobileRobotGymEnv-v0, 4 env OBJECTS behind the reference-shaped
                                    (Dummy)VecEnv plumbing, random agent, 1600 steps (rank 0; BASELINE.md B3)
                 render_kuka      = image observations (SURVEY 8(f).4): one srl_sim_render of 4096 Kuka frames, 224 x 224 (rank 0)
                 ppo2_config3     = configs[2], PPO2 from rl_baselines.train on 4096 Kuka envs, 14 updates (rank 0)
  --impl reference : the reference arm.  PyBullet is not installable here, so it times the oracle -- the CPU
          restatement of the reference's step -- with every host thread, on the same configs.
  --dump-outputs DIR : after the timed steps, write what the headline rollout returned in the last timed step (rank 0's envs) as
          DIR/<name>.npy, so that two builds run with the same arguments can be compared output for output (see dump_outputs).
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "robotics-rl-srl_b200"))

KUKA_ENVS_PER_GPU = 4096      # BASELINE.json configs[1]
MOBILE_ENVS_PER_GPU = 8192    # BASELINE.json configs[3]
# Algorithmic HBM bytes (DESIGN.md "Measurement"): SoA state in + out once per launch, per-step I/O floor.
KUKA_STATE_BYTES = 2 * 224            # 12 float4 + 2 int4 records, read + written once per launch
KUKA_STEP_BYTES = 4 + 4 + 12 + 4 + 1  # action i32 + noise f32 in, obs f32[3] + reward f32 + done u8 out
# Algorithmic fp32 work of one Kuka env step = one applyAction + stepSimulation in steady state (no active contact):
#   150 sweeps x [12 motor rows x (2 x 12 flop velocity update + 6 flop row) + 3 button rows x 8 flop] = 150 x 384 = 57 600
#   + once per step: FK 3.2 k, CRBA + RNEA 4.8 k, Cholesky + M^-1 2.2 k, IK (7x7 normal equations) 2.4 k, rows / integration 0.6 k = 13.2 k
# SURVEY.md 8(d) quotes 1.6e5: it assumed 20 constraint rows of width 50 (contact, friction and limit rows always present);
# in steady state the solve has 15 rows of width 12, which is what the kernel (and PyBullet) actually iterates.
KUKA_FLOP_PER_STEP = 150 * (12 * (2 * 12 + 6) + 3 * 8) + 13200   # 70 800
MOBILE_STATE_BYTES = 2 * 80
MOBILE_STEP_BYTES = 4 + 8 + 4 + 1     # action in, obs f32[2] + reward + done out (in-kernel actions: no action read)
FP32_LANES_PER_SM = 128


def effective_cores():
    """Host threads that can actually run: min(visible CPUs, cgroup CPU quota).  The GPU boxes show 128 CPUs but the
    container's cgroup grants 16 CPUs of time (cpu.max = 1600000 100000); the oracle scales linearly to 16 threads and is
    flat beyond (scripts/cpu_scaling.py), so that is the core count reported with the CPU numbers."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(round(float(quota) / float(period)))))
    except Exception:
        pass
    return n


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed regions (B200_PROFILING.md recipe), through NVML at ~100 Hz (a bench of 20
    launches lasts ~0.15 s: nvidia-smi at 5 Hz saw one sample of it); falls back to nvidia-smi polling when NVML is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.sm, self.mx, self.reasons, self.n = [], [], set(), 0
        self._halt = threading.Event()
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else gpu_index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._phys = phys
        except Exception:
            self._nvml = None
            self._phys = gpu_index

    def _sample_nvml(self):
        nv = self._nvml
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)))
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)
        self.n += 1

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-i", str(self._phys)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            s = [x.strip() for x in out.split(",")]
            if s[1].replace(".", "").isdigit():
                self.sm.append(float(s[1]))
            if s[2].replace(".", "").isdigit():
                self.mx.append(float(s[2]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)
            self.n += 1

    def run(self):
        while not self._halt.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._halt.wait(0.01 if self._nvml is not None else 0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_min_mhz": min(self.sm) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons), "samples": self.n,
                "source": "nvml @100 Hz over the device-timed and the e2e region" if self._nvml is not None else "nvidia-smi @5 Hz"}


def make_inputs(workload, n, T, seed):
    rng = np.random.default_rng(seed)
    if workload == "kuka":
        acts = rng.integers(0, 6, (T, n), dtype=np.int32)
        noise = rng.normal(0, 0.01, (T, n)).astype(np.float32)
        return acts, noise
    return rng.integers(0, 4, (T, n), dtype=np.int32), None


DUMP_BUDGET_BYTES = 64 << 20
DUMP_SAMPLE_SEED = 12345


def dump_outputs(outdir, arrays):
    """Write host arrays laid out [T, n, ...] as <outdir>/<name>.npy.  float32 stays float32; integer outputs become float64, which holds
    them exactly.  When the arrays exceed DUMP_BUDGET_BYTES together, every one keeps the same env columns, a sample drawn from a fixed
    seed, so the files of two runs with the same arguments cover the same envs."""
    def out_dtype(a):
        return np.float32 if a.dtype == np.float32 else np.float64
    n = next(iter(arrays.values())).shape[1]
    total = sum(a.size * np.dtype(out_dtype(a)).itemsize for a in arrays.values())
    if total > DUMP_BUDGET_BYTES:
        cols = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(n, n * DUMP_BUDGET_BYTES // total, replace=False))
        arrays = {k: a[:, cols] for k, a in arrays.items()}
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), np.ascontiguousarray(a, dtype=out_dtype(a)))


def workload_spec(workload):
    if workload == "kuka":
        return dict(env_id="KukaButtonGymEnv-v0", n=KUKA_ENVS_PER_GPU, T=128, obs_dim=3, state_bytes=KUKA_STATE_BYTES,
                    step_bytes=KUKA_STEP_BYTES, cfg=dict(is_discrete=True, random_target=False, force_down=True, action_repeat=1, max_distance=0.8))
    return dict(env_id="MobileRobotGymEnv-v0", n=MOBILE_ENVS_PER_GPU, T=1024, obs_dim=2, state_bytes=MOBILE_STATE_BYTES,
                step_bytes=MOBILE_STEP_BYTES, cfg=dict(is_discrete=True, random_target=True))


def metric_and_config(workload, world):
    """`metric` / `config` of the JSON line -- shared by the b200 arm and the reference arm (the driver compares the two lines)."""
    spec = workload_spec(workload)
    n, T = spec["n"], spec["T"]
    metric = "env-steps/sec %s ground_truth @%d envs/GPU" % (spec["env_id"], n)
    config = {"workload": "%s ground_truth, %d envs/GPU, one bench step = one fused rollout of T=%d env steps (random discrete actions%s)"
                          % (spec["env_id"], n, T, " + N(0,0.01) step noise" if workload == "kuka" else ""),
              "envs_per_gpu": n, "env_steps_per_bench_step": n * T,
              "l2_flush_between_steps": "write 256 MB + read 256 MB between timed steps, outside the event bracket",
              "parallelism": "env-shard x%d" % world}
    return metric, config


def model_blob(workload):
    if workload != "kuka":
        return None
    from srl_sim.model import load_kuka_scene
    return load_kuka_scene().blob


# ------------------------------------------------------------------- committed ncu captures, keyed by SASS hash ----
KERNEL_PATTERN = {"kuka": "kuka_kernelILb0ELb0ELb0ELb1E", "mobile": "mobile_rollout_kernelILi4ELb1ELb0ELb0ELb1E"}   # 4096 Kuka envs run the four-lanes-per-env instantiation


def kernel_sass_sha16(lib_path, workload):
    """sha256 (16 hex digits) of the INSTRUCTION STREAM of the workload's dominant kernel as shipped in `lib_path`: `cuobjdump -sass`, the
    opcode + operand text of that one function, without addresses, encodings or the mangled name (which move when unrelated code is added
    to the translation unit while the kernel's code stays the same).  The ncu-derived constants of the roofline block are only valid for
    this exact code."""
    import re
    try:
        out = subprocess.run(["cuobjdump", "-sass", lib_path], capture_output=True, text=True, timeout=120).stdout
    except Exception:
        return None
    pat, keep, ins = KERNEL_PATTERN[workload], False, []
    for ln in out.splitlines():
        if "Function :" in ln:
            keep = pat in ln
            continue
        if keep:
            m = re.search(r"/\*[0-9a-f]{4,6}\*/\s+(.*?);", ln)
            if m:
                ins.append(re.sub(r"\s+", " ", m.group(1)).strip())
    if not ins:
        return None
    return hashlib.sha256("\n".join(ins).encode()).hexdigest()[:16]


def load_profile(workload, lib_path):
    """profiles/r02_<workload>_ncu.json (written by scripts/ncu_to_json.py from an `ncu --set full` capture of this bench) if it was taken
    from the SASS that is loaded now; otherwise (None, reason)."""
    p = os.path.join(ROOT, "profiles", "r02_%s_ncu.json" % workload)
    if not os.path.isfile(p):
        return None, "no committed capture (%s)" % os.path.relpath(p, ROOT)
    with open(p) as f:
        prof = json.load(f)
    sha = kernel_sass_sha16(lib_path, workload)
    if sha is None:
        return None, "cuobjdump unavailable: cannot check that the capture matches the loaded kernel"
    if prof.get("sass_sha16") != sha:
        return None, "stale capture: %s was taken from SASS %s, the loaded kernel is %s" % (os.path.basename(p), prof.get("sass_sha16"), sha)
    return prof, "profiles/%s (sass %s)" % (os.path.basename(p), sha)


def roofline_block(workload, spec, n, T, launch_s, clocks, lib_path, sms):
    peaks, peak_src = _peaks()
    launch_bytes = n * (spec["state_bytes"] + T * spec["step_bytes"])
    hbm_ach = launch_bytes / launch_s / 1e9
    prof, prof_note = load_profile(workload, lib_path)
    hbm = {"achieved": hbm_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_ach / peaks["hbm_gbs"],
           "peak_source": "%s (MEASURED_PEAKS.json hbm_gbs)" % peak_src, "algorithmic_bytes_per_launch": launch_bytes}
    traffic = prof.get("dram_bytes_per_launch") if prof else None
    if workload != "kuka":
        roof = dict(hbm)
        roof.update({"bound": "hbm", "traffic": traffic, "kernel": "mobile_rollout_kernel", "ncu_capture": prof_note})
        if prof:
            roof["note"] = ("frac is by ALGORITHMIC bytes; ncu saw %.1f MB reach DRAM per launch (the rest of the outputs is still in the 126 MB L2 "
                            "when the kernel ends), so part of this rate is L2-assisted" % (traffic / 1e6))
        return roof
    clk_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
    issue_peak = sms * 4 * clk_mhz * 1e-3                       # G warp-instructions/s: one per scheduler per cycle
    fp32_peak = sms * FP32_LANES_PER_SM * 2 * clk_mhz * 1e-6    # TFLOP/s, theoretical (no fp32 peak in MEASURED_PEAKS.json)
    fl = n * T * KUKA_FLOP_PER_STEP / launch_s / 1e12
    roof = {"bound": "fp32-issue", "unit": "G warp-inst/s", "peak": issue_peak, "achieved": None, "frac": None, "lane_util": None,
            "useful_lane_frac": None, "traffic": traffic, "kernel": "kuka_kernel", "ncu_capture": prof_note,
            "peak_source": "SMs x 4 schedulers x SM clock under load (%d x 4 x %.0f MHz)" % (sms, clk_mhz),
            "fp32": {"achieved": fl, "peak": fp32_peak, "unit": "TFLOP/s", "frac": fl / fp32_peak, "flop_per_env_step": KUKA_FLOP_PER_STEP,
                     "peak_source": "theoretical: SMs x 128 lanes x 2 x SM clock (MEASURED_PEAKS.json has no fp32 figure)"},
            "hbm": hbm,
            "note": "issue-bound fp32 kernel (150 strictly sequential PGS sweeps per env step), not HBM-bound; frac = warp instructions issued / "
                    "issue slots, lane_util = live threads per warp instruction / 32, distinct_lane_util discounts the lanes that repeat another lane's work (4 lanes per env run the sweeps redundantly), useful_lane_frac = frac x distinct_lane_util"}
    if prof:
        ach = prof["warp_inst_per_launch"] / launch_s / 1e9
        lane_util = prof["threads_per_warp_inst"] / 32.0
        # an env is a group of 4 lanes; in the sweeps (hot_loop_inst_share of the instructions) the 4 lanes compute the SAME values, so only a
        # quarter of those live lanes does distinct work; in the once-per-step code the 4 lanes split the work
        hot = prof.get("hot_loop_inst_share")
        lanes_per_env = 4.0 if "<0, 0, 0, 1>" in prof.get("kernel", "") or "ELb1EEE" in prof.get("kernel", "") else 1.0
        distinct = lane_util * ((hot / lanes_per_env + (1.0 - hot)) if hot is not None else 1.0 / lanes_per_env)
        roof.update({"achieved": ach, "frac": ach / issue_peak, "lane_util": lane_util, "distinct_lane_util": distinct,
                     "useful_lane_frac": ach / issue_peak * distinct, "lanes_per_env": lanes_per_env, "sweep_inst_share": hot,
                     "warp_inst_per_launch": prof["warp_inst_per_launch"]})
    return roof


# ------------------------------------------------------------------------------- CPU oracle legs --------
def _oracle_library():
    from srl_sim._abi import SimLibrary
    path = os.path.join(ROOT, "oracle", "liboracle_sim.so")
    if not os.path.isfile(path):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    return SimLibrary(path)


def _oracle_backend():
    from srl_sim.backend import Backend
    return Backend(_oracle_library(), -1)


class OraclePool(object):
    """The CPU oracle sharded over `threads` host threads (ctypes releases the GIL), one sim handle per thread --
    the same one-env-group-per-worker shape as the reference's SubprocVecEnv (rl_baselines/utils.py:216-220)."""

    def __init__(self, workload, n_total, T, threads, seed=0):
        spec = workload_spec(workload)
        be = _oracle_backend()
        self.T, self.n_total, self.threads = T, n_total, max(1, min(threads, n_total))
        blob = model_blob(workload)
        bounds = np.linspace(0, n_total, self.threads + 1).astype(int)
        self.parts = []
        acts, noise = make_inputs(workload, n_total, T, seed + 100)
        for k in range(self.threads):
            lo, hi = int(bounds[k]), int(bounds[k + 1])
            if hi == lo:
                continue
            sim = be.make_sim(spec["env_id"], hi - lo, seed=seed, model_blob=blob, global_env_offset=lo, **spec["cfg"])
            sim.reset()
            a = np.ascontiguousarray(acts[:, lo:hi]); nz = None if noise is None else np.ascontiguousarray(noise[:, lo:hi])
            obs = np.zeros((T, hi - lo, spec["obs_dim"]), np.float32); rew = np.zeros((T, hi - lo), np.float32)
            done = np.zeros((T, hi - lo), np.uint8)
            self.parts.append((sim, a, nz, obs, rew, done))

    def step(self):
        ths = [threading.Thread(target=lambda p=p: p[0].rollout(self.T, p[1], p[2], p[3], p[4], p[5])) for p in self.parts]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        return time.perf_counter() - t0


def cpu_sample_T(workload):
    return workload_spec(workload)["T"] if workload == "kuka" else 256


def cpu_baseline(workload, cores):
    spec = workload_spec(workload)
    # bounded sample: a slice of the same workload worth ~10-30 s of single-core work
    T, n = cpu_sample_T(workload), spec["n"]
    pool = OraclePool(workload, n, T, cores)
    pool.step()  # warm-up (page in, caches)
    dt = min(pool.step() for _ in range(2))
    return {"value": n * T / dt, "unit": "env-steps/s", "cores": pool.threads, "kind": "port",
            "sample": "%d envs x %d steps of %s, oracle/liboracle_sim.so (float64 CPU restatement, no rendering, no Python in the "
                      "loop), %d host threads" % (n, T, spec["env_id"], pool.threads)}


def plumbing_config1(library, device, steps=1600, num_cpu=4, seed=0):
    """BASELINE.json configs[0] / BASELINE.md B3: MobileRobotGymEnv-v0, ground_truth, 4 env OBJECTS behind the reference-shaped VecEnv
    plumbing (createEnvs -> makeEnv thunks -> DummyVecEnv -> VecFrameStack -> VecNormalize), stepped by the random agent's loop
    (/root/reference/rl_baselines/random_agent.py:28-42) for 1600 env steps (/root/reference/tests/test_pipeline.py:14, NUM_TIMESTEP).
    `library`/`device`: the sm_100a library on a GPU (product) or the oracle with device -1 (reference arm)."""
    import types
    from srl_sim import backend as srl_backend
    from rl_baselines.utils import createEnvs
    prev = srl_backend._override
    srl_backend.use_library(library, device)
    try:
        args = types.SimpleNamespace(env="MobileRobotGymEnv-v0", num_cpu=num_cpu, seed=seed, num_stack=1, srl_model="ground_truth",
                                     per_env_objects=True, log_dir=None)
        envs = createEnvs(args, env_kwargs=dict(is_discrete=True))
        envs.action_space.seed(seed)
        envs.reset()
        n_updates = steps // num_cpu
        for _ in range(20):                                              # warm-up
            envs.step([envs.action_space.sample() for _ in range(num_cpu)])
        t0 = time.perf_counter()
        ndone = 0
        for _ in range(n_updates):
            _, _, dones, _ = envs.step([envs.action_space.sample() for _ in range(num_cpu)])
            ndone += int(np.sum(dones))
        dt = time.perf_counter() - t0
        envs.close()
    finally:
        srl_backend._override = prev
    return {"metric": "env-steps/sec MobileRobotGymEnv-v0 ground_truth, %d env objects, random agent (reference-shaped VecEnv plumbing)" % num_cpu,
            "value": n_updates * num_cpu / dt, "unit": "env-steps/s", "env_steps": n_updates * num_cpu, "episodes_finished": ndone,
            "launches_per_env_step": 1, "note": "one N=1 simulator launch + one synchronising read-back per env object and step: Python / launch-latency bound"}


def render_leg(be, n=4096, width=224, height=224, reps=10):
    """Image observations (SURVEY 8(f).4): device time of one srl_sim_render of n Kuka frames (primitive lists, prepared primitives, raster:
    3 launches), CUDA events, a 256 MB L2 flush between repetitions; the kernel is instruction-issue bound, so the roofline entry is the
    byte floor of the output only (3 W H bytes per frame at the measured HBM peak)."""
    import numpy as np
    import torch
    from srl_sim.model import load_kuka_scene
    from srl_sim.render import KUKA_CAMERA, camera
    st = be.stream()
    sim = be.make_sim("KukaButtonGymEnv-v0", n, model_blob=load_kuka_scene().blob, seed=0, random_target=True)
    sim.reset(stream=st)
    T = 32
    acts = torch.randint(0, 6, (T, n), dtype=torch.int32, device=be.torch_device)
    o = be.zeros((T, n, 3), np.float32); r = be.zeros((T, n), np.float32); d = be.zeros((T, n), np.uint8)
    sim.rollout(T, acts, None, o, r, d, stream=st)
    buf = be.zeros((n, height, width, 3), np.uint8)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=be.torch_device)
    cam = camera(**KUKA_CAMERA)
    for _ in range(3):
        sim.render(cam, width, height, buf, stream=st)
    ms = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream()); sim.render(cam, width, height, buf, stream=st); e1.record(torch.cuda.current_stream())
        torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
    sim.close()
    t = float(np.median(ms)) * 1e-3
    out_bytes = 3 * width * height * n
    peaks, src = _peaks()
    hbm = float(peaks.get("hbm_gbs", 0.0) or 0.0) * 1e9
    return {"metric": "frames/sec srl_sim_render KukaButtonGymEnv-v0 %dx%d @%d envs" % (width, height, n), "value": n / t, "unit": "frames/s",
            "ms_per_call": t * 1e3, "gpu_launches_per_call": 3, "bytes_written_per_call": out_bytes,
            "roofline": {"bound": "issue (ray / primitive arithmetic; profiles/r02_render_raster_ncu.txt: 80 % of the issue slots)",
                         "hbm_floor_ms": (out_bytes / hbm * 1e3) if hbm else None, "hbm_frac": (out_bytes / t / hbm) if hbm else None, "peak_source": src},
            "config": {"workload": "one 224 x 224 RGB frame per env through the env's fixed camera, analytic-primitive ray caster (DESIGN.md 5.3)",
                       "l2": "256 MB flush between repetitions", "reps": reps}}


def ppo2_leg(device_index, updates=14):
    """BASELINE configs[2]: KukaButtonGymEnv-v0 ground_truth, PPO2 from rl_baselines.train, 4096 envs on one B200 -- the trainer's own loop (policy step,
    lockstep simulator step with next-episode records, observation filter: three launches per env step inside a captured graph; GAE and the
    16 minibatch gradients through srl_ppo2_gae / srl_ppo2_grad; clip + Adam in torch).  `value` = env-steps/s over the updates after the
    first four (graph captures and warm-up excluded), `cumulative` includes them."""
    from rl_baselines.ppo2 import train
    n, T = 4096, 128
    t0 = time.time()
    hist = train("KukaButtonGymEnv-v0", n, n * T * updates, seed=0, verbose=0, device=device_index)
    wall = time.time() - t0
    times = [st / fps for st, _, fps in hist]                  # seconds since the training loop started, per update
    k = min(4, len(hist) - 2)
    steady = (hist[-1][0] - hist[k][0]) / max(times[-1] - times[k], 1e-9)
    return {"metric": "env-steps/sec PPO2 training KukaButtonGymEnv-v0 ground_truth @4096 envs (rl_baselines.train --algo ppo2)", "value": steady, "unit": "env-steps/s",
            "cumulative_incl_graph_capture": hist[-1][2], "updates": len(hist), "steady_state_over_updates": [k + 2, len(hist)],
            "ms_per_update": 1e3 * (times[-1] - times[k]) / (len(hist) - 1 - k), "mean_episode_return_last": hist[-1][1], "wall_s_incl_env_setup": wall,
            "config": {"workload": "n_steps 128, nminibatches 4, noptepochs 4 (reference hyper-parameters), 524 288 samples per update", "data": "synthetic: the env's own random resets"}}


def render_reference_leg(cores, frames_per_thread=4, width=224, height=224):
    """The render leg on the host: the CPU checker of the ray caster (oracle/liboracle_sim.so, the same primitive lists and per-pixel arithmetic
    as the CUDA kernels, csrc/render_core.h) on every host thread, one env shard per thread, a bounded sample of the 4096-frame call.  The
    reference itself renders with PyBullet's TinyRenderer (CPU, one 224 x 224 frame per env step: the published 250 FPS on 8 cores includes it)."""
    from srl_sim.model import load_kuka_scene
    from srl_sim.render import KUKA_CAMERA, camera
    be = _oracle_backend()
    blob = load_kuka_scene().blob
    parts = []
    for k in range(max(1, cores)):
        sim = be.make_sim("KukaButtonGymEnv-v0", frames_per_thread, seed=0, model_blob=blob, global_env_offset=k * frames_per_thread, random_target=True)
        sim.reset()
        parts.append((sim, np.zeros((frames_per_thread, height, width, 3), np.uint8)))
    cam = camera(**KUKA_CAMERA)

    def once():
        ths = [threading.Thread(target=lambda p=p: p[0].render(cam, width, height, p[1])) for p in parts]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        return time.perf_counter() - t0
    once()
    t = min(once() for _ in range(2))
    n = frames_per_thread * len(parts)
    return {"metric": "frames/sec srl_sim_render KukaButtonGymEnv-v0 %dx%d (CPU checker)" % (width, height), "value": n / t, "unit": "frames/s", "cores": len(parts),
            "sample": "%d frames (%d per host thread) of the 4096-frame call, every pixel against every primitive (the CPU checker does not cull)" % (n, frames_per_thread)}


def run_reference(args):
    """--impl reference: the CPU restatement of the reference's own step on all host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = effective_cores()

    def run(workload, steps, warmup):
        spec = workload_spec(workload)
        n, T = spec["n"], cpu_sample_T(workload)
        pool = OraclePool(workload, n, T, cores)
        for _ in range(warmup):
            pool.step()
        times = [pool.step() for _ in range(steps)]
        return n, T, pool.threads, sum(times), pool

    spec = workload_spec(args.workload)
    n, T, threads, total, pool = run(args.workload, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {name: np.concatenate([p[k] for p in pool.parts], axis=1)
                                         for name, k in (("obs", 3), ("reward", 4), ("done", 5))})
    value = n * T * args.steps / total
    sample = ("%d envs x %d steps per step, %d host threads (container CPU quota; %d CPUs visible), CPU oracle "
              "(PyBullet itself is not installable offline)" % (n, T, threads, os.cpu_count() or 1))
    metric, config = metric_and_config(args.workload, 1)
    config["parallelism"] = "%d host threads, one env shard each (rank 0 only)" % threads
    config["l2_flush_between_steps"] = "n/a (CPU run)"
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        config["reference_shard"] = ("rank 0 alone steps ONE %d-env shard on all host threads (the CPU is saturated by it); the b200 arm steps one shard per GPU "
                                     "-- the two lines compare throughput with throughput" % n)
    if T != spec["T"]:
        config["reference_sample"] = "bounded sample: %d of the %d env steps per bench step" % (T, spec["T"])
    line = {"impl": "reference", "metric": metric, "value": value, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not args.no_secondary and args.workload == "kuka":
        sec = {}
        mn, mT, mth, mtot, _ = run("mobile", 3, 1)
        sec["mobile_config4"] = {"metric": metric_and_config("mobile", 1)[0], "value": mn * mT * 3 / mtot, "unit": "env-steps/s", "cores": mth,
                                 "sample": "%d envs x %d steps per step x 3 (bounded sample of the T=1024 rollout), CPU oracle" % (mn, mT)}
        sec["plumbing_config1"] = plumbing_config1(_oracle_library(), -1)
        sec["plumbing_config1"]["impl"] = "CPU oracle behind the same Python env objects (stand-in for PyBullet + SubprocVecEnv)"
        try:
            sec["render_kuka"] = render_reference_leg(cores)
        except Exception as ex:
            sec["render_kuka"] = {"error": repr(ex)}
        line["secondary"] = sec
    print(json.dumps(line))


# ----------------------------------------------------------------------------------- GPU arm -------------
def measure_b200(be, workload, args, rank, world, local_rank, dist, sampler_holder, dump_dir=None):
    """Device-timed and end-to-end throughput of one workload on this rank's GPU; max over ranks.  Returns a dict on every rank.
    With `dump_dir`, rank 0 writes the outputs of the last timed rollout there (dump_outputs)."""
    import torch
    spec = workload_spec(workload)
    n, T, D = spec["n"], spec["T"], spec["obs_dim"]
    sim = be.make_sim(spec["env_id"], n, seed=args.seed, model_blob=model_blob(workload), global_env_offset=rank * n, **spec["cfg"])
    st = be.stream()
    sim.reset(stream=st)
    acts_h, noise_h = make_inputs(workload, n, T, args.seed + 1000 * rank)
    acts = be.from_host(acts_h)
    noise = None if noise_h is None else be.from_host(noise_h)
    obs = be.zeros((T, n, D), np.float32); rew = be.zeros((T, n), np.float32); done = be.zeros((T, n), np.uint8)
    ep_ret = be.zeros((T, n), np.float32); ep_len = be.zeros((T, n), np.int32)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=be.torch_device)  # > 126 MB L2
    flush_rd = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=be.torch_device)  # 256 MB, only ever read
    sink = torch.zeros((), dtype=torch.float32, device=be.torch_device)

    def step():
        sim.rollout(T, acts, noise, obs, rew, done, ep_ret, ep_len, stream=st)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    steps, warmup = args.steps, max(args.warmup, 3)
    for _ in range(warmup):
        step()
    barrier()
    launches0 = sim.launch_count
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    wall0 = time.perf_counter()
    for k in range(steps):
        # evict L2 between timed iterations (outside the event bracket): WRITE a buffer larger than L2, then READ another
        # one so that the timed kernel starts from a cold L2 holding clean lines -- otherwise it would also pay the DRAM
        # write-back of up to 126 MB of the flush buffer's dirty lines, which is not its traffic
        flush.fill_(k & 0xff)
        sink += flush_rd.sum()
        ev[k][0].record()
        step()
        ev[k][1].record()
    barrier()
    wall = time.perf_counter() - wall0
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"obs": be.to_host(obs), "reward": be.to_host(rew), "done": be.to_host(done),
                                "episode_return": be.to_host(ep_ret), "episode_length": be.to_host(ep_len)})
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    launches = sim.launch_count - launches0

    # ---- e2e: host buffers through srl_sim_rollout_host ----
    pin = lambda a: torch.from_numpy(a).pin_memory()
    h_acts = pin(acts_h); h_noise = None if noise_h is None else pin(noise_h)
    h_obs = torch.empty((T, n, D), dtype=torch.float32).pin_memory(); h_rew = torch.empty((T, n), dtype=torch.float32).pin_memory()
    h_done = torch.empty((T, n), dtype=torch.uint8).pin_memory()

    def e2e_step():
        sim.rollout_host(T, h_acts, h_noise, h_obs, h_rew, h_done)

    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if sampler else None
    h2d = h_acts.numel() * 4 + (0 if h_noise is None else h_noise.numel() * 4)
    d2h = h_obs.numel() * 4 + h_rew.numel() * 4 + h_done.numel()

    # ---- max over ranks; cross-rank episode-return all-gather (the only collective; off the step path) ----
    tms = torch.tensor([total_ms, e2e_s * 1e3, wall * 1e3], device=be.torch_device, dtype=torch.float64)
    d = done.bool()
    ep_stats = torch.stack([ep_ret[d].sum().double(), d.sum().double()])
    slow_rank = None
    if world > 1:
        per_rank = [torch.zeros_like(tms) for _ in range(world)]
        dist.all_gather(per_rank, tms)
        per_rank = torch.stack(per_rank)
        slow_rank = {"rank": int(per_rank[:, 0].argmax().item()), "device_ms_per_step_by_rank": [float(x) / steps for x in per_rank[:, 0].tolist()]}
        tms = per_rank.max(0).values
        gathered = [torch.zeros_like(ep_stats) for _ in range(world)]
        dist.all_gather(gathered, ep_stats)
        ep_stats = torch.stack(gathered).sum(0)
    total_ms, e2e_ms, wall_ms = [float(x) for x in tms.tolist()]
    sim.close()
    del flush, flush_rd
    torch.cuda.empty_cache()
    units = n * T * world
    sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    launch_s = (total_ms / steps) * 1e-3
    res = {"value": units * steps / (total_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": total_ms / steps, "steps": steps, "warmup": warmup,
           "gpu_launches": launches, "clocks": clocks,
           "e2e": {"value": units * steps / (e2e_ms * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
           "wall_ms_total_incl_flush": wall_ms, "episodes_finished": int(ep_stats[1].item()),
           "episode_return_mean": float(ep_stats[0].item() / max(1.0, ep_stats[1].item()))}
    if slow_rank:
        res["slowest_rank"] = slow_rank
    if rank == 0:
        res["roofline"] = roofline_block(workload, spec, n, T, launch_s, clocks, be.library.path, sms)
    return res


def run_b200(args):
    import torch
    import torch.distributed as dist
    from srl_sim._abi import load_cuda_library
    from srl_sim.backend import Backend

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    be = Backend(load_cuda_library(), local_rank)
    main = measure_b200(be, args.workload, args, rank, world, local_rank, dist, None, dump_dir=args.dump_outputs)
    secondary = {}
    if not args.no_secondary and args.workload == "kuka":
        m = measure_b200(be, "mobile", args, rank, world, local_rank, dist, None)
        if rank == 0:
            mmetric, mconfig = metric_and_config("mobile", world)
            m.update({"metric": mmetric, "config": mconfig, "dtype": "f64", "scaling": "weak", "n_gpus": world})
            secondary["mobile_config4"] = m
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if not args.no_secondary and args.workload == "kuka":
        try:
            secondary["plumbing_config1"] = plumbing_config1(be.library, local_rank)
        except Exception as ex:      # never lose the headline line to the secondary leg
            secondary["plumbing_config1"] = {"error": repr(ex)}
        try:
            secondary["render_kuka"] = render_leg(be)
        except Exception as ex:
            secondary["render_kuka"] = {"error": repr(ex)}
        try:
            secondary["ppo2_config3"] = ppo2_leg(local_rank)
        except Exception as ex:
            secondary["ppo2_config3"] = {"error": repr(ex)}
    metric, config = metric_and_config(args.workload, world)
    line = {"metric": metric, "value": main["value"], "unit": "env-steps/s",
            "n_gpus": world, "steps": main["steps"], "warmup": main["warmup"], "ms_per_step": main["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.workload == "kuka" else "f64", "data": "synthetic",
            "config": config,
            "clocks": main["clocks"], "gpu_launches": main["gpu_launches"],
            "e2e": main["e2e"], "roofline": main["roofline"],
            "wall_ms_total_incl_flush": main["wall_ms_total_incl_flush"],
            "episodes_finished": main["episodes_finished"], "episode_return_mean": main["episode_return_mean"]}
    if "slowest_rank" in main:
        line["slowest_rank"] = main["slowest_rank"]
    if secondary:
        line["secondary"] = secondary
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args.workload, effective_cores())
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="kuka", choices=["kuka", "mobile"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs[3] / configs[0] legs (A/B scripts, ncu captures)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
