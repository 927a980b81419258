"""Device time of every kuka_kernel instantiation <JOINTS, TWOB, PREFETCH, COOP> on one seeded workload each (run on a GPU machine):

    SRL_SIM_CUDA_LIB=<lib.so> python scripts/kuka_instantiation_timing.py

COOP = 1 at 4096 envs (four lanes per env), COOP = 0 at 16 384 envs (one thread per env, chosen above 4736 envs).  Rollouts: median of
4 timed 128-step launches after 3 warm-up launches.  PREFETCH: lockstep srl_sim_step with next-episode records, median of 128 launches
after 10 warm-up rollouts.  Meant for A/B runs of two builds of the same code in one session."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "robotics-rl-srl_b200"))
import torch  # noqa: E402
from srl_sim._abi import load_cuda_library  # noqa: E402
from srl_sim.backend import Backend  # noqa: E402
from srl_sim.model import load_kuka_scene  # noqa: E402

T = 128
# "<JOINTS,TWOB" of the instantiation -> (env kind, action kind, make_sim config)
VARIANTS = {
    "<0,0": ("KukaButtonGymEnv-v0", "discrete", dict(is_discrete=True)),
    "<1,0": ("KukaButtonGymEnv-v0", "joints", dict(is_discrete=False, action_joints=True)),
    "<0,1": ("Kuka2ButtonGymEnv-v0", "discrete", dict(is_discrete=True)),
    "<1,1": ("Kuka2ButtonGymEnv-v0", "joints", dict(is_discrete=False, action_joints=True)),
}


def _actions(be, kind, n):
    rs = np.random.RandomState(1)
    if kind == "discrete":
        return be.from_host(rs.randint(0, 6, size=(T, n)).astype(np.int32))
    return be.from_host(rs.uniform(-1, 1, size=(T, n, 7)).astype(np.float32))


def main():
    be = Backend(load_cuda_library(), 0)
    blob = load_kuka_scene().blob
    st = be.stream()
    for n, coop in ((4096, 1), (16384, 0)):
        obs = be.zeros((T, n, 3), np.float32); rew = be.zeros((T, n), np.float32); done = be.zeros((T, n), np.uint8)
        for name, (kind, akind, cfg) in VARIANTS.items():
            sim = be.make_sim(kind, n, model_blob=blob, seed=1, **cfg)
            sim.reset(stream=st)
            a = _actions(be, akind, n)
            ms = []
            for it in range(7):
                sim.rollout(T, a, None, obs, rew, done, stream=st)
                if it >= 3:
                    ms.append(sim.last_kernel_ms())
            torch.cuda.synchronize()
            sim.close()
            print("kuka_kernel%s,0,%d> %5d envs: rollout %.3f ms (median of %d; spread %.3f)"
                  % (name, coop, n, np.median(ms), len(ms), max(ms) - min(ms)), flush=True)
        sim = be.make_sim("KukaButtonGymEnv-v0", n, model_blob=blob, seed=0, prefetch_resets=True, is_discrete=True)
        o1 = be.zeros((n, 3), np.float32); r1 = be.zeros((n,), np.float32); d1 = be.zeros((n,), np.uint8)
        sim.reset(obs_out=o1, stream=st)
        a = _actions(be, "discrete", n)
        for _ in range(10):
            sim.rollout(T, a, None, obs, rew, done, stream=st)
        sim.prefetch_resets(stream=st)
        ms = []
        for t in range(T):
            sim.step(a[t], None, o1, r1, d1, None, None, stream=st)
            ms.append(sim.last_kernel_ms())
        torch.cuda.synchronize()
        sim.close()
        print("kuka_kernel<0,0,1,%d> %5d envs: lockstep step %.1f us (median of %d)" % (coop, n, 1e3 * np.median(ms), len(ms)), flush=True)


if __name__ == "__main__":
    main()
