"""Bit-for-bit A/B of two builds of the sm_100a library on seeded Kuka runs (run on a GPU machine):

    python scripts/kuka_ab_bitexact.py <libA.so> <libB.so>

Each library runs every case in a process of its own (SRL_SIM_CUDA_LIB selects it); every output array -- observations, rewards, done
flags, episode returns / lengths and the final joint state -- must be byte-equal.  The cases cover the kernel instantiations a change to
the Kuka device code can reach: BASELINE configs 2 and 5, action_repeat = 3, force_down = False, the two-button env, action_joints, a
lockstep run with next-episode records (prefetch_resets) and a batch above 4736 envs (one thread per env instead of four lanes)."""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# name -> (env kind, envs, steps, action kind, make_sim config, lockstep)
CASES = {
    "config2": ("KukaButtonGymEnv-v0", 4096, 256, "discrete", dict(seed=0, is_discrete=True, force_down=True, action_repeat=1, max_distance=0.8), False),
    "config5": ("KukaRandButtonGymEnv-v0", 4096, 256, "continuous", dict(seed=0, is_discrete=False, random_target=True, force_down=True, action_repeat=1, max_distance=0.8), False),
    "action_repeat3": ("KukaButtonGymEnv-v0", 1024, 200, "discrete", dict(seed=1, is_discrete=True, action_repeat=3), False),
    "no_force_down": ("KukaButtonGymEnv-v0", 1024, 300, "discrete", dict(seed=2, is_discrete=True, force_down=False), False),
    "two_button": ("Kuka2ButtonGymEnv-v0", 1024, 300, "discrete", dict(seed=3, is_discrete=True), False),
    "action_joints": ("KukaButtonGymEnv-v0", 1024, 200, "joints", dict(seed=4, is_discrete=False, action_joints=True, max_steps=150), False),
    "lockstep_prefetch": ("KukaButtonGymEnv-v0", 512, 120, "discrete", dict(seed=5, is_discrete=True, max_steps=40, prefetch_resets=True), True),
    "thread_per_env": ("KukaButtonGymEnv-v0", 6144, 128, "discrete", dict(seed=6, is_discrete=True), False),
}


def _actions(kind, T, n, seed):
    rs = np.random.RandomState(seed)
    if kind == "discrete":
        return rs.randint(0, 6, size=(T, n)).astype(np.int32)
    if kind == "continuous":
        return rs.uniform(-1, 1, size=(T, n, 3)).astype(np.float32)
    return rs.uniform(-1, 1, size=(T, n, 7)).astype(np.float32)


def _run_cases(out_dir):
    sys.path.insert(0, os.path.join(ROOT, "robotics-rl-srl_b200"))
    import torch
    from srl_sim import _abi
    from srl_sim._abi import load_cuda_library
    from srl_sim.backend import Backend
    from srl_sim.model import load_kuka_scene
    be = Backend(load_cuda_library(), 0)
    blob = load_kuka_scene().blob
    for name, (kind, n, T, akind, cfg, lockstep) in CASES.items():
        sim = be.make_sim(kind, n, model_blob=blob, **cfg)
        st = be.stream()
        a = be.from_host(_actions(akind, T, n, 100 + len(name)))
        if lockstep:
            obs = be.zeros((n, 3), np.float32); rew = be.zeros((n,), np.float32); done = be.zeros((n,), np.uint8)
            ep_ret = be.zeros((n,), np.float32); ep_len = be.zeros((n,), np.int32)
            sim.reset(obs_out=obs, stream=st)
            sim.prefetch_resets(stream=st)
            out = {k: [] for k in ("obs", "rew", "done", "ep_ret", "ep_len")}
            for t in range(T):
                sim.step(a[t], None, obs, rew, done, ep_ret, ep_len, stream=st)
                for k, v in (("obs", obs), ("rew", rew), ("done", done), ("ep_ret", ep_ret), ("ep_len", ep_len)):
                    out[k].append(be.to_host(v).copy())
            out = {k: np.stack(v) for k, v in out.items()}
        else:
            obs0 = be.zeros((n, 3), np.float32)
            sim.reset(obs_out=obs0, stream=st)
            obs = be.zeros((T, n, 3), np.float32); rew = be.zeros((T, n), np.float32); done = be.zeros((T, n), np.uint8)
            ep_ret = be.zeros((T, n), np.float32); ep_len = be.zeros((T, n), np.int32)
            sim.rollout(T, a, None, obs, rew, done, ep_ret, ep_len, stream=st)
            out = dict(obs0=be.to_host(obs0).copy(), obs=be.to_host(obs).copy(), rew=be.to_host(rew).copy(), done=be.to_host(done).copy(),
                       ep_ret=be.to_host(ep_ret).copy(), ep_len=be.to_host(ep_len).copy())
        torch.cuda.synchronize()
        out["q"] = sim.get_state(_abi.F_JOINT_POS); out["qd"] = sim.get_state(_abi.F_JOINT_VEL)
        sim.close()
        np.savez(os.path.join(out_dir, name + ".npz"), **out)
        print(f"  {name}: {n} envs x {T} steps, {int(out['done'].sum())} episodes finished", flush=True)


def main():
    if len(sys.argv) == 3 and sys.argv[1] == "--run":
        _run_cases(sys.argv[2])
        return 0
    if len(sys.argv) != 3:
        print(__doc__)
        return 2
    libs = [os.path.abspath(p) for p in sys.argv[1:]]
    with tempfile.TemporaryDirectory() as tmp:
        dirs = []
        for k, lib in enumerate(libs):
            d = os.path.join(tmp, str(k)); os.makedirs(d); dirs.append(d)
            print(os.path.basename(lib), flush=True)
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "--run", d], env=dict(os.environ, SRL_SIM_CUDA_LIB=lib))
        bad = 0
        for name in CASES:
            a = np.load(os.path.join(dirs[0], name + ".npz")); b = np.load(os.path.join(dirs[1], name + ".npz"))
            diff = [k for k in a.files if a[k].dtype != b[k].dtype or a[k].shape != b[k].shape or a[k].tobytes() != b[k].tobytes()]
            print(f"{name}: {'byte-equal' if not diff else 'DIFFERENT: ' + ', '.join(diff)} ({len(a.files)} arrays)")
            bad += bool(diff)
    print("all cases byte-equal" if not bad else f"{bad} case(s) differ")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
