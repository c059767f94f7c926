"""Data-parallel K4 with per-trunk widths, one process per GPU (launched by tests/test_k4_trunks_gpu.py under
torch.distributed.run): every rank trains a mixed-width policy and its 64-64 embedding (zeros in the extra rows and
columns) on its own environment columns through the in-kernel all-reduce, and checks that both give the same bits and
that the replicas agree.  ICRL_DP_TRUNKS_WIDE=1 forces the many-cluster kernel."""
import ctypes as C
import os
import sys

import numpy as np
import torch as th
import torch.distributed as dist

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

TRUNKS = ((64, 64), (32, 32), (16, 48))


def train(dev, comm, trunks, P, loc, perm_dev, T, E_local, B_local, n_epochs):
    from icrl_b200 import _lib
    from icrl_b200.policies import ActorTwoCriticsPolicy
    from icrl_b200.spaces import Box
    D, A = loc["observations"].shape[-1], loc["actions"].shape[-1]
    pol = ActorTwoCriticsPolicy(Box(-np.inf, np.inf, (D,)), Box(-1, 1, (A,)), lambda _: 3e-4,
                                net_arch=[dict(zip(("pi", "vf", "cvf"), (list(t) for t in trunks)))], device=dev)
    pol.load_state_dict(P)
    spe = -(-T * E_local // B_local)
    cfg = pol.make_cfg(T=T, E=E_local, batch_size=B_local, n_epochs=n_epochs, has_target_kl=0, clip_range=0.2,
                       ent_coef=0.01, reward_vf_coef=0.5, cost_vf_coef=0.5, max_grad_norm=0.5, nu=0.7)
    data = _lib.PpoData()
    for k, v in loc.items():
        setattr(data, k, v.data_ptr())
    data.perm = perm_dev.data_ptr()
    advsums = th.zeros(n_epochs * spe, 4, dtype=th.float64, device=dev)
    stats = th.zeros(n_epochs * spe, 8, device=dev)
    result = th.zeros(4, dtype=th.int32, device=dev)
    L = _lib.lib()
    for _ in range(2):
        _lib.check(L.icrl_ppo_local_advsums(C.byref(cfg), C.byref(data), _lib.ptr(advsums), _lib.current_stream()))
        comm.all_reduce_sum(advsums)
        d = comm.descriptor(advsums)
        _lib.check(L.icrl_ppo_train_dist(C.byref(cfg), C.byref(data), _lib.ptr(pol._params), _lib.ptr(pol._adam_m),
                                         _lib.ptr(pol._adam_v), pol.optimizer.step_count, _lib.ptr(stats),
                                         _lib.ptr(result), C.byref(d), _lib.current_stream()))
        th.cuda.synchronize()
        res = result.cpu().numpy()
        assert res[2] == 0 and res[1] == n_epochs * spe, res
        pol.optimizer.step_count += int(res[1])
        comm.advance(int(res[1]))

    def named(flat):
        return {n: flat[off:off + int(np.prod(s))].reshape(s).cpu() for n, (off, s) in
                zip(pol.parameter_names(), pol._slices)}
    return pol, named(pol._params), named(pol._adam_m), named(pol._adam_v), stats.cpu()


def main():
    from icrl_b200.distributed import PpoComm, shard_envs
    from k4_trunks_helpers import embed, init_policy_trunks
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = th.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    th.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    wide = os.environ.get("ICRL_DP_TRUNKS_WIDE", "0") == "1"
    D, A, T, E_local, B_local, n_epochs = 18, 6, 32, 2, 32, 3
    if wide:
        T, E_local, B_local, n_epochs = 96, 4, 160, 2
        os.environ["ICRL_PPO_WIDE"], os.environ["ICRL_PPO_WIDE_CLUSTERS"] = "1", "6"
    E = E_local * world
    rng = np.random.default_rng(7)                       # identical global data on every rank
    g = {"observations": rng.standard_normal((T, E, D)).astype(np.float32),
         "actions": rng.standard_normal((T, E, A)).astype(np.float32)}
    for k in ("old_log_prob", "old_reward_values", "reward_advantages", "reward_returns", "old_cost_values",
              "cost_advantages", "cost_returns"):
        g[k] = rng.standard_normal((T, E)).astype(np.float32)
    g["old_log_prob"] = g["old_log_prob"] * 0.1 - 8.5
    lo, hi = shard_envs(E, rank, world)
    loc = {k: th.from_numpy(np.ascontiguousarray(v[:, lo:hi])).to(dev) for k, v in g.items()}
    n_local = T * E_local
    perm = np.stack([np.random.RandomState(100 * e + rank).permutation(n_local) for e in range(n_epochs)])
    perm_dev = th.from_numpy(perm.astype(np.int32)).to(dev)
    P = init_policy_trunks(D, A, False, TRUNKS, generator=th.Generator().manual_seed(3))
    P64 = embed(P, D, A, False)
    comm = PpoComm()
    ok = True
    try:
        pol, p, m, v, st = train(dev, comm, TRUNKS, P, loc, perm_dev, T, E_local, B_local, n_epochs)
        pol64, p64, m64, v64, st64 = train(dev, comm, ((64, 64),) * 3, P64, loc, perm_dev, T, E_local, B_local, n_epochs)
        ok &= th.equal(st, st64)
        for got, big in ((p, p64), (m, m64), (v, v64)):
            for n, t in got.items():
                inner = tuple(slice(0, s) for s in t.shape)
                pad = big[n].clone()
                pad[inner] = 0.0
                ok &= th.equal(t, big[n][inner]) and th.equal(pad, th.zeros_like(pad))
        allp = [th.empty_like(pol.parameters_flat()) for _ in range(world)]
        dist.all_gather(allp, pol.parameters_flat().contiguous())
        ok &= all(th.equal(x, allp[0]) for x in allp)
    finally:
        comm.close()
    flag = th.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("dp trunks ok" if flag.item() == 1.0 else "dp trunks MISMATCH", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
