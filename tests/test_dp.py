"""Data-parallel host logic.  CPU: world_size-2 gloo run of the pieces that do not need a GPU (shard
filter of the global permutation, all-reduce plumbing).  GPU: 1-vs-2-GPU equivalence via torchrun."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GLOO_WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200")); sys.path.insert(0, ROOT)
from diamond.agents import _PermWorker, _Dist, permutation_plan
from oracle.dp_oracle import shard_filter
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
d = _Dist(None, True, "global")
assert d.enabled and d.world == world and d.rank == rank and d.global_perm
# ranks start from different numpy streams; sync_numpy_stream puts everyone on rank 0's
np.random.seed(5 + 17 * rank)
np.random.normal()                                         # leaves a cached gaussian on every rank (part of the legacy state)
d.sync_numpy_stream()
T, NL, MB, E = 8, 6, 4, 3
NG, B = NL * world, T * NL * world
M = B // MB
plan = permutation_plan(T * NL, world, MB, True)
assert plan["B_perm"] == B and plan["filter"] and plan["rows"] <= T * NL
outs = [np.empty(B, np.int32) for _ in range(E)]
w = _PermWorker(B, E, MB, outs); w.start()
for e in range(E): w.wait(e)
w.finish()
h = torch.tensor([w.state_hash, w.state_hash ** 2], dtype=torch.float64); d.all_reduce_sum(h)
assert abs(float(h[1]) * world - float(h[0]) ** 2) < 0.5    # the lockstep check learn() carries through its all-reduce
after = torch.tensor(np.random.randint(0, 2**31, 2)); ref_after = after.clone(); dist.broadcast(ref_after, src=0)
assert torch.equal(after, ref_after)                        # streams still agree after the permutations
for e in range(E):
    everyone = [None] * world
    dist.all_gather_object(everyone, outs[e].tolist())
    assert all(x == everyone[0] for x in everyone)          # the same global permutation on every rank
    idx, counts, overflow = shard_filter(outs[e], NG, rank * NL, NL, MB, plan["rows"])
    assert overflow == 0
    seen = []
    for k in range(MB):
        loc = idx[k, :counts[k]]
        assert (idx[k, counts[k]:] == -1).all()
        t, env = np.divmod(loc, NL)
        glob = t * NG + env + rank * NL                     # local flat index -> global flat index
        seg = outs[e][k * M:(k + 1) * M]
        mine = seg[(seg % NG >= rank * NL) & (seg % NG < (rank + 1) * NL)]
        assert np.array_equal(glob, mine), (e, k)           # same members, same order as the global minibatch
        seen.append(loc)
        cnt = torch.tensor([int(counts[k])]); dist.all_reduce(cnt); assert int(cnt) == M     # shards partition every minibatch
    assert sorted(np.concatenate(seen).tolist()) == list(range(T * NL))
# epoch ownership: rank e % world shuffles epoch e, the others only advance the stream (skip) -- same stream on every rank afterwards,
# and the owned permutations are the ones the plain generator produces
np.random.seed(21)
plain = [np.random.permutation(B) for _ in range(E)]
tail_ref = np.random.randint(0, 2**31, 2)
np.random.seed(21)
outs2 = [np.full(B, -7, np.int32) for _ in range(E)]
w3 = _PermWorker(B, E, MB, outs2, lambda e: e % world == rank); w3.start(); w3.finish()
assert np.array_equal(np.random.randint(0, 2**31, 2), tail_ref)
for e in range(E):
    if e % world == rank: assert np.array_equal(outs2[e], plain[e])
    else: assert (outs2[e] == -7).all()
# a rank whose stream was consumed differently is caught by the hash check
if rank == 1: np.random.random()
w2 = _PermWorker(B, 1, MB, [np.empty(B, np.int32)])
h = torch.tensor([w2.state_hash, w2.state_hash ** 2], dtype=torch.float64); d.all_reduce_sum(h)
assert abs(float(h[1]) * world - float(h[0]) ** 2) > 0.5
x = torch.full((5,), float(rank + 1), dtype=torch.float64); d.all_reduce_sum(x)
assert torch.equal(x, torch.full((5,), float(sum(range(1, world + 1))), dtype=torch.float64))
dist.destroy_process_group()
print("ok", rank)
'''


def test_permutation_plan_bounds():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
    from diamond.agents import permutation_plan
    assert permutation_plan(524288, 1, 8, False) == dict(B_perm=524288, rows=65536, filter=False)
    assert permutation_plan(65536, 8, 8, False) == dict(B_perm=65536, rows=8192, filter=False)        # rank-local permutation
    for world in (2, 4, 8):
        p = permutation_plan(524288 // world, world, 8, True)
        mean = 65536 / world
        sigma = (65536 * (1 / world) * (1 - 1 / world)) ** 0.5
        assert p["B_perm"] == 524288 and p["filter"] and p["rows"] % 128 == 0
        assert mean + 6 * sigma <= p["rows"] <= mean + 6 * sigma + 16 + 128
    # tiny shards: a rank can never own more rows than it has
    assert permutation_plan(32, 2, 4, True)["rows"] <= 16


def test_speculative_permutation_worker_is_adopted_only_while_the_numpy_stream_is_untouched():
    """learn() starts the NEXT learn()'s permutation worker in the background (the permutations depend on nothing but numpy's
    global stream).  It may stand in for a fresh worker only if np.random has not moved in between; either way the permutations and
    the final stream state equal numpy's own (ppo.py:252-255)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "diamond-ppo_b200"))
    from diamond.agents import _PermWorker
    B, E, MB = 40000, 3, 4                       # > 16384: generated on a thread, not inline

    def outs():
        return [np.empty(B, dtype=np.int32) for _ in range(E)]

    np.random.seed(11)
    ref = [np.random.permutation(B) for _ in range(2 * E)]
    after = np.random.get_state(legacy=True)
    np.random.seed(11)
    o1 = outs()
    w = _PermWorker(B, E, MB, o1)
    w.start(); w.finish()                        # "learn() k": the global stream now stands where learn() k + 1 will find it
    o2 = outs()
    spec = _PermWorker(B, E, MB, o2)
    spec.start()                                 # speculative worker of learn() k + 1
    assert spec.continues(B, E, MB) and not spec.continues(B, E + 1, MB) and not spec.continues(2 * B, E, MB)
    spec.finish()
    for e in range(E):
        assert np.array_equal(o1[e], ref[e]) and np.array_equal(o2[e], ref[E + e])
    st = np.random.get_state(legacy=True)
    assert st[2] == after[2] and np.array_equal(st[1], after[1])
    # the stream moves between two learn() calls: the speculative worker must be refused
    np.random.seed(11)
    w = _PermWorker(B, E, MB, outs()); w.start(); w.finish()
    spec = _PermWorker(B, E, MB, outs()); spec.start()
    np.random.random()
    assert not spec.continues(B, E, MB)
    spec.join()


def test_dp_host_logic_gloo_world2(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(f"ROOT = {ROOT!r}\n" + GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29533", str(script)], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("ok") == 2


@pytest.mark.gpu
def test_dp_two_gpus_equal_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29534", os.path.join(ROOT, "tests", "dp_equivalence.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "OK" in r.stdout
