"""Row-sharded tables (tf_repos_b200/sharded.py): routing kernels vs the numpy plan, G = 1 degenerate case
on one GPU, and (when >= 2 GPUs are visible) a 2-rank NCCL run that must reproduce the single-GPU engine on
the concatenated batch."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_bucket_kernels_match_plan(G):
    from tf_repos_b200 import dist_plan as dp
    from tf_repos_b200 import ops
    d = torch.device("cuda:0")
    rng = np.random.default_rng(G)
    ids = rng.integers(0, 50_000, size=20_000).astype(np.int32)
    uniq, inverse = np.unique(ids, return_inverse=True)
    U = len(uniq)
    n = len(ids)
    i32 = dict(dtype=torch.int32, device=d)
    counts = torch.zeros(G, **i32); cursor = torch.zeros(G, **i32)
    order = torch.empty(n, **i32); pos_of = torch.empty(n, **i32); local_ids = torch.empty(n, **i32)
    uq = torch.zeros(n, **i32); uq[:U] = torch.from_numpy(uniq).to(d)
    ops.a2a_bucket_ids(uq, torch.tensor([U], **i32), n, G, counts, cursor, order, pos_of, local_ids)
    ref_counts, ref_order, ref_local = dp.route_plan(uniq.astype(np.int64), G)
    assert counts.tolist() == ref_counts.tolist()
    o = order[:U].cpu().numpy(); p = pos_of[:U].cpu().numpy(); l = local_ids[:U].cpu().numpy()
    assert sorted(o.tolist()) == list(range(U)) and np.array_equal(p[o], np.arange(U))
    own = uniq[o] % G
    assert np.all(np.diff(own) >= 0) and np.array_equal(l.astype(np.int64) * G + own, uniq[o])
    remap = torch.empty(n, **i32)
    ops.remap_ids(torch.from_numpy(inverse.astype(np.int32)).to(d), pos_of, n, remap)
    assert np.array_equal(uniq[o][remap.cpu().numpy()], ids)
    # composite routing keys: one sort gives the same plan, deterministically
    from tf_repos_b200.ops import UniqueWorkspace
    N = 50_000
    npad = (N + G - 1) // G
    keys = torch.empty(n, **i32)
    ops.shard_keys(torch.from_numpy(ids).to(d), N, G, keys)
    assert np.array_equal(keys.cpu().numpy(), (ids % G) * npad + ids // G)
    uw = UniqueWorkspace(n, G * npad, d)
    ops.unique_segment(keys, uw)
    counts2 = torch.zeros(G, **i32); local2 = torch.empty(n, **i32)
    ops.shard_split(uw.uniq, uw.n_uniq, n, N, G, counts2, local2)
    assert uw.n_uniq.item() == U and counts2.tolist() == ref_counts.tolist()
    assert np.array_equal(local2[:U].cpu().numpy(), ref_local)                    # bucket-major, ascending id inside
    cache_ids = ref_local * G + np.repeat(np.arange(G), ref_counts)               # global id of every cache position
    assert np.array_equal(cache_ids[uw.inverse[:n].cpu().numpy()], ids)           # inverse == cache position
    W = torch.randn(50_000, device=d); out = torch.empty(n, device=d)
    ops.gather_scalar(torch.from_numpy(ids).to(d), W, out)
    assert torch.equal(out, W[torch.from_numpy(ids).long().to(d)])


@pytest.mark.parametrize("mode", ["exact", "exact_deferred", "lazy"])
def test_sharded_world1_equals_plain_engine(mode):
    from tf_repos_b200 import synth
    from tf_repos_b200.deepfm import DeepFM
    from tf_repos_b200.sharded import ShardedDeepFM
    B, N, K, F = 128, 5000, 8, 39
    kw = dict(deep_layers="32,16", dropout="1.0,1.0", l2_reg=1e-4, learning_rate=5e-4, optimizer="Adam",
              update_mode=mode, epoch_steps=3, device="cuda:0")
    a = DeepFM(F, N, K, B, **kw)
    b = ShardedDeepFM(F, N, K, B, **kw)
    g = torch.Generator().manual_seed(0)
    fv, fw = torch.randn(N, K, generator=g) * 0.1, torch.randn(N, generator=g) * 0.1
    a.load_variables({"fm_v": fv, "fm_w": fw}); b.load_global_tables(fv, fw)
    b.dense.flat.copy_(a.dense.flat)
    for step in range(5):
        ids, vals, labels = synth.criteo_batch(B, N, F, seed=step, device="cuda")
        pa = a.predict(ids, vals).clone(); pb = b.predict(ids, vals).clone()
        assert torch.allclose(pa, pb, rtol=1e-6, atol=1e-7)
        la = a.train_step(ids, vals, labels); lb = b.train_step(ids, vals, labels)
        assert torch.allclose(la[0], lb[0], rtol=1e-6)
    av = a.variables()
    bv, bw = b.gather_global_tables()
    assert torch.allclose(av["fm_v"], bv, rtol=0, atol=2e-5 * av["fm_v"].abs().max().item())
    assert torch.allclose(av["fm_w"], bw, rtol=0, atol=2e-5 * av["fm_w"].abs().max().item())
    assert torch.allclose(a.dense.flat, b.dense.flat, rtol=0, atol=2e-5)


WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from tf_repos_b200 import synth
from tf_repos_b200.deepfm import DeepFM
from tf_repos_b200.sharded import ShardedDeepFM
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=dev)
B, N, K, F = 128, 5001, 8, 39
mode = sys.argv[1]
kw = dict(deep_layers="32,16", dropout="1.0,1.0", l2_reg=1e-4, learning_rate=5e-4, optimizer="Adam", update_mode=mode,
          epoch_steps=3, device=dev)
g = torch.Generator().manual_seed(0)
fv, fw = torch.randn(N, K, generator=g) * 0.1, torch.randn(N, generator=g) * 0.1
sh = ShardedDeepFM(F, N, K, B, **kw)
sh.load_global_tables(fv, fw)
single = DeepFM(F, N, K, world * B, **kw)
single.load_variables({"fm_v": fv, "fm_w": fw})
sh.dense.flat.copy_(single.dense.flat)
for step in range(5):
    bs = [synth.criteo_batch(B, N, F, seed=10 * step + r, device=dev) for r in range(world)]
    sh.train_step(*bs[rank])
    single.train_step(torch.cat([b[0] for b in bs]), torch.cat([b[1] for b in bs]), torch.cat([b[2] for b in bs]))
bv, bw = sh.gather_global_tables()
sv = single.variables()
e1 = ((bv - sv["fm_v"]).abs().max() / sv["fm_v"].abs().max()).item()
e2 = ((bw - sv["fm_w"]).abs().max() / sv["fm_w"].abs().max()).item()
e3 = (sh.dense.flat - single.dense.flat).abs().max().item()
print("RESULT", rank, mode, e1, e2, e3, flush=True)
assert e1 < 2e-5 and e2 < 2e-5 and e3 < 2e-5
dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("mode", ["exact", "exact_deferred", "lazy"])
def test_sharded_two_ranks_equal_single_engine(tmp_path, mode):
    script = tmp_path / "w.py"
    script.write_text(WORKER % ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", str(script), mode],
                       capture_output=True, text=True, timeout=250)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("RESULT") == 2
