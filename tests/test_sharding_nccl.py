"""The real multi-GPU data path on hardware (needs >= 2 GPUs; skipped otherwise): one process per GPU over NCCL,
``sharding.sample_sharded`` with the REAL sampler (TargetDiffB200 on each rank's shard), ONE all-gather - against the
unsharded run of the same batch on one GPU with the same injected noise: bit-equal per graph (graphs never interact and
every kernel is batch-independent and deterministic)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from cbgbench_b200 import sharding, synthetic

pytestmark = pytest.mark.gpu
T, LAYERS = 4, 3
N_PROT, N_LIG = [120, 45, 80, 30, 64], [12, 6, 9, 4, 8]


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _model(dev):
    from cbgbench_b200.targetdiff import TargetDiffB200
    m = TargetDiffB200(synthetic.targetdiff_config(num_steps=T, num_layers=LAYERS))
    m.load_state_dict(synthetic.seeded_state_dict(m, seed=0), strict=True)
    return m.to(dev).eval()


def _final(model, sub, lig_index, pn, tu):
    """Final (x, v) of a (sub-)batch with the global noise restricted to its ligand atoms."""
    traj = model.sample(sub, pos_noise=[p[lig_index] for p in pn], type_uniform=[u[lig_index] for u in tu], traj_mode='final')
    x, c, _ = traj[0]
    dev = next(model.parameters()).device
    return x.to(dev), c.argmax(-1).to(dev)


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    try:
        torch.set_grad_enabled(False)
        batch = synthetic.make_batch(N_PROT, N_LIG, seed=5)
        pn, tu = synthetic.make_noise(T, sum(N_LIG), 13, seed=3)
        model = _model(dev)
        parts = sharding.assign_graphs(sharding.graph_sizes(batch).tolist(), world)
        mine = torch.as_tensor(parts[rank], dtype=torch.long)
        lig_index = torch.nonzero(torch.isin(batch['ligand_element_batch'], mine)).flatten()
        calls = {'n': 0}
        orig = dist.all_gather

        def counting(*a, **k):
            calls['n'] += 1
            return orig(*a, **k)

        dist.all_gather = counting
        x, v, gid = sharding.sample_sharded(lambda sub: _final(model, sub, lig_index, pn, tu), batch)
        dist.all_gather = orig
        torch.save({'x': x.cpu(), 'v': v.cpu(), 'gid': gid.cpu(), 'collectives': calls['n'], 'graphs': parts[rank]},
                   os.path.join(out_dir, f'r{rank}.pt'))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_sample_sharded_nccl_matches_unsharded(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    torch.set_grad_enabled(False)
    dev = torch.device('cuda', 0)
    batch = synthetic.make_batch(N_PROT, N_LIG, seed=5)
    pn, tu = synthetic.make_noise(T, sum(N_LIG), 13, seed=3)
    want_x, want_v = _final(_model(dev), batch, torch.arange(sum(N_LIG)), pn, tu)
    seen = set()
    for r in range(world):
        got = torch.load(os.path.join(str(tmp_path), f'r{r}.pt'))
        assert got['collectives'] == 1                                   # the single gather of final coordinates
        assert torch.equal(got['gid'], batch['ligand_element_batch'])
        assert torch.equal(got['v'], want_v.cpu())
        assert torch.equal(got['x'], want_x.cpu())                       # bit-equal: sharding changes nothing
        seen |= set(got['graphs'])
    assert seen == set(range(len(N_PROT)))
