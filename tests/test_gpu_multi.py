"""N > 1 on real GPUs: two NCCL ranks shard trajectories / clips with sharding.shard_range, run the library on their shard and
gather the fixed-size records; every rank must hold exactly what one rank computes alone.  Skipped on a machine with one GPU;
tests/test_multi_rank.py covers the same host logic with gloo on CPU."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _records_single(dev, n):
    from oracle import uplift as oup
    from upliftingtabletennis_b200 import ops, sharding, synthetic
    from upliftingtabletennis_b200.uplift import get_model
    m = get_model('connectstage', 'large', 'dynamic', 'new').to(dev).eval()
    m.load_state_dict(oup.random_state_dict(5))
    args = [torch.from_numpy(a).to(dev) for a in synthetic.trajectories(n, seed=21)]
    return m, args, ops, sharding


def _worker(rank, world, port, n, out_dir):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    m, args, ops, sharding = _records_single(dev, n)
    a, b = sharding.shard_range(n, rank, world)
    rot, pos = m(*(x[a:b] for x in args))
    spin = ops.rotation_local(rot, pos)
    lens = args[2][a:b].sum(dim=1).long().tolist()
    recs = torch.stack([sharding.pack_record(spin[i], pos[i, :lens[i]]) for i in range(b - a)])
    table = sharding.gather_records(recs, n, world)
    np.save(os.path.join(out_dir, 'rank%d.npy' % rank), table.cpu().numpy())
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
@pytest.mark.parametrize('n', [37, 64])
def test_two_ranks_nccl_gather_equals_single_rank(tmp_path, n):
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, n, str(tmp_path)), nprocs=2, join=True)
    dev = torch.device('cuda:0')
    m, args, ops, sharding = _records_single(dev, n)
    rot, pos = m(*args)
    spin = ops.rotation_local(rot, pos)
    lens = args[2].sum(dim=1).long().tolist()
    expect = torch.stack([sharding.pack_record(spin[i], pos[i, :lens[i]]) for i in range(n)]).cpu().numpy()
    for r in range(2):
        got = np.load(os.path.join(str(tmp_path), 'rank%d.npy' % r))
        assert got.shape == (n, sharding.RECORD_FLOATS)
        # fp32 path: a trajectory's result does not depend on which other trajectories share its launch
        np.testing.assert_array_equal(got, expect)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_one_process_two_devices():
    """One process driving two GPUs: per-device kernel attributes are set on each device, every model's weights live on the device it
    first ran on, results agree bit for bit, and a handle refuses to run while another device is current."""
    from oracle import hrnet as ohr, uplift as oup, vitpose as ovp
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import WASBNet
    from upliftingtabletennis_b200.uplift import get_model
    from upliftingtabletennis_b200.vitpose import VitPose
    sd_w = ohr.random_state_dict(9, 3, seed=3)
    hp, wp = ovp.tokens_hw(64, 96)
    sd_v = ovp.random_state_dict(4, 9, hp * wp, 1)
    sd_u = oup.random_state_dict(5)
    x_w = torch.randn(2, 9, 64, 96)
    traj = [torch.from_numpy(a) for a in synthetic.trajectories(16, seed=2)]
    outs = []
    for d in (0, 1):
        dev = torch.device('cuda', d)
        with torch.cuda.device(d):
            w = WASBNet(in_frames=3, resolution=(96, 64)).to(dev).eval()
            w.load_state_dict(sd_w)
            v = VitPose(in_frames=3, resolution=(96, 64)).to(dev).eval()
            v.load_state_dict(sd_v)
            u = get_model('connectstage', 'large', 'dynamic', 'new').to(dev).eval()
            u.load_state_dict(sd_u)
            outs.append((w(x_w.to(dev))[0].cpu(), v(x_w.to(dev))[0].cpu(), u(*(t.to(dev) for t in traj))[1].cpu()))
            if d == 0:
                first = (w, x_w.to(dev))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    with torch.cuda.device(1):                      # the cuda:0 model while device 1 is current
        with pytest.raises(RuntimeError, match='device'):
            first[0](first[1])
