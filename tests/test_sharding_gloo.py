"""N>1 host logic on CPU: world_size-2 gloo processes shard a batch by image with no data-path
collective and agree on the max-over-ranks time (the bench contract)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import common


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, total, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    common.package()
    from dgtd_b200.twig import sharding
    lo, hi = sharding.shard_range(total, world, rank)
    # every rank regenerates only its own images (seed = global image index)
    imgs = [common.synthetic_inputs(1, 16, seed=i)[0] for i in range(lo, hi)]
    checksum = float(sum(float(t.double().sum()) for t in imgs))
    t_max = sharding.max_over_ranks(0.5 + rank, torch.device("cpu"))
    n_sum = sharding.sum_over_ranks(hi - lo, torch.device("cpu"))
    q.put((rank, lo, hi, checksum, t_max, n_sum))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_by_image():
    world, total = 2, 7
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, total, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, lo0, hi0, c0, t0, n0), (r1, lo1, hi1, c1, t1, n1) = res
    assert (lo0, hi0, lo1, hi1) == (0, 4, 4, 7)                    # disjoint cover, sizes differ by <= 1
    assert t0 == t1 == 1.5 and n0 == n1 == total                  # max / sum over ranks agree everywhere
    ref = sum(float(common.synthetic_inputs(1, 16, seed=i)[0].double().sum()) for i in range(total))
    assert abs((c0 + c1) - ref) < 1e-9                             # the union of shards is the whole batch


def test_shard_ranges_cover_without_overlap():
    common.package()
    from dgtd_b200.twig import sharding
    for total in (0, 1, 8, 13, 64):
        for world in (1, 2, 4, 8):
            spans = [sharding.shard_range(total, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = sharding.shard_sizes(total, world)
            assert max(sizes) - min(sizes) <= 1 and sum(sizes) == total


# ---- bucketed gradient all-reduce over the flat buffer (twig/buckets.py), world_size 2 on CPU ----------------
def _bucket_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    common.package()
    from dgtd_b200.twig import flat
    from dgtd_b200.twig.buckets import GradBucketer
    torch.manual_seed(0)                                         # identical replicas
    net = torch.nn.Sequential(torch.nn.Linear(7, 33), torch.nn.Tanh(), torch.nn.Linear(33, 129), torch.nn.Tanh(),
                              torch.nn.Linear(129, 5), torch.nn.Linear(5, 3))
    unused = torch.nn.Linear(4, 4)                               # never in the graph (prompt_encoder.adaptor's role)
    params = list(net.parameters()) + list(unused.parameters())
    offs, total = flat.flat_offsets(params)
    fg = torch.zeros(total)
    flat.bind_views(params, fg, "grad")
    bk = GradBucketer(params, fg, bucket_bytes=4 * 500)          # ~500-element buckets -> three buckets
    x = torch.randn(6, 7, generator=torch.Generator().manual_seed(10 + rank))      # different data per rank

    def step():
        fg.zero_()
        bk.begin()
        net(x).pow(2).mean().backward()
        bk.finish()
    step()                                                       # calibration pass: local gradients only
    local = fg.clone()
    bk.calibrate()
    step()
    order = list(bk.launch_order)
    # numpy arrays travel by value; a tensor would be shared by file descriptor from this process, which exits after
    # the barrier below -- possibly before the parent has fetched it
    q.put((rank, local.numpy(), fg.numpy().copy(), [(b["lo"], b["hi"], b["need"]) for b in bk.buckets], order, offs,
           total))
    dist.barrier()
    dist.destroy_process_group()


def test_bucketed_gradient_allreduce_two_ranks():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_bucket_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=120) for _ in range(world)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (_, l0, g0, b0, o0, offs, total), (_, l1, g1, b1, o1, _, _) = res
    l0, g0, l1, g1 = (torch.from_numpy(a) for a in (l0, g0, l1, g1))
    assert b0 == b1 and len(b0) >= 3
    # buckets tile the flat buffer from its END (reverse registration order = the order backward fills it)
    assert b0[0][1] == total and b0[-1][0] == 0 and all(a[0] == b[1] for a, b in zip(b0, b0[1:]))
    assert all(o % 32 == 0 for o in offs)                        # twig/flat.py alignment
    # every rank ends with the MEAN of the local gradients; the unused tail stays zero
    assert torch.allclose(g0, (l0 + l1) / 2, atol=1e-7) and torch.equal(g0, g1)
    assert not torch.equal(l0, l1)
    # reductions were launched bucket by bucket while backward ran: the last-registered used parameters first
    used = [i for i, b in enumerate(b0) if b[2] > 0]
    assert o0 == used == o1
