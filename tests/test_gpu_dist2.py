"""Multi-GPU checks (need N = 2, 4 or 8 GPUs on one machine; skipped with fewer): the index-sharded sumcheck over N ranks produces
exactly the single-GPU proof of the same global polynomial - both binding orders, the all-reduce inside the resident
kernel over NVLink peer memory and the NCCL path - and the term-sharded MSM equals the single-GPU MSM. Every world
size the box offers is exercised (SURVEY 8e; mirrors crates/jolt-kernels/src/optimized/parity.rs:79-118: byte-equal
round polynomials against a second implementation). Spawns its own NCCL process group."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, log_n_local, m, q, p2p=True, order=1):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import jolt_b200
    from jolt_b200 import LOW_TO_HIGH, Polynomial, ProductMember
    from jolt_b200.dist import init_comm, prove_sharded, shard_of, sharded_claim
    from oracle.coracle import rand_limbs
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sess = jolt_b200.Session(rank, cuda_stream=stream.cuda_stream)
    n = 1 << log_n_local
    glob = [rand_limbs(900 + j, n * world) for j in range(m)]
    shard = [shard_of(g, rank, world, order) for g in glob]      # contiguous block (l2h) / strided slice (h2l)
    init_comm(sess, dist, p2p=p2p)
    polys = [Polynomial.new(sess, s) for s in shard]
    claim = sharded_claim(sess, polys, dist)
    res, fe = prove_sharded(sess, polys, claim, seed=11, gather_log=6, order=order)
    # term-sharded MSM: rank g holds bases (g*n + i + 1) * G and its slice of the scalars
    from jolt_b200 import G1Bases, g1_jacobian_to_affine
    from oracle import bn254 as O
    G = np.array(O.to_mont_limbs(1, O.Q_MOD) + O.to_mont_limbs(2, O.Q_MOD), dtype=np.uint64)
    nm = 1 << 12
    allb = G1Bases.generate_multiples(sess, G, nm * world).affine()
    mine = G1Bases.from_affine(sess, allb[rank * nm:(rank + 1) * nm])
    sc = rand_limbs(4242, nm * world)
    msm_pt = g1_jacobian_to_affine(mine.msm_sharded(sc[rank * nm:(rank + 1) * nm]))
    q.put((rank, res.challenges, res.final_claim, fe, [p.coefficients for p in res.round_polynomials], msm_pt))
    dist.barrier()
    dist.destroy_process_group()


def _worlds():
    try:
        import torch
        n = torch.cuda.device_count()
    except Exception:
        n = 0
    return [w for w in (2, 4, 8) if w <= n] or [2]


@pytest.mark.parametrize("world", _worlds())
@pytest.mark.parametrize("log_n_local,m,p2p,order", [(10, 2, True, 1), (9, 3, True, 0), (10, 2, False, 1), (10, 2, False, 0),
                                                     (14, 2, True, 1), (13, 2, True, 0)])
def test_sharded_equals_single_gpu(world, log_n_local, m, p2p, order):
    """p2p=True: the per-round all-reduce runs inside the resident round kernel over NVLink peer memory;
    p2p=False: ncclAllReduce. order 1 = LowToHigh (contiguous blocks), 0 = HighToLow (strided shards).
    All must reproduce the single-GPU proof of the same global polynomial exactly."""
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    import torch.multiprocessing as mp
    import jolt_b200
    from jolt_b200 import BatchMember, LOW_TO_HIGH, Polynomial, ProductMember
    from jolt_b200 import field as F
    from oracle.coracle import rand_limbs
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, log_n_local, m, q, p2p, order)) for r in range(world)]
    for p in procs:
        p.start()
    outs = sorted([q.get(timeout=300) for _ in procs])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for o in outs[1:]:
        assert o[1:] == outs[0][1:]                     # identical on every rank
    # single GPU on the same global polynomial, same stand-in transcript
    sess = jolt_b200.Session(0)
    n = (1 << log_n_local) * world
    glob = [rand_limbs(900 + j, n) for j in range(m)]
    probe = ProductMember(sess, [Polynomial.new(sess, g) for g in glob], order)
    ev = probe.prove_round_evals(None, 0)
    claim = (ev[0] + ev[1]) % F.R_MOD
    mem = ProductMember(sess, [Polynomial.new(sess, g) for g in glob], order)
    L = log_n_local + world.bit_length() - 1
    one = jolt_b200.prove_batch_native([BatchMember(claim, 1, L, 0)], [mem], L, m, claim, seed=11)
    assert outs[0][1] == one.challenges and outs[0][2] == one.final_claim
    assert outs[0][3] == mem.final_evals()
    assert outs[0][4] == [p.coefficients for p in one.round_polynomials]
    # sharded MSM == single-GPU MSM over all terms
    from jolt_b200 import G1Bases, g1_jacobian_to_affine
    from oracle import bn254 as O
    G = np.array(O.to_mont_limbs(1, O.Q_MOD) + O.to_mont_limbs(2, O.Q_MOD), dtype=np.uint64)
    nm = 1 << 12
    full = G1Bases.generate_multiples(sess, G, nm * world)
    assert outs[0][5] == g1_jacobian_to_affine(full.msm(rand_limbs(4242, nm * world)))
