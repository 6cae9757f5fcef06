"""Index-sharded product sumcheck across the GPUs of one box (one process per GPU, torch.distributed
for the plumbing) - SURVEY.md section 8e.

Partitioning: LowToHigh binding pairs (2i, 2i+1) (crates/jolt-poly/src/dense.rs:236-238), so rank g
owning the CONTIGUOUS global block [g*n, (g+1)*n) keeps every pair local while its shard is longer
than one element; HighToLow pairs (i, i + half) (dense.rs:196-199), so rank g owns the STRIDED shard
global[g::G] (`shard_of` below cuts either). Per round each rank produces degree+1 partial sums (its fused bind+eval pass); they
leave the kernel as 8 x u64 lanes of 32-bit limbs, ONE integer all-reduce (ncclSum, exact) combines
them, and the carry + mod-r fold happens on the O(degree) result. No table data crosses NVLink until
the shards are tiny: at 2^GATHER_LOG entries per rank the bound shards are all-gathered once (rank
order == global order) and every rank finishes the remaining rounds redundantly with no further
communication - results are identical on every rank and identical to the single-GPU run on the same
global polynomial (the stand-in transcript depends on the round polynomials only)."""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib
from . import field as F
from .api import (BatchMember, LOW_TO_HIGH, Polynomial, ProductMember, ProvedBatch, Session, SumcheckError,
                  UnivariatePoly, _p, prove_batch_native)

GATHER_LOG = 12  # all-gather the shards once each is <= 2^12 entries (128 KiB per table per rank)


def lanes_to_ints(lanes_host: np.ndarray) -> list[int]:
    """(count, 8) u64 lanes (sums of 32-bit limbs) -> canonical field values, via the C-ABI host fold."""
    lanes_host = np.ascontiguousarray(lanes_host, dtype=np.uint64).reshape(-1, 8)
    out = np.empty((lanes_host.shape[0], 4), dtype=np.uint64)
    st = _lib.load().jb_lanes_reduce_host(_p(lanes_host), lanes_host.shape[0], _p(out))
    if st != _lib.JB_OK:
        raise RuntimeError("jb_lanes_reduce_host failed")
    return F.limbs_to_ints(out)


def elems_to_lanes(limbs: np.ndarray) -> np.ndarray:
    """(count, 4) u64 Montgomery limbs -> (count, 8) lanes of 32-bit limbs (host mirror of the kernel epilogue)."""
    a = np.ascontiguousarray(limbs, dtype=np.uint64).reshape(-1, 4)
    lo = a & np.uint64(0xFFFFFFFF)
    hi = a >> np.uint64(32)
    return np.stack([lo, hi], axis=2).reshape(-1, 8)


def splitmix_challenge(seed: int, poly: UnivariatePoly) -> int:
    """The stand-in transcript of the C++ engine (jb_absorb_round_splitmix125), called from Python so
    sharded and single-GPU runs derive identical challenges."""
    lib = _lib.load()
    coeffs = F.ints_to_limbs(poly.coefficients)
    out = np.zeros(4, dtype=np.uint64)
    s = ctypes.c_uint64(seed)
    lib.jb_absorb_round_splitmix125(ctypes.cast(ctypes.byref(s), ctypes.c_void_p), 0, _p(coeffs), coeffs.shape[0], _p(out))
    return F.from_limbs(out)


def init_comm(sess: Session, dist, p2p: bool = True) -> None:
    """Creates the context's NCCL communicator: rank 0 draws the unique id, torch.distributed (the
    rendezvous the launcher already set up) broadcasts it, every rank joins. Per-round collectives are
    then issued by the C++ side directly on the context's stream."""
    import torch
    lib = sess.lib
    buf = (ctypes.c_uint8 * 128)()
    if dist.get_rank() == 0:
        st = lib.jb_comm_unique_id(buf, None)
        if st != _lib.JB_OK:
            raise RuntimeError(f"jb_comm_unique_id failed ({st}): libnccl not loadable")
    t = torch.tensor(list(buf), dtype=torch.uint8, device="cuda")
    dist.broadcast(t, src=0)
    host = t.cpu().numpy().tobytes()
    buf = (ctypes.c_uint8 * 128).from_buffer_copy(host)
    sess.check(lib.jb_comm_init(sess.h, dist.get_world_size(), dist.get_rank(), buf, None))
    if p2p and dist.get_world_size() > 1:
        # peer-memory exchange (CUDA IPC over NVLink): the per-round all-reduce moves into the round kernel
        world = dist.get_world_size()
        mine = (ctypes.c_uint8 * 64)()
        ok = lib.jb_comm_p2p_handle(sess.h, mine) == _lib.JB_OK
        hs = torch.zeros((world, 65), dtype=torch.uint8, device="cuda")
        row = torch.tensor(list(mine) + [1 if ok else 0], dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(hs, row)
        hs = hs.cpu().numpy()
        if hs[:, 64].all():
            flat = np.ascontiguousarray(hs[:, :64]).reshape(-1)
            arr = (ctypes.c_uint8 * flat.size).from_buffer_copy(flat.tobytes())
            opened = lib.jb_comm_p2p_open(sess.h, arr) == _lib.JB_OK
        else:
            opened = False
        agree = torch.tensor([1 if opened else 0], device="cuda")
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        if not int(agree.item()):  # not available everywhere: every rank falls back to the NCCL all-reduce
            lib.jb_comm_p2p_open(sess.h, None)


def shard_of(global_table, rank: int, world: int, order: int = LOW_TO_HIGH):
    """This rank's share of a global table (any indexable with len and slicing) under the partition that
    keeps `order`'s pairs local: the contiguous block for LowToHigh, the strided slice for HighToLow."""
    n = len(global_table) // world
    return global_table[rank * n:(rank + 1) * n] if order == LOW_TO_HIGH else global_table[rank::world]


class ShardedProductMember(ProductMember):
    """ProveRounds member over this rank's shard of the global tables (jb_sharded_member_create): the
    contiguous block under LowToHigh, the strided slice under HighToLow.
    Reports log2(local) + log2(world) rounds; `previous_claim` is the global claim."""

    def __init__(self, session: Session, polys: list[Polynomial], gather_log: int = GATHER_LOG, order: int = LOW_TO_HIGH):
        self.s = session
        handles = np.array([p.handle for p in polys], dtype=np.uint64)
        h = ctypes.c_void_p()
        session.check(session.lib.jb_sharded_member_create(session.h, _p(handles), len(polys), order, gather_log,
                                                           ctypes.byref(h)))
        for p in polys:
            p.handle = 0
        self.h = h
        self.m = len(polys)


def sharded_claim(sess: Session, polys: list[Polynomial], dist) -> int:
    """sum_x prod_j f_j(x) over the GLOBAL tables: one eval-only pass per rank + one all-reduce."""
    import torch
    m = len(polys)
    probe = ProductMember(sess, [p.clone() for p in polys], LOW_TO_HIGH)
    lanes = torch.zeros((m + 1) * 8, dtype=torch.int64, device="cuda")
    sess.check(sess.lib.jb_member_prove_round_partials(probe.h, None, 0, 0, ctypes.c_void_p(lanes.data_ptr())))
    sess.synchronize()
    dist.all_reduce(lanes)
    ev = lanes_to_ints(lanes.cpu().numpy().view(np.uint64))
    probe.close()
    return (ev[0] + ev[1]) % F.R_MOD


def prove_sharded(sess: Session, polys: list[Polynomial], claim: int, seed: int, gather_log: int = GATHER_LOG,
                  raw: bool = False, order: int = LOW_TO_HIGH):
    """One index-sharded product sumcheck through the C++ engine (jb_prove_batch): no Python in the
    round loop. Returns (ProvedBatch, final_evals); identical on every rank."""
    mem = ShardedProductMember(sess, polys, gather_log, order)
    rounds = mem.num_rounds()
    res = prove_batch_native([BatchMember(claim, 1, rounds, 0)], [mem], rounds, mem.m, claim, seed=seed, raw=raw)
    fe = mem.final_evals(raw=raw)
    mem.close()
    return res, fe


def parity_self_check(sess: Session, dist, log_n: int = 14, m: int = 2, order: int = LOW_TO_HIGH, seed: int = 7) -> dict:
    """Driver-visible multi-GPU parity (the optimized tier's run_lockstep, crates/jolt-kernels/src/optimized/parity.rs:
    79-118, across ranks): an index-sharded product sumcheck over 2^log_n entries per rank against the single-GPU
    proof of the same GLOBAL polynomial on rank 0 - challenges, every round polynomial, the final claim and the
    final evaluations must be identical on every rank and equal to the single-GPU run. Collective: call on every rank."""
    import torch
    world, rank = dist.get_world_size(), dist.get_rank()
    n = 1 << log_n
    shards = []
    for j in range(m):
        g = torch.Generator(device="cuda").manual_seed(0x9A17 + 64 * rank + j)
        t = torch.randint(0, 2 ** 62, (n, 4), dtype=torch.int64, device="cuda", generator=g)
        t[:, 3] &= (1 << 60) - 1
        shards.append(t)
    clones = [t.clone() for t in shards]  # the proof binds its tables in place: work on copies (kept alive below)
    polys = [Polynomial.wrap_device(sess, c.data_ptr(), n) for c in clones]
    claim = sharded_claim(sess, polys, dist)
    res, fe = prove_sharded(sess, polys, claim, seed, order=order)
    # every rank must hold the same proof
    digest = torch.tensor([hash((tuple(res.challenges), res.final_claim, tuple(fe),
                                 tuple(tuple(p.coefficients) for p in res.round_polynomials))) & ((1 << 62) - 1)],
                          dtype=torch.int64, device="cuda")
    lo, hi = digest.clone(), digest.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    same_on_all_ranks = bool(int(lo.item()) == int(hi.item()))
    gathered = [[torch.empty_like(t) for _ in range(world)] for t in shards]
    for j, t in enumerate(shards):
        dist.all_gather(gathered[j], t)
    out = {"log_n_per_gpu": log_n, "world": world, "m": m, "order": "l2h" if order == LOW_TO_HIGH else "h2l",
           "same_on_all_ranks": same_on_all_ranks}
    if rank == 0:
        tabs = []
        for j in range(m):
            if order == LOW_TO_HIGH:
                tabs.append(torch.cat(gathered[j], dim=0).contiguous())                       # contiguous blocks
            else:
                tabs.append(torch.stack(gathered[j], dim=1).reshape(n * world, 4).contiguous())  # global[j * G + g]
        gp = [Polynomial.wrap_device(sess, t.data_ptr(), n * world) for t in tabs]
        mem = ProductMember(sess, gp, order)
        rounds = log_n + world.bit_length() - 1
        one = prove_batch_native([BatchMember(claim, 1, rounds, 0)], [mem], rounds, m, claim, seed=seed)
        one_fe = mem.final_evals()
        mem.close()
        prod = 1
        for v in fe:
            prod = prod * v % F.R_MOD
        out.update(
            challenges_equal=one.challenges == res.challenges,
            round_polynomials_equal=[p.coefficients for p in one.round_polynomials] == [p.coefficients for p in res.round_polynomials],
            final_claim_equal=one.final_claim == res.final_claim,
            final_evals_equal=one_fe == fe,
            final_claim_is_product_of_final_evals=prod == res.final_claim)
        out["identical_to_single_gpu"] = bool(out["challenges_equal"] and out["round_polynomials_equal"] and
                                              out["final_claim_equal"] and out["final_evals_equal"] and same_on_all_ranks)
    sess.synchronize()
    del clones
    return out
