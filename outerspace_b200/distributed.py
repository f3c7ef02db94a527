"""k-sharded multi-GPU SpGEMM: host side (one process per GPU, launched by torchrun).

BASELINE.json north_star: "Across the 8 GPUs of one box the k dimension shards naturally: each GPU runs
the outer products for its k-range, then partial products are exchanged by output-row ownership with an
NCCL all-to-allv over NVLink and merged locally."  The exchange and the merge live in the CUDA library
(``osp_dist_spgemm``, outerspace_b200/csrc/osp_dist.inl); this module only

* cuts the operands into k-range shards (``k_ranges``, ``shard_operands``) -- contiguous slices of
  CSC(A) and CSR(B), balanced by the multiply work sum_k nnz(A(:,k)) * nnz(B(k,:)) (the quantity
  simulator/SimSpGEMM.cpp:884-891 calls mulflops);
* boots the library's NCCL communicator from ``torch.distributed`` (the 128-byte unique id travels as a
  broadcast tensor);
* drives the benchmark loop of ``bench.py --gpus N``.

``torch.distributed`` is plumbing here: no tensor math, no collective on the data path.
"""
from __future__ import annotations

import ctypes as C
import time
from typing import List, Tuple

import numpy as np

from . import api
from .formats import CSRMatrix, ELEM


# ------------------------------------------------------------------------------------------------
# sharding (pure numpy: also exercised by the CPU tests)
# ------------------------------------------------------------------------------------------------
def k_ranges(a_csr: CSRMatrix, b_csr: CSRMatrix, n_k: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous k-ranges [k0, k1) with balanced multiply work; covers [0, n_k) exactly."""
    nnzc = np.bincount(a_csr.data["idx"], minlength=n_k).astype(np.int64)[:n_k]
    nnzr = np.diff(b_csr.pos.astype(np.int64))
    work = nnzc * nnzr + nnzc + nnzr                       # products, plus the operand reads as a tie-breaker
    cum = np.concatenate([[0], np.cumsum(work)])
    total = int(cum[-1])
    cuts = [0]
    for r in range(1, world):
        target = total * r // world
        k = int(np.searchsorted(cum, target, side="left"))
        cuts.append(min(max(k, cuts[-1]), n_k))
    cuts.append(n_k)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def shard_operands(a_csr: CSRMatrix, b_csr: CSRMatrix, k0: int, k1: int) -> Tuple[CSRMatrix, CSRMatrix]:
    """(CSR(A[:, k0:k1]) with k ids relative to k0, CSR(B[k0:k1, :])) in the reference's layouts."""
    idx = a_csr.data["idx"]
    keep = (idx >= k0) & (idx < k1)
    rows = np.repeat(np.arange(a_csr.NRow(), dtype=np.int64), np.diff(a_csr.pos.astype(np.int64)))
    pos = np.zeros(a_csr.NRow() + 1, dtype=np.uint64)
    np.cumsum(np.bincount(rows[keep], minlength=a_csr.NRow()), out=pos[1:])
    data = a_csr.data[keep].copy()
    data["idx"] -= np.uint32(k0)
    a_g = CSRMatrix(pos, np.ascontiguousarray(data, dtype=ELEM))
    bp = b_csr.pos.astype(np.uint64)
    b_g = CSRMatrix(np.ascontiguousarray(bp[k0:k1 + 1] - bp[k0]), np.ascontiguousarray(b_csr.data[int(bp[k0]):int(bp[k1])]))
    return a_g, b_g


def row_block(rows_c: int, world: int, rank: int) -> Tuple[int, int]:
    """Owner r holds rows [rows*r/world, rows*(r+1)/world) of C (osp_dist_rows)."""
    return rows_c * rank // world, rows_c * (rank + 1) // world


# ------------------------------------------------------------------------------------------------
# engine wrapper
# ------------------------------------------------------------------------------------------------
class DistEngine:
    """One rank of the k-sharded engine (osp_dist over this process's osp_ctx)."""

    def __init__(self, engine: api.Engine, rank: int, world: int, unique_id: bytes):
        self._engine = engine
        self._lib = engine._lib
        self.rank, self.world = rank, world
        assert len(unique_id) == 128
        buf = C.create_string_buffer(unique_id, 128)
        h = C.c_void_p()
        engine._check(self._lib.osp_dist_create(engine._h, buf, rank, world, C.byref(h)))
        self._h = h

    @staticmethod
    def make_unique_id() -> bytes:
        lib = api.load_library()
        buf = C.create_string_buffer(128)
        rc = lib.osp_dist_unique_id(buf)
        if rc != api.OSP_OK:
            raise api.OspError(rc, (lib.osp_last_error(None) or b"").decode())
        return buf.raw

    @classmethod
    def from_torch(cls, engine: api.Engine) -> "DistEngine":
        """Boots the communicator inside an initialised torch.distributed process group."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        dev = torch.device("cuda", engine.device)
        t = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(cls.make_unique_id()), dtype=torch.uint8))
        dist.broadcast(t, 0)
        return cls(engine, rank, world, bytes(t.cpu().numpy().tobytes()))

    def rows(self, rows_c: int) -> Tuple[int, int]:
        b, e = C.c_uint64(), C.c_uint64()
        self._engine._check(self._lib.osp_dist_rows(self._h, rows_c, C.byref(b), C.byref(e)))
        return b.value, e.value

    def spgemm(self, a_g: CSRMatrix, b_g: CSRMatrix, rows_c: int, cols_b: int, flags: int = 0) -> api.Result:
        """Host shard operands -> this rank's row block of C (collective call)."""
        args = api.SpgemmArgs(a_g.NRow(), a_g.pos.ctypes.data, api._ptr(a_g.data), b_g.NRow(), b_g.pos.ctypes.data,
                              api._ptr(b_g.data), rows_c, cols_b, flags | api.OSP_A_IS_CSR, 0, 0, 0)
        self._keep = (a_g, b_g, args)
        h = C.c_void_p()
        self._engine._check(self._lib.osp_dist_spgemm(self._h, C.byref(args), C.byref(h)))
        return api.Result(self._engine, h)

    def spgemm_device(self, a_slices: int, a_pos_ptr: int, a_data_ptr: int, n_k: int, b_pos_ptr: int, b_data_ptr: int,
                      rows_c: int, cols_b: int, flags: int = 0, a_nnz: int = 0, b_nnz: int = 0) -> api.Result:
        args = api.SpgemmArgs(a_slices, a_pos_ptr, a_data_ptr, n_k, b_pos_ptr, b_data_ptr, rows_c, cols_b,
                              flags | api.OSP_A_IS_CSR | api.OSP_DEVICE_POINTERS, 0, a_nnz, b_nnz)
        h = C.c_void_p()
        self._engine._check(self._lib.osp_dist_spgemm(self._h, C.byref(args), C.byref(h)))
        return api.Result(self._engine, h)

    def close(self) -> None:
        if self._h is not None:
            self._lib.osp_dist_destroy(self._h)
            self._h = None


# ------------------------------------------------------------------------------------------------
# bench.py --gpus N
# ------------------------------------------------------------------------------------------------
def bench_sharded(a: CSRMatrix, b: CSRMatrix, dims: dict, args, rank: int, world: int, local_rank: int, flush_l2, sampler,
                  sampled_parity=None):
    """Strong scaling of one workload over `world` ranks.  Returns the dict bench.py prints from."""
    import torch
    import torch.distributed as dist

    dev = torch.device("cuda", local_rank)
    eng = api.Engine(local_rank)
    deng = DistEngine.from_torch(eng)
    k0, k1 = k_ranges(a, b, dims["n_k"], world)[rank]
    a_g, b_g = shard_operands(a, b, k0, k1)

    def up(x):
        return torch.from_numpy(x.view(np.uint8).reshape(-1).copy()).to(dev)
    t = [up(a_g.pos), up(a_g.data), up(b_g.pos), up(b_g.data)]
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)

    def step(flags=0):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        res = deng.spgemm_device(a_g.NRow(), t[0].data_ptr(), t[1].data_ptr(), b_g.NRow(), t[2].data_ptr(), t[3].data_ptr(),
                                 dims["rows"], dims["cols"], flags=flags, a_nnz=a_g.nnz, b_nnz=b_g.nnz)
        e1.record(stream)
        e1.synchronize()
        return res, e0.elapsed_time(e1)

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    sampler.start()                                 # sampled through warm-up and the timed steps
    for _ in range(args.warmup):
        flush_l2()
        barrier()
        res, _ = step()
        res.free()
    barrier()
    wall0 = time.perf_counter()
    ms_steps, launches, st = [], 0, None
    for _ in range(args.steps):
        flush_l2()
        barrier()                                   # every rank enters the step together
        res, ms = step()
        st = res.stats()
        launches += st["kernel_launches"]
        tm = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)   # a step takes as long as its slowest rank
        ms_steps.append(float(tm[0]))
        res.free()
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()

    kernel_rows = []
    for _ in range(3):
        flush_l2()
        barrier()
        res, _ = step(api.OSP_PROFILE_KERNELS)
        kernel_rows.append(res.kernel_times())
        res.free()

    # e2e: pinned host shards -> osp_dist_spgemm -> this rank's rows of C on the host
    def pinned_like(x):
        buf = torch.empty(max(x.nbytes, 8), dtype=torch.uint8, pin_memory=True)
        v = buf.numpy()[: x.nbytes].view(x.dtype)
        v[...] = x
        return buf, v
    keep = [pinned_like(x) for x in (a_g.pos, a_g.data, b_g.pos, b_g.data)]
    ha, hb = CSRMatrix(keep[0][1], keep[1][1]), CSRMatrix(keep[2][1], keep[3][1])
    out_pos = torch.empty((st["rows_c"] + 1) * 8, dtype=torch.uint8, pin_memory=True).numpy().view(np.uint64)
    out_dat = torch.empty(max(st["nnz_c"], 1) * 8 + 64, dtype=torch.uint8, pin_memory=True).numpy()[: max(st["nnz_c"], 1) * 8].view(ELEM)
    e2e = []
    for i in range(2 + min(args.steps, 5)):
        flush_l2()
        barrier()
        t0 = time.perf_counter()
        res = deng.spgemm(ha, hb, dims["rows"], dims["cols"])
        res.copy_into(out_pos[: res.rows + 1], out_dat[: res.nnz])
        dt = (time.perf_counter() - t0) * 1e3
        res.free()
        tm = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        if i >= 2:
            e2e.append(float(tm[0]))

    # parity, outside every timed region: sampled rows of THIS rank's block of C against the oracle, every rank's verdict gathered
    parity = None
    if sampled_parity is not None:
        flush_l2()
        barrier()
        res, _ = step()
        r0, r1 = row_block(dims["rows"], world, rank)
        par = sampled_parity(res, a, b, dims, n_rows=24, heavy=1, row_lo=r0, row_hi=r1, seed=7 + rank)
        res.free()
        pt = torch.tensor([0 if par["ok"] else 1, par["rows_checked"], par["products_checked"]], dtype=torch.int64, device=dev)
        dist.all_reduce(pt)
        parity = {"ok": int(pt[0]) == 0, "ranks_failing": int(pt[0]), "rows_checked": int(pt[1]), "products_checked": int(pt[2]),
                  "how": "every rank: seeded sample of rows of its own block + the heaviest, engine rows vs oracle rows, bit for bit"}
    barrier()

    # whole-job sums
    tot = torch.tensor([st["products"], st["nnz_c"], st["algorithmic_bytes"], st["nnz_a"], st["exchange_bytes_out"],
                        a_g.pos.nbytes + a_g.data.nbytes + b_g.pos.nbytes + b_g.data.nbytes,
                        (st["rows_c"] + 1) * 8 + st["nnz_c"] * 8], dtype=torch.int64, device=dev)
    dist.all_reduce(tot)
    tot = [int(x) for x in tot.cpu()]
    stats = dict(st)
    stats.update(products=tot[0], nnz_c=tot[1], algorithmic_bytes=tot[2], nnz_a=tot[3], rows_c=dims["rows"], n_k=dims["n_k"],
                 exchange_bytes=tot[4], ms_exchange_rank0=st["ms_exchange"])
    deng.close()
    eng.close()

    # per-kernel table of this rank (ms per step, launches per step), sorted by time
    agg, cnt = {}, {}
    for rows in kernel_rows:
        for name, ms in rows:
            agg[name] = agg.get(name, 0.0) + ms
            cnt[name] = cnt.get(name, 0) + 1
    nk = max(len(kernel_rows), 1)
    table = {k: (agg[k] / nk, cnt[k] / nk) for k in sorted(agg, key=lambda k: -agg[k])}
    # this rank's own sizes for the roofline of its dominant kernel: the merge reads what the rank OWNS
    p_owned = (st["algorithmic_bytes"] - 8 * st["products"] - 8 * st["nnz_c"] - 24 * st["nnz_a"] - 8 * st["nnz_b"]
               - 8 * (2 * st["rows_c"] + 3 * st["n_k"] + 5)) // 8
    rank_stats = dict(st)
    if next(iter(table), "").find("merge") >= 0:
        rank_stats["products"] = p_owned
    return dict(ms_per_step=sum(ms_steps) / len(ms_steps), timed_steps=len(ms_steps), wall=wall, clocks=clocks, launches=launches, stats=stats,
                kernel_table=table, rank_stats=rank_stats, parity=parity,
                e2e_ms=sum(e2e) / len(e2e), h2d=tot[5], d2h=tot[6])
