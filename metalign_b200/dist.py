"""Read-sharded multi-GPU run (SURVEY.md 8e): one process per GPU, database replicated, each rank probes
its own contiguous share of the reads, then ONE exchange step -- the sum over ranks of the per-database-k-mer
occurrence counters, each rank's counters clamped first (to ci_min, or higher: reduce_query's clamp) -- and the
per-genome table is derived from the summed counters.  Per-genome tables of shards are never summed: the >= ci_min
threshold is global and hits have set semantics.

The sum comes in two equivalent forms (NCCL over NVLink on GPUs, gloo on CPU):
  "sparse" (default)  the counter table is >99.9 % zeros, so every rank all-gathers its non-zero counters
                      (64-bit entries: index | count << 32, a few MB) and adds the other ranks' entries into
                      its own table;
  "dense"             one uint8 sum all-reduce of the whole table (|D| bytes, 0.16 GB for the default-scale
                      database) -- MLG_EXCHANGE=dense.

The read k-mers of sharded reads (reads_60mers) take another route: share_read_kmers hands every rank's device copy
of its reads to every other rank, each rank counts one share of the k-mer key order over all the reads, and
write_reads_kmc joins the ranks' KMC databases into one file.

The reference has nothing to compare with (it is a single process around subprocesses,
scripts/select_db.py:50-76); this module is the new host-side plumbing, on torch.distributed.
"""
from __future__ import annotations

import os
from typing import Tuple


class _DevMem:
    """Zero-copy view of library-owned device memory through __cuda_array_interface__."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 3,
                                         "strides": None}


def device_view_u8(ptr: int, n: int, device: int = 0):
    """torch uint8 tensor aliasing n bytes of device memory at ptr (no copy)."""
    import torch
    return torch.as_tensor(_DevMem(ptr, n), device="cuda:%d" % device)


def shard_range(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced [begin, end) share of n_items for this rank."""
    base, rem = divmod(n_items, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def max_summed_count(clamp: int, world: int) -> int:
    return clamp * world


def check_reducible(clamp: int, world: int) -> None:
    """clamp: the level each rank's counters are clamped to before the sum (the query's ci_min unless set higher)"""
    if max_summed_count(clamp, world) > 255:
        raise ValueError("exchange clamp * world_size must fit in uint8 for the counter all-reduce")


def allreduce_counts(counts, group=None):
    """In-place sum over ranks of a uint8 tensor of clamped counters (NCCL on GPU, gloo on CPU)."""
    import torch.distributed as dist
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    return counts


def device_view_i64(ptr: int, n: int, device: int = 0):
    """torch int64 tensor aliasing n 8-byte words of device memory at ptr (no copy)."""
    import torch

    class _M:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 3, "strides": None}
    return torch.as_tensor(_M(), device="cuda:%d" % device)


def allgather_sparse(entries, group=None):
    """entries: 1-D int64 tensor (CPU for gloo, CUDA for NCCL) of this rank's sparse counters.  Returns the list
    of every rank's entries (zero-padded to the longest; padding has count 0 and is ignored by the merge) and the
    true lengths."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    n_loc = torch.tensor([entries.numel()], dtype=torch.int64, device=entries.device)
    flat = entries.is_cuda          # NCCL: one flat output buffer per collective; gloo: the list form
    if flat:
        sz = torch.empty(world, dtype=torch.int64, device=entries.device)
        dist.all_gather_into_tensor(sz, n_loc, group=group)
        sizes = sz.tolist()
    else:
        szl = [torch.zeros_like(n_loc) for _ in range(world)]
        dist.all_gather(szl, n_loc, group=group)
        sizes = [int(x.item()) for x in szl]
    m = max(max(sizes), 1)
    send = torch.zeros(m, dtype=torch.int64, device=entries.device)
    send[:entries.numel()] = entries
    if flat:
        out = torch.empty(world * m, dtype=torch.int64, device=entries.device)
        dist.all_gather_into_tensor(out, send, group=group)
        recv = [out[r * m:(r + 1) * m] for r in range(world)]
    else:
        recv = [torch.empty(m, dtype=torch.int64, device=entries.device) for _ in range(world)]
        dist.all_gather(recv, send, group=group)
    return recv, sizes


EXCHANGE_MODES = ("sparse", "dense", "p2p")


def exchange_mode() -> str:
    """MLG_EXCHANGE, default "p2p" (the direct NVLink-store form; if the ranks cannot map each other's memory it falls
    back to "sparse", the NCCL all-gather of the same blocks)"""
    m = os.environ.get("MLG_EXCHANGE", "p2p")
    if m not in EXCHANGE_MODES:
        raise ValueError("MLG_EXCHANGE must be one of %s" % (EXCHANGE_MODES,))
    return m


def effective_mode(ctx, mode: str) -> str:
    """the form the exchange of this context really takes ("p2p" degrades to "sparse" when peer mapping failed)"""
    for key, cur in _EXCHANGES.items():
        if key[0] == id(ctx) and mode == "p2p" and cur.get("p2p_failed"):
            return "sparse"
    return mode


def describe_exchange(mode: str, world: int) -> str:
    """what bench.py prints in config.parallelism"""
    return {"sparse": "1 NCCL all-gather of the non-zero per-k-mer counters (fixed-size blocks, no host round trip)",
            "dense": "1 NCCL uint8 sum all-reduce of the whole per-k-mer counter table",
            "p2p": "non-zero per-k-mer counters stored straight into the peers' NVLink-mapped mailboxes by a kernel "
                   "(system-scope release/acquire flags, no NCCL call, no host round trip)"}[mode]


_EXCHANGES = {}          # (id(ctx), world, rank, mode in ('p2p', 'gather')) -> (Exchange, torch views)
_DEFAULT_CAP = 1 << 20   # entries per rank: 8 MiB blocks; grown on demand (MLG_ERR_RETRY)


def _comp_stream(ctx, device):
    import torch
    return torch.cuda.ExternalStream(ctx.streams()[0], device=device)


def _get_exchange(ctx, device: int, group, p2p: bool, cap: int = 0):
    """the persistent exchange of this context (created collectively on first use; re-created with larger blocks when
    `cap` asks for more)"""
    import torch
    import torch.distributed as dist
    from .api import Exchange
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    key = (id(ctx), world, rank)
    cur = _EXCHANGES.get(key)
    if cur is not None and cur["ex"].cap >= max(cap, 1) and (cur["connected"] or not p2p):
        return cur
    if cur is not None and cur["ex"].cap < cap:
        cur["ex"].close()
        cur = None
    if cur is None:
        ex = Exchange(ctx, world, rank, max(cap, int(os.environ.get("MLG_EXCHANGE_CAP", _DEFAULT_CAP))))
        send = device_view_i64(ex.send_ptr, ex.block_words, device)
        recv = device_view_i64(ex.recv_ptr, ex.block_words * world, device)
        cur = dict(ex=ex, send=send, recv=recv, connected=False)
        _EXCHANGES[key] = cur
    if p2p and not cur["connected"] and not cur.get("p2p_failed"):
        mine = torch.frombuffer(bytearray(cur["ex"].local_handle()), dtype=torch.uint8)
        on_gpu = dist.get_backend(group) == "nccl"
        if on_gpu:
            mine = mine.to("cuda:%d" % device)
        allh = torch.empty(64 * world, dtype=torch.uint8, device=mine.device)
        dist.all_gather_into_tensor(allh, mine, group=group)
        ok = 1
        try:
            cur["ex"].connect(bytes(allh.cpu().numpy().tobytes()))
        except Exception as e:  # noqa: BLE001  (no peer access / IPC not permitted in this container)
            ok, cur["p2p_error"] = 0, str(e)
        flag = torch.tensor([ok], dtype=torch.int32, device=mine.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)       # every rank takes the same path
        if int(flag.item()):
            cur["connected"] = True
        else:
            cur["p2p_failed"] = True
    return cur


def reduce_query(query, device: int = 0, group=None, mode: str = None, clamp: int = None) -> None:
    """The exchange step for a live GPU Query (see the module docstring).  Nothing here synchronises the host: every
    kernel and the collective are queued on the library's compute stream, and `query.finish()` is the join.  If some
    rank had more non-zero counters than the persistent blocks hold, finish() comes back asking for a repeat, and the
    closure left in `query._exchange_retry` redoes the exchange with larger blocks (collectively: every rank sees the
    same gathered counts).  clamp (ci_min .. 255, default ci_min): the level every rank's counters are clamped to before
    the sum; with counter_max (3) the intersection files of every rank have the counts of one query over all the reads."""
    import torch
    import torch.distributed as dist
    if not (dist.is_initialized() and dist.get_world_size(group) > 1):
        return
    world = dist.get_world_size(group)
    check_reducible(query_ci_min(query) if clamp is None else int(clamp), world)
    if clamp is not None:
        query.set_exchange_clamp(clamp)
    mode = mode or exchange_mode()
    ctx = query.db.ctx
    if mode == "dense":
        ptr, n = query.exchange_dense()
        with torch.cuda.stream(_comp_stream(ctx, device)):
            allreduce_counts(device_view_u8(ptr, n, device), group)
        return

    def run(cap=0):
        st = _get_exchange(ctx, device, group, mode == "p2p", cap)
        if mode == "p2p" and st["connected"]:
            query.exchange_p2p(st["ex"])
        else:
            query.exchange_pack(st["ex"])
            with torch.cuda.stream(_comp_stream(ctx, device)):
                dist.all_gather_into_tensor(st["recv"], st["send"], group=group)
            query.exchange_merge(st["ex"])

    query._exchange_retry = lambda need: run(1 << (2 * int(need) - 1).bit_length())
    run()


def _world_rank(group):
    import torch.distributed as dist
    if dist.is_initialized():
        return dist.get_world_size(group), dist.get_rank(group)
    return 1, 0


def all_ok(ok: bool, device: int = 0, group=None) -> bool:
    """Collective: every rank's ok, and-ed over the ranks (ok itself without a process group)"""
    import torch
    import torch.distributed as dist
    if _world_rank(group)[0] == 1:
        return ok
    on_gpu = dist.get_backend(group) == "nccl"
    t = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda:%d" % device if on_gpu else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    return bool(t.item())


def share_read_kmers(query, device: int = 0, group=None) -> None:
    """Collective: make this passes-mode query (Database.query(read_kmers=True, read_kmer_passes=True), every read pushed)
    rank r of a W-rank read k-mer count.  Every rank's device copy of its reads goes to every other rank -- an all-gather
    of the blob sizes, then one broadcast per source rank on the library's compute stream, each followed by the import on
    the receivers -- so that read_kmers / write_reads_kmc of rank r give share r of the key order, counted over all the
    reads.  Peak memory beside the archive: this rank's blob plus one receive buffer as large as the largest peer's blob,
    returned to the device when the exchange ends.  Reads move, not k-mers: the reads are 0.375 bytes per base, their
    distinct k-mers many times that.  A rank that fails (its blob, the receive buffer or an import) still takes part in
    every broadcast, and then every rank raises."""
    import torch
    import torch.distributed as dist
    world, rank = _world_rank(group)
    if world == 1:
        query.read_kmer_archive(0, 1)
        return
    err, ptr, nbytes = None, 0, 0
    try:
        ptr, nbytes = query.read_kmer_archive(rank, world)
    except Exception as e:  # noqa: BLE001  (every rank has to take part in the collectives below)
        err = e
    dev = "cuda:%d" % device
    n = torch.tensor([nbytes if err is None else -1], dtype=torch.int64, device=dev)
    sizes = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(sizes, n, group=group)
    sizes = sizes.tolist()
    if min(sizes) < 0:
        raise err or RuntimeError("read k-mer exchange: a rank could not pack its read archive")
    comp = _comp_stream(query.db.ctx, device)
    recv = None
    try:
        with torch.cuda.stream(comp):
            recv = torch.empty(max(sizes[r] for r in range(world) if r != rank), dtype=torch.uint8, device=dev)
    except Exception as e:  # noqa: BLE001
        err = e
    if not all_ok(err is None, device, group):
        raise err or RuntimeError("read k-mer exchange: a rank could not allocate its receive buffer")
    try:
        with torch.cuda.stream(comp):
            for src in range(world):
                buf = device_view_u8(ptr, nbytes, device) if src == rank else recv[:sizes[src]]
                dist.broadcast(buf, src=src if group is None else dist.get_global_rank(group, src), group=group)
                if src != rank and err is None:
                    try:
                        query.add_read_kmer_archive(buf.data_ptr(), sizes[src])
                    except Exception as e:  # noqa: BLE001
                        err = e
        ok = all_ok(err is None, device, group)
    finally:
        comp.synchronize()
        del recv
        torch.cuda.empty_cache()                 # budget 0 plans the passes from the free device memory
    if not ok:
        raise err or RuntimeError("read k-mer exchange: another rank could not add a peer's archive")


def write_reads_kmc(query, prefix: str, min_count: int = 2, counter_max: int = 3, device: int = 0, group=None) -> dict:
    """Collective, after share_read_kmers: <prefix>.kmc_pre / .kmc_suf of all the ranks' reads, the file a single query
    over all of them writes.  Every rank writes its share as <prefix>.part<r>, rank 0 joins the parts (api.kmc_concat),
    and the parts are removed whatever happens; if any rank fails, every rank raises and no database is left.  Rank 0
    reads every rank's part, so across nodes the prefix must be on storage every rank shares.  Returns the seconds this
    rank spent writing its part and (rank 0) joining the parts."""
    import time
    from .api import kmc_concat
    world, rank = _world_rank(group)
    parts = ["%s.part%d" % (prefix, r) for r in range(world)]
    err = None
    t0 = time.perf_counter()
    try:
        query.write_reads_kmc(parts[rank], min_count, counter_max)
    except Exception as e:  # noqa: BLE001  (every rank has to take part in the all-reduces below)
        err = e
    times = dict(part_s=time.perf_counter() - t0, concat_s=0.0)
    try:
        written = all_ok(err is None, device, group)
        if rank == 0 and written:
            t0 = time.perf_counter()
            try:
                kmc_concat(prefix, parts)
            except Exception as e:  # noqa: BLE001
                err = e
            times["concat_s"] = time.perf_counter() - t0
        joined = all_ok(err is None, device, group) and written
    finally:
        for ext in (".kmc_pre", ".kmc_suf"):
            try:
                os.remove(parts[rank] + ext)
            except FileNotFoundError:
                pass
    if err is not None:
        raise err
    if not joined:
        raise RuntimeError("the reads KMC database %s was not written: another rank failed" % prefix)
    return times


def all_gather_rows(rows, group=None) -> list:
    """Collective: every rank's list of rows (any picklable objects), joined in rank order, on every rank"""
    import torch.distributed as dist
    world, _rank = _world_rank(group)
    if world == 1:
        return list(rows)
    every = [None] * world
    dist.all_gather_object(every, list(rows), group=group)
    return [r for part in every for r in part]


def close_exchanges():
    for cur in _EXCHANGES.values():
        cur["ex"].close()
    _EXCHANGES.clear()


def query_ci_min(query) -> int:
    return getattr(query, "ci_min", 2)


def bind_to_gpu_numa(local_gpu: int) -> dict:
    """Pin this process to the CPU cores of the NUMA node its GPU hangs off, so that the pinned host buffers it
    allocates afterwards (first touch) and its copy-issuing threads are local to that GPU's PCIe root.  With 8
    ranks streaming reads from host memory, remote-node buffers halve the aggregate host->device rate.
    Best effort: returns what it did, never raises."""
    info = {"gpu": local_gpu, "numa_node": None, "cpus": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = local_gpu
        if vis:
            try:
                phys = int(vis.split(",")[local_gpu])
            except (ValueError, IndexError):
                phys = local_gpu
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:          # NVML pads the PCI domain to 8 hex digits, sysfs uses 4
            bus = bus[4:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return info
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use:
            os.sched_setaffinity(0, use)
            info.update(numa_node=node, cpus=len(use))
    except Exception as e:  # noqa: BLE001
        info["error"] = str(e)
    return info


def init_from_env(backend: str = "nccl"):
    """torchrun-style rendezvous (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend="nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world, local
