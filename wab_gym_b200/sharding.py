"""Data-parallel sharding of an environment batch over the GPUs of one box.

Environments never interact (each reference env owns all of its state, ``wab_env.py:234-238``; v2 worlds are
per-``WAB_Environment2``, ``WAB_Environment2.py:57``), so the batch is cut into contiguous blocks of global env
ids, one per rank, with NO data-path collective. The only exchange is a 64-byte all-reduce of the
episode-statistics vector, issued on a side stream every few launches (SURVEY.md §8(e)) so that the stream
the step kernels run on never waits for it. Keys of the random draws depend on the GLOBAL env id, so results
are identical for any world size.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Tuple

import torch

from .vec_env import STAT_NAMES


def shard_range(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """(first global env id, count) of `rank`'s contiguous shard; the first `total % world` ranks get one more."""
    if not (0 <= rank < world_size) or total_envs < 0:
        raise ValueError("bad shard request")
    base, extra = divmod(total_envs, world_size)
    count = base + (1 if rank < extra else 0)
    first = rank * base + min(rank, extra)
    return first, count


def population_shards(member_envs: int, world_size: int) -> List[Tuple[int, int]]:
    """Every rank's ``(first, c)`` of a data-parallel population whose members have ``member_envs`` = n envs each: rank r
    holds ids ``[first, first + c)`` of every member (``shard_range``). Raises ``ValueError`` (on every rank alike: it
    depends on n and the world size only) unless every c is a positive multiple of 128, which the population kernels
    need."""
    shards = [shard_range(int(member_envs), r, int(world_size)) for r in range(int(world_size))]
    bad = [(r, c) for r, (_, c) in enumerate(shards) if c < 128 or c % 128 != 0]
    if bad:
        raise ValueError("a data-parallel population needs each rank's share of a member's %d envs to be a positive multiple "
                         "of 128; over %d ranks rank %d would hold %d" % (int(member_envs), int(world_size), *bad[0]))
    return shards


def blocked_env_ids(rows: torch.Tensor, blocks: int, block_envs: int, block_stride: int, env_id_base: int) -> torch.Tensor:
    """The global env ids of ``rows`` (int64) on a handle of ``blocks`` blocks of ``block_envs`` rows: ``env_id_base +
    (row // block_envs) block_stride + row % block_envs`` (``VecEnv(blocks=, block_stride=)``; block_stride 0 repeats the
    ids, as replicas do; one block is the plain handle)."""
    rows = torch.as_tensor(rows, dtype=torch.int64)
    return int(env_id_base) + torch.div(rows, int(block_envs), rounding_mode="floor") * int(block_stride) + rows % int(block_envs)


def blocked_env_slots(ids: torch.Tensor, blocks: int, block_envs: int, block_stride: int, env_id_base: int) -> torch.Tensor:
    """The inverse of ``blocked_env_ids`` for unique ids (block_stride >= block_envs, or one block): the row of every id of
    ``ids``. Raises ``ValueError`` for an id the handle does not hold."""
    off = torch.as_tensor(ids, dtype=torch.int64) - int(env_id_base)
    if int(blocks) == 1:
        k, j = torch.zeros_like(off), off
    else:
        k, j = torch.div(off, int(block_stride), rounding_mode="floor"), off % int(block_stride)
    bad = (off < 0) | (k >= int(blocks)) | (j >= int(block_envs))
    if bool(bad.any()):
        first = int(off[bad][0]) + int(env_id_base)
        raise ValueError("env id %d is outside this handle's ids (%d blocks of %d from %d, %d apart)"
                         % (first, int(blocks), int(block_envs), int(env_id_base), int(block_stride)))
    return k * int(block_envs) + j


# ---- checkpoints over shards: pure functions on state dicts (VecEnv.state_dict / VecWorld2.state_dict) ------------------
# Draws are keyed by the global env id, so a record resumes bit for bit on whichever rank now holds its id.

def merge_state_dicts(sds) -> dict:
    """One state dict from the state dicts of several shards: records and ids concatenated, statistics summed."""
    sds = list(sds)
    if not sds:
        raise ValueError("nothing to merge")
    head = sds[0]
    for sd in sds[1:]:
        if sd["format"] != head["format"] or int(sd["fingerprint"]) != int(head["fingerprint"]):
            raise ValueError("state dicts of different formats or fingerprints cannot be merged")
        if sd["records"].shape[1:] != head["records"].shape[1:]:
            raise ValueError("state dicts with different record sizes cannot be merged")
    return {"format": head["format"], "fingerprint": int(head["fingerprint"]),
            "env_ids": torch.cat([torch.as_tensor(sd["env_ids"], dtype=torch.int64) for sd in sds]),
            "records": torch.cat([sd["records"] for sd in sds]),
            "stats": torch.stack([torch.as_tensor(sd["stats"], dtype=torch.int64) for sd in sds]).sum(0)}


def select_shard_records(sd: dict, env_id_base: int, num_envs: int, fingerprint: int, record_width: int,
                         state_format: int = 1) -> torch.Tensor:
    """The records of global ids ``env_id_base .. env_id_base + num_envs - 1`` in slot order (CPU). Raises ``ValueError``
    on a format or fingerprint mismatch, a record size that does not fit, and an id of the range that is missing or
    present more than once."""
    if sd.get("format") != state_format:
        raise ValueError("state format %r, expected %d" % (sd.get("format"), state_format))
    if int(sd["fingerprint"]) != int(fingerprint):
        raise ValueError("state fingerprint %#x does not match this handle (%#x): different options, seed or kernel family"
                         % (int(sd["fingerprint"]), int(fingerprint)))
    records = sd["records"]
    ids = torch.as_tensor(sd["env_ids"], dtype=torch.int64).reshape(-1)
    if records.dim() != 2 or records.shape[1] != record_width or records.shape[0] != ids.numel():
        raise ValueError("records must be [n, %d] with one env id per record" % record_width)
    sel = (ids >= env_id_base) & (ids < env_id_base + num_envs)
    local = ids[sel] - env_id_base
    counts = torch.bincount(local, minlength=num_envs)
    if bool((counts == 0).any()):
        missing = (torch.nonzero(counts == 0).reshape(-1)[:4] + env_id_base).tolist()
        raise ValueError("the state dict has no record for env id(s) %s" % missing)
    if bool((counts > 1).any()):
        dup = (torch.nonzero(counts > 1).reshape(-1)[:4] + env_id_base).tolist()
        raise ValueError("the state dict has more than one record for env id(s) %s" % dup)
    return records[sel][torch.argsort(local)]


def merge_trainer_state_dicts(sds) -> dict:
    """One trainer state dict (``A2CTrainer`` / ``PPOTrainer.state_dict``) from those of the ranks of a data-parallel run:
    the env parts merged with ``merge_state_dicts``, the shared parts (policy, Adam state, noise counter, sampling seed,
    iteration) taken once. Raises ``ValueError`` unless the shared parts are bit-equal on every rank."""
    return _merge_run_state_dicts(sds)


def merge_population_state_dicts(sds) -> dict:
    """One ``PPOPopulation.state_dict`` from those of the ranks of a data-parallel population: the env parts (each rank's
    blocked ids of every member) merged with ``merge_state_dicts``, the shared parts (every member's policy, Adam state and
    hyper-parameters, the noise counter, sampling seed and iteration) taken once. Raises ``ValueError`` unless the shared
    parts are bit-equal on every rank. The result loads into a population of any layout, a single process included."""
    return _merge_run_state_dicts(sds)


def _merge_run_state_dicts(sds) -> dict:
    sds = list(sds)
    if not sds:
        raise ValueError("nothing to merge")
    head = sds[0]
    for i, sd in enumerate(sds[1:], 1):
        if set(sd) != set(head):
            raise ValueError("trainer state dict %d has other keys than the first" % i)
        for key in head:
            if key != "env" and not _bit_equal(sd[key], head[key]):
                raise ValueError("trainer state dict %d differs from the first in %r: not one data-parallel run" % (i, key))
    out = {k: v for k, v in head.items() if k != "env"}
    out["env"] = merge_state_dicts([sd["env"] for sd in sds])
    return out


def _bit_equal(a, b) -> bool:
    if isinstance(a, torch.Tensor) or isinstance(b, torch.Tensor):
        return (isinstance(a, torch.Tensor) and isinstance(b, torch.Tensor) and a.dtype == b.dtype and a.shape == b.shape
                and torch.equal(a.cpu().view(-1).view(torch.uint8), b.cpu().view(-1).view(torch.uint8)))
    if isinstance(a, dict):
        return isinstance(b, dict) and set(a) == set(b) and all(_bit_equal(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return type(a) is type(b) and len(a) == len(b) and all(_bit_equal(x, y) for x, y in zip(a, b))
    return type(a) is type(b) and a == b


# ---- data-parallel training: the host-side arithmetic of the trainers' `group` argument ---------------------------------

def check_trainer_shards(infos) -> int:
    """``infos``: per rank in rank order, ``(env_id_base, num_envs, signature)``. Returns the total env count; raises
    ``ValueError`` unless the shards tile ``[0, total)`` contiguously in rank order and every signature (fingerprint,
    horizon, hyper-parameters, ...) equals rank 0's."""
    infos = list(infos)
    nxt = 0
    for r, (first, count, sig) in enumerate(infos):
        if int(first) != nxt or int(count) < 1:
            raise ValueError("rank %d holds envs [%d, %d), expected a non-empty shard starting at %d: the shards must tile "
                             "[0, total) contiguously in rank order" % (r, int(first), int(first) + int(count), nxt))
        nxt += int(count)
        if sig != infos[0][2]:
            raise ValueError("rank %d's trainer differs from rank 0's (%r vs %r)" % (r, sig, infos[0][2]))
    return nxt


def check_population_shards(infos, members: int) -> Tuple[int, int]:
    """``infos``: per rank in rank order, ``(env_id_base, num_envs, blocks, block_stride, signature)`` of a data-parallel
    population of ``members`` = P. Returns ``(B, n)``: the population's first id (rank 0's env_id_base) and the env count
    of each member. Raises ``ValueError`` unless every rank holds ``VecEnv(P c_r, env_id_base=B + first_r, blocks=P,
    block_stride=n)`` with the shards ``[first_r, first_r + c_r)`` tiling ``[0, n)`` in rank order, every c_r a positive
    multiple of 128, and every signature equal to rank 0's."""
    infos, P = list(infos), int(members)
    B = int(infos[0][0])
    counts = []
    for r, (base, num, blocks, stride, sig) in enumerate(infos):
        if int(num) % P != 0 or int(num) // P < 128 or (int(num) // P) % 128 != 0:
            raise ValueError("rank %d holds %d envs: a data-parallel population of %d members needs %d c envs per rank, c a "
                             "positive multiple of 128" % (r, int(num), P, P))
        if int(blocks) != P:
            raise ValueError("rank %d's VecEnv has %d blocks; a data-parallel population of %d members needs blocks=%d (one "
                             "per member)" % (r, int(blocks), P, P))
        counts.append(int(num) // P)
        if sig != infos[0][4]:
            raise ValueError("rank %d's population differs from rank 0's (%r vs %r)" % (r, sig, infos[0][4]))
    n, nxt = sum(counts), 0
    for r, (base, num, blocks, stride, sig) in enumerate(infos):
        if int(base) != B + nxt:
            raise ValueError("rank %d's shard starts at id %d, expected %d: the shards must tile [%d, %d) contiguously in "
                             "rank order" % (r, int(base), B + nxt, B, B + n))
        if P > 1 and int(stride) != n:
            raise ValueError("rank %d's VecEnv has block_stride %d; members of %d envs need block_stride=%d" % (r, int(stride), n, n))
        nxt += counts[r]
    return B, n


def minibatch_bounds(rows: int, minibatches: int):
    """Row offsets of the ``minibatches`` contiguous slices of a permutation of ``rows`` rows (``PPOTrainer``)."""
    return [k * rows // minibatches for k in range(minibatches + 1)]


def global_minibatch_counts(rows_per_rank, minibatches: int):
    """Rows of minibatch k summed over the ranks: what each rank divides minibatch k's per-row weights by."""
    out = [0] * minibatches
    for rows in rows_per_rank:
        b = minibatch_bounds(int(rows), minibatches)
        for k in range(minibatches):
            out[k] += b[k + 1] - b[k]
    return out


def rank_order_sum(t: torch.Tensor, group=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The sum of ``t`` over the ranks of ``group``, added in rank order: an all-gather, then the same additions on every
    rank, so every rank gets the same bits whatever the collective's algorithm. ``out`` [world, *t.shape] is the
    gather buffer (allocated when not given)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    if out is None:
        out = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
    dist.all_gather(list(out.unbind(0)), t.contiguous(), group=group)
    s = out[0].clone()
    for r in range(1, world):
        s += out[r]
    return s


def global_mean_std(x: torch.Tensor, group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Mean and unbiased standard deviation of ``x`` over every rank's elements (device scalars of x's dtype): fp64 sum
    and count, then the fp64 sum of squared deviations from that mean, each summed over the ranks in rank order."""
    x64 = x.detach().reshape(-1).double()
    sc = rank_order_sum(torch.stack([x64.sum(), torch.full((), float(x64.numel()), dtype=torch.float64, device=x.device)]), group)
    mean = sc[0] / sc[1]
    ss = rank_order_sum(((x64 - mean) ** 2).sum().reshape(1), group)[0]
    return mean.to(x.dtype), (ss / (sc[1] - 1.0)).sqrt().to(x.dtype)


def global_mean_std_members(x: torch.Tensor, group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """``global_mean_std`` of every member at once: x [P, ...] holds member p's elements in ``x[p]``. Returns mean and
    std [P] (x's dtype), each bit-equal to ``global_mean_std(x[p].contiguous(), group)``, with two collectives in all
    instead of 2 P: the per-member fp64 sums are formed as that call forms them, one member at a time."""
    P = x.shape[0]
    x64 = [x[p].detach().reshape(-1).double() for p in range(P)]
    sc = rank_order_sum(torch.stack([torch.stack([v.sum(), torch.full((), float(v.numel()), dtype=torch.float64, device=x.device)])
                                     for v in x64]), group)
    mean = sc[:, 0] / sc[:, 1]
    ss = rank_order_sum(torch.stack([((v - mean[p]) ** 2).sum() for p, v in enumerate(x64)]), group)
    return mean.to(x.dtype), (ss / (sc[:, 1] - 1.0)).sqrt().to(x.dtype)


def process_group(group, who: str):
    """The group a population-level object works over: ``None`` for a single process (no group, or a group of one rank),
    else ``group``. Raises ``ValueError`` for a group given without an initialised ``torch.distributed``."""
    import torch.distributed as dist
    if group is None:
        return None
    if not (dist.is_available() and dist.is_initialized()):
        raise ValueError("%s was given a group, but torch.distributed is not initialised" % who)
    return group if dist.get_world_size(group) > 1 else None


def _distributed(group=None) -> bool:
    import torch.distributed as dist
    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


def reduce_stats(local_stats: torch.Tensor, group=None) -> Dict[str, int]:
    """Blocking form: sum the int64[8] statistics vector over all ranks (NCCL on GPUs, gloo on CPU) and read it
    on the host. Synchronises the caller's stream — keep it out of any timed or latency-critical region and use
    ``AsyncStatsReducer`` there."""
    import torch.distributed as dist
    t = local_stats.clone()
    if _distributed(group):
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return dict(zip(STAT_NAMES, (int(v) for v in t.cpu())))


class AsyncStatsReducer:
    """The statistics all-reduce off the critical path.

    ``submit(fetch)`` records an event on the caller's current stream, makes a private side stream wait for it,
    runs ``fetch()`` there (it must enqueue — not synchronise — and return the int64[8] device tensor, e.g.
    ``VecEnv.stats_tensor``) and starts an asynchronous ``all_reduce`` of the result. Nothing is waited for and
    nothing is read on the host until ``result()``; the compute stream is never made to wait. On CPU tensors
    (gloo, the ``-m "not gpu"`` tests) the same calls run without streams.
    """

    def __init__(self, device: Optional[torch.device] = None, group=None):
        self.device = torch.device(device) if device is not None else None
        self.group = group
        self.cuda = self.device is not None and self.device.type == "cuda"
        self.side = torch.cuda.Stream(device=self.device) if self.cuda else None
        self._pending = None          # (tensor, work or None)
        self.submitted = 0

    def submit(self, fetch: Callable[[], torch.Tensor]) -> None:
        import torch.distributed as dist
        if self.cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            self.side.wait_event(ev)
            with torch.cuda.stream(self.side):
                t = fetch()
                work = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group, async_op=True) if _distributed(self.group) else None
        else:
            t = fetch().clone()
            work = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group, async_op=True) if _distributed(self.group) else None
        self._pending = (t, work)     # an earlier submission still in flight stays ordered before this one on the side stream
        self.submitted += 1

    def result(self) -> Optional[Dict[str, int]]:
        """Totals of the LAST submission (blocks the host until that one collective has finished)."""
        if self._pending is None:
            return None
        t, work = self._pending
        if self.cuda:
            with torch.cuda.stream(self.side):
                if work is not None:
                    work.wait()
                host = t.cpu()
        else:
            if work is not None:
                work.wait()
            host = t
        return dict(zip(STAT_NAMES, (int(v) for v in host)))


# ---- host side of the host-buffer step at N > 1: NUMA placement -----------------------------------------------------
# Every rank of `wab_vec_step_host_packed` streams ~1.5 MB per step into pinned host memory. With eight ranks on one
# box the host side decides the scaling: a rank whose threads and pinned pages sit on the other socket pushes all of its
# PCIe traffic over the socket interconnect (round-1 verdict: 0.68 of linear at 8 GPUs with every rank left on node 0).

def parse_cpulist(text: str) -> set:
    """'0-3,8,10-11' -> {0, 1, 2, 3, 8, 10, 11} (the format of sysfs cpulist files)."""
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def gpu_numa_info(pci_bus_id: str, sysfs: str = "/sys") -> Dict[str, object]:
    """NUMA node and local CPUs of a PCI device ('0000:1b:00.0'), from sysfs; node -1 when the platform has none."""
    import os
    base = os.path.join(sysfs, "bus", "pci", "devices", pci_bus_id.lower())
    info: Dict[str, object] = {"pci_bus_id": pci_bus_id.lower(), "numa_node": -1, "local_cpus": set()}
    try:
        with open(os.path.join(base, "numa_node")) as fh:
            info["numa_node"] = int(fh.read().strip())
        with open(os.path.join(base, "local_cpulist")) as fh:
            info["local_cpus"] = parse_cpulist(fh.read())
    except (OSError, ValueError):
        pass
    return info


def _set_mempolicy_preferred(node: int) -> bool:
    """set_mempolicy(MPOL_PREFERRED, {node}): pages this process touches from now on (pinned buffers included) come from
    `node` when it has room. Raw syscall (no libnuma in the image); False when the kernel refuses."""
    import ctypes
    import platform
    nr = {"x86_64": 238, "aarch64": 237}.get(platform.machine())
    if nr is None or node < 0 or node >= 1024:
        return False
    libc = ctypes.CDLL(None, use_errno=True)
    mask = (ctypes.c_ulong * 16)()                       # 1024 node bits
    mask[node // 64] = 1 << (node % 64)
    MPOL_PREFERRED = 1
    return libc.syscall(ctypes.c_long(nr), ctypes.c_int(MPOL_PREFERRED), mask, ctypes.c_ulong(1024 + 1)) == 0


def bind_to_gpu_numa(device_index: int, pci_bus_id: Optional[str] = None, sysfs: str = "/sys") -> Dict[str, object]:
    """Move this process next to its GPU: CPU affinity = the GPU's local CPUs (those this process is allowed to use),
    memory policy = prefer the GPU's NUMA node. Call it before allocating pinned host buffers. Returns what was done
    (for the benchmark record); a platform without NUMA information is left alone."""
    import os
    if pci_bus_id is None:
        p = torch.cuda.get_device_properties(device_index)
        pci_bus_id = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
    info = gpu_numa_info(pci_bus_id, sysfs)
    allowed = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else set()
    local = set(info["local_cpus"]) & set(allowed)
    out = {"pci_bus_id": info["pci_bus_id"], "numa_node": info["numa_node"], "cpus_before": len(allowed),
           "cpus_after": len(allowed), "cpu_bound": False, "mem_bound": False}
    if local and local != set(allowed):
        try:
            os.sched_setaffinity(0, local)
            out["cpu_bound"], out["cpus_after"] = True, len(local)
        except OSError:
            pass
    if int(info["numa_node"]) >= 0:
        out["mem_bound"] = _set_mempolicy_preferred(int(info["numa_node"]))
    return out
