"""Multi-GPU decomposition of the hot path: one process per GPU, inputs replicated, independent
units sharded, one small gather per call (SURVEY.md §8(e)).

* PreSync / DebugPreSync: contiguous offset ranges per rank.  Every frame's reduction stays on
  one GPU and the RNG is keyed by the global offset index, so the gathered curve equals the
  single-GPU curve bit for bit.
* Sync: syncpoint i goes to rank i % world; each rank advances its syncpoints side by side on its
  own device (in independent lanes); (cost, delay) pairs are gathered at the end.
* The orientation / rotation and readout searches: variant or readout k on rank k % world, RNG call
  number call_no_base + k, results gathered at the end.

The functions only need a `torch.distributed` process group (NCCL on GPUs, gloo in the CPU tests)
and a problem object with the SyncProblem methods, so the logic is testable without a GPU.
"""
from __future__ import annotations

import numpy as np


def shard_range(n, rank, world):
    """contiguous [lo, hi) slice of n units for `rank`"""
    return n * rank // world, n * (rank + 1) // world


def _gather_rows(local, sizes, group_size, device, dist):
    """ONE collective: rank r contributes sizes[r] rows of `local`'s width (the shard sizes follow
    from (n, rank, world), so they need no exchange); returns the rows of all ranks, concatenated.
    The rows are born on the host (the engine's C ABI returns host arrays), NCCL moves device
    memory: one copy each way around the collective."""
    import torch
    local = np.ascontiguousarray(local, dtype=np.float64)
    if local.ndim == 1:
        local = local.reshape(-1, 1)
    cols = local.shape[1]
    m = max(max(sizes), 1)
    buf = torch.zeros((m, cols), dtype=torch.float64, device=device)
    if local.shape[0]:
        buf[:local.shape[0]] = torch.from_numpy(local).to(device)
    out = [torch.empty((m, cols), dtype=torch.float64, device=device) for _ in range(group_size)]
    dist.all_gather(out, buf)
    return np.concatenate([out[r][:sizes[r]].cpu().numpy() for r in range(group_size)], axis=0)


def presync_grid_sharded(problem, frame_begin, frame_end, delays, *, stream=1, call_no=0, rank=0, world=1,
                         device="cpu"):
    """Loss curve of `delays` with the offsets sharded over `world` ranks; every rank returns the
    full curve."""
    delays = np.ascontiguousarray(delays, dtype=np.float64)
    lo, hi = shard_range(delays.shape[0], rank, world)
    local = problem.presync_grid(frame_begin, frame_end, delays[lo:hi], stream=stream, call_no=call_no,
                                 offset_index_base=lo)
    if world == 1:
        return np.asarray(local)
    import torch.distributed as dist
    sizes = [shard_range(delays.shape[0], r, world)[1] - shard_range(delays.shape[0], r, world)[0] for r in range(world)]
    return _gather_rows(np.asarray(local), sizes, world, device, dist)[:, 0]


def argmin_cost_delay(costs, delays):
    """std::min_element over (cost, delay) pairs, core_private.cpp:89"""
    best = 0
    for i in range(1, len(costs)):
        if costs[i] < costs[best] or (costs[i] == costs[best] and delays[i] < delays[best]):
            best = i
    return best


def presync_sharded(problem, initial_delay, frame_begin, frame_end, search_step, search_radius, delays, *,
                    call_no=0, rank=0, world=1, device="cpu"):
    """PreSync (rssync.h:19-21) over `world` ranks; `delays` is pre_sync's grid (presync_delays)."""
    curve = presync_grid_sharded(problem, frame_begin, frame_end, delays, stream=1, call_no=call_no, rank=rank,
                                 world=world, device=device)
    b = argmin_cost_delay(curve, delays)
    return float(curve[b]), float(delays[b])


def sync_sharded(problem, initial_delay, frame_begin, frame_end, search_center, search_radius, *, call_no_base=0,
                 rank=0, world=1, device="cpu"):
    """n independent Sync calls (one per syncpoint), syncpoint i on rank i % world.  Result i equals the
    i-th of n consecutive Sync calls of a single problem whose call counter starts at call_no_base."""
    ini = np.ascontiguousarray(initial_delay, dtype=np.float64)
    n = ini.shape[0]
    fb = np.ascontiguousarray(frame_begin, dtype=np.int64)
    fe = np.ascontiguousarray(frame_end, dtype=np.int64)
    cen = np.ascontiguousarray(np.broadcast_to(search_center, (n,)), dtype=np.float64)
    rad = np.ascontiguousarray(np.broadcast_to(search_radius, (n,)), dtype=np.float64)
    mine = np.arange(rank, n, world)
    if mine.size:
        cost, delay = problem.sync_batch(ini[mine], fb[mine], fe[mine], cen[mine], rad[mine],
                                         call_nos=call_no_base + mine.astype(np.uint64))
    else:
        cost, delay = np.empty(0), np.empty(0)
    if world == 1:
        return cost, delay
    import torch.distributed as dist
    both = _gather_rows(np.stack([cost, delay], axis=1), [len(range(r, n, world)) for r in range(world)], world,
                        device, dist)
    # rank r contributed syncpoints r, r+world, ...: undo the round-robin
    order = np.concatenate([np.arange(r, n, world) for r in range(world)])
    outc, outd = np.empty(n), np.empty(n)
    outc[order] = both[:, 0]
    outd[order] = both[:, 1]
    return outc, outd


def orientation_search_sharded(problem, search_fn, orientations, *, seed, call_no_base=0, rank=0, world=1,
                               device="cpu", batch_fn=None):
    """The 48-variant orientation search (core_testcode.cpp:184-233) with variant k on rank k % world.
    `search_fn(problem, [orientation])` runs one variant (integrate, ingest, PreSync) and returns
    ([cost], [delay]); the RNG call number of variant k is call_no_base + k on every rank, so the
    gathered result equals the single-process loop.  `batch_fn(problem, orientations, call_nos)`, when
    given, runs all of the rank's variants in one call with those explicit call numbers (the engine then
    prepares the variants on host threads while the device evaluates the ones that are ready).
    Every rank returns all (cost, delay) pairs."""
    n = len(orientations)
    mine = list(range(rank, n, world))
    cost, delay = np.empty(len(mine)), np.empty(len(mine))
    if batch_fn is not None and mine:
        problem.set_rng(seed, call_no_base)
        c, d = batch_fn(problem, [orientations[k] for k in mine],
                        np.array([call_no_base + k for k in mine], dtype=np.uint64))
        cost[:], delay[:] = c, d
        mine_loop = []
    else:
        mine_loop = list(enumerate(mine))
    for j, k in mine_loop:
        problem.set_rng(seed, call_no_base + k)
        c, d = search_fn(problem, [orientations[k]])
        cost[j], delay[j] = c[0], d[0]
    if world == 1:
        return cost, delay
    import torch.distributed as dist
    both = _gather_rows(np.stack([cost, delay], axis=1), [len(range(r, n, world)) for r in range(world)], world,
                        device, dist)
    order = np.concatenate([np.arange(r, n, world) for r in range(world)])
    outc, outd = np.empty(n), np.empty(n)
    outc[order] = both[:, 0]
    outd[order] = both[:, 1]
    return outc, outd


def readout_search_sharded(problem, readouts, initial_delay, frame_begin, frame_end, search_step, search_radius, *,
                           call_no_base=0, rank=0, world=1, device="cpu", curves=False):
    """The rolling-shutter readout search (problem.readout_search) with readout k on rank k % world and
    RNG call number call_no_base + k, so the gathered result equals one problem's readout_search whose
    call counter starts at call_no_base.  Every rank needs the frames' row fractions (ingested there, or
    replicate_state + replicate_row_fractions).  Every rank returns (costs, delays), plus the n x D cost
    curves when curves=True."""
    r = np.ascontiguousarray(readouts, dtype=np.float64).ravel()
    n = r.shape[0]
    mine = np.arange(rank, n, world)
    out = problem.readout_search(r[mine], initial_delay, frame_begin, frame_end, search_step, search_radius,
                                 call_nos=call_no_base + mine.astype(np.uint64), curves=curves)
    if world == 1:
        return out
    import torch.distributed as dist
    rows = np.column_stack([out[0], out[1]] + ([out[2]] if curves else []))
    both = _gather_rows(rows, [len(range(q, n, world)) for q in range(world)], world, device, dist)
    # rank q contributed readouts q, q+world, ...: undo the round-robin
    order = np.concatenate([np.arange(q, n, world) for q in range(world)])
    res = np.empty_like(both)
    res[order] = both
    return (res[:, 0], res[:, 1], res[:, 2:]) if curves else (res[:, 0], res[:, 1])


class _DevicePtr:
    """a raw device allocation as something torch can wrap (CUDA array interface, bytes)"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False),
                                         "version": 2}


def device_buffers(problem):
    """the problem's finished device state as uint8 torch tensors that ALIAS the engine's buffers
    (ray arena, orig / pos planes, spline records), plus the sizes an adopting problem needs"""
    import torch
    st = problem.device_state()
    bufs = {}
    for k in ("rays", "orig", "pos", "spline_records"):
        ptr, nbytes = st[k]
        bufs[k] = torch.as_tensor(_DevicePtr(ptr, nbytes), device="cuda") if nbytes else None
    return bufs, st


_FT_DTYPE = np.dtype([("id", "<i8"), ("off", "<i4"), ("n", "<i4"), ("ts_lo", "<f8"), ("ts_hi", "<f8")])
_last_table = {}  # id(problem) -> bytes of the frame table it holds / last sent


_side_streams = {}  # device index -> the stream the replication's collectives are issued on
_wrapped = {}       # (device index, buffer name) -> torch view of the engine's buffer (re-made when it moves)


def _merge_chunks(chunks, groups, arena=None, max_pieces=16):
    """in-flight chunks [(lo, hi), ...] (stream order) -> the pieces [(k_last, lo, hi)] to send:
    consecutive chunks go together, at most `groups` pieces, each once the last of its chunks has
    landed (k_last).  With `arena` given, the parts of [0, arena) that no chunk in flight covers come
    first, with k_last = -1: they are already on the device (an ingest that had to grow the arena has
    waited for its first chunks; frames set one by one are uploaded by the flush)."""
    n = len(chunks)
    out = []
    if arena is not None:
        at = 0
        for lo, hi in sorted(chunks):
            if lo > at:
                out.append((-1, at, lo))
            at = max(at, hi)
        if arena > at:
            out.append((-1, at, arena))
    g_n = min(groups, n)
    for g in range(g_n):
        a, b = n * g // g_n, n * (g + 1) // g_n
        out.append((b - 1, min(c[0] for c in chunks[a:b]), max(c[1] for c in chunks[a:b])))
    if len(out) > max_pieces:  # scattered updates: one piece behind the last chunk
        return [(n - 1, 0, arena)]
    return out


def replicate_state(problem, *, rank, world, device, src=0, groups=2):
    """Inputs ingested on rank `src` only: its finished device state goes to every other rank's
    problem over NVLink (NCCL broadcasts straight into the engines' own allocations -- no staging
    copy), instead of every rank validating, staging and uploading the same host data.  Afterwards
    all ranks compute identical results.

    Pipelined behind the source's ingest: a bulk SetTrackResult is still on its way to the source's
    device, chunk by chunk, when this is called; each group of chunks is broadcast as soon as it
    has landed (on a side stream, so that neither the source's nor the receivers' own stream waits
    for the whole upload), and the receivers' engines are told which arena ranges are still coming
    (expect_chunk), so the PreSync grid that follows starts on the first frames while the last are
    on the bus -- on every rank, as it does on the source.  Per call: one header, the frame table
    only when it changed since the last call, the spline records, three broadcasts per group (two
    groups: the grid, not the bus, is what the receivers wait for, and every collective costs host
    time on both sides); the only host synchronisation is the receivers' read of the header."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return
    key = id(problem)
    didx = torch.device(device).index or 0
    side = _side_streams.get(didx)
    if side is None:
        side = _side_streams[didx] = torch.cuda.Stream(device=device)
    max_groups = 16
    if rank == src:
        ft = problem.frame_table()
        raw = ft.tobytes()
        changed = _last_table.get(key) != raw
        st = problem.device_state_pipelined()
        if st["chunks"] is None:  # more chunks in flight than the call reports: wait for the ingest instead
            st = problem.device_state()
        chunks = st.get("chunks") or []
        pieces = _merge_chunks(chunks, groups, st["arena_rays"], max_groups)
        head = [ft.shape[0], st["arena_rays"], st["gyro_samples"], st["sample_rate"], st["first_timestamp"],
                1.0 if changed else 0.0, len(pieces)]
        for _, lo, hi in pieces:
            head += [lo, hi]
        head += [0.0] * (7 + 2 * max_groups - len(head))
        head = torch.tensor(head, dtype=torch.float64, device=device)
    else:
        head = torch.empty(7 + 2 * max_groups, dtype=torch.float64, device=device)
    dist.broadcast(head, src)
    if rank != src:
        h = head.cpu().tolist()
        nf, arena, nq, changed = int(h[0]), int(h[1]), int(h[2]), h[5] != 0.0
        pieces = [(None, int(h[7 + 2 * g]), int(h[8 + 2 * g])) for g in range(int(h[6]))]
    else:
        arena = st["arena_rays"]
    if changed:
        if rank == src:
            ftt = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).to(device)
        else:
            ftt = torch.empty(nf * _FT_DTYPE.itemsize, dtype=torch.uint8, device=device)
        dist.broadcast(ftt, src)
        if rank == src:
            _last_table[key] = raw
        else:
            _last_table[key] = ftt.cpu().numpy().tobytes()
    if rank != src:
        table = np.frombuffer(_last_table[key], dtype=_FT_DTYPE)
        problem.adopt_state(table, arena, nq, h[3], h[4])
        st = problem.device_state()
    bufs = {}
    for k in ("rays", "orig", "pos", "spline_records"):
        ptr, nbytes = st[k]
        t = _wrapped.get((didx, k))
        if nbytes and (t is None or t.data_ptr() != ptr or t.numel() != nbytes):
            t = _wrapped[(didx, k)] = torch.as_tensor(_DevicePtr(ptr, nbytes), device="cuda")
        bufs[k] = t if nbytes else None
    handle = side.cuda_stream
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        if rank == src:
            problem.stream_wait_chunk(-1, handle)
        if bufs["spline_records"] is not None:
            dist.broadcast(bufs["spline_records"], src)
        if rank != src:
            problem.expect_chunk(0, arena, handle)  # every frame waits at least for the records
        for k_last, lo, hi in pieces:
            if hi <= lo:
                continue
            if rank == src and k_last is not None and k_last >= 0:
                problem.stream_wait_chunk(k_last, handle)
            works = [dist.broadcast(bufs[name][lo * width:hi * width], src, async_op=True)
                     for name, width in (("rays", 64), ("orig", 4), ("pos", 4)) if bufs[name] is not None]
            if works:
                works[-1].wait()  # the side stream follows the collectives' stream (in order: the last covers all)
            if rank != src:
                problem.expect_chunk(lo, hi, handle)
        if rank == src:
            problem.note_reader(handle)  # the next Set* call waits for these sends


def replicate_row_fractions(problem, *, rank, world, device, src=0):
    """The row fractions of rank `src`'s frames (retime_table and the row-fraction plane) to every other
    rank, so that readout_search and set_readout run there too.  Call it after replicate_state, whose
    adoption drops them.  The table travels like the frame table (host bytes, one broadcast), the plane
    as one broadcast on the replication's side stream straight into the receivers' allocations, which
    are told that the plane is in flight (expect_chunk): their re-timing waits for it."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return
    rt_dtype = np.dtype([("id", "<i8"), ("frame_ts_a", "<f8"), ("frame_ts_b", "<f8")])
    if rank == src:
        raw = problem.retime_table().tobytes()
        head = torch.tensor([len(raw) // rt_dtype.itemsize], dtype=torch.int64, device=device)
    else:
        head = torch.empty(1, dtype=torch.int64, device=device)
    dist.broadcast(head, src)
    nf = int(head.item())
    if nf:
        if rank == src:
            tab = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).to(device)
        else:
            tab = torch.empty(nf * rt_dtype.itemsize, dtype=torch.uint8, device=device)
        dist.broadcast(tab, src)
    if rank != src:
        problem.adopt_row_fractions(np.frombuffer(tab.cpu().numpy().tobytes(), dtype=rt_dtype) if nf
                                    else np.empty(0, dtype=rt_dtype))
    if not nf:
        return
    ptr, nbytes = problem.row_fraction_plane()
    plane = torch.as_tensor(_DevicePtr(ptr, nbytes), device="cuda")
    didx = torch.device(device).index or 0
    side = _side_streams.get(didx)
    if side is None:
        side = _side_streams[didx] = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        dist.broadcast(plane, src, async_op=True).wait()  # the side stream follows the collective's stream
        if rank == src:
            problem.note_reader(side.cuda_stream)  # the next Set* call waits for this send
        else:
            problem.expect_chunk(0, nbytes // 16, side.cuda_stream)
