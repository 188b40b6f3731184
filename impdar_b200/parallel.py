"""Multi-GPU sharding of the hot path (SURVEY.md 8e): one process per GPU, torch.distributed for plumbing.

* Independent profiles (the vbp -> hfilt -> Stolt pipeline, any per-profile call) shard round-robin with no
  collective at all: ``profiles_for_rank``.
* One large Kirchhoff radargram (the serial trace loop of migrationlib/mig_python.py:35-60) shards by contiguous
  OUTPUT-trace ranges.  Every output trace needs input traces up to one aperture away: each rank gets the input
  columns of its range plus one aperture each side (halo exchange) and the finished image lands on the rank that holds
  the radargram, everything moving and computing bottom-up in row chunks.  Three transports, chosen at run time and
  identically on every rank: peer-mapped memory (csrc/peer.cu: the kernels store their blocks straight into the
  holder's image over NVLink, the holder pushes the windows with copy-engine copies, NCCL carries one-element
  signals), one all_to_all per chunk, or the round-1 scheme (full broadcast + all-gather: every rank ends with the
  whole image).  Ranges are equal on uniform trace spacing (the table kernels cost per trace) and balanced by pair
  count otherwise.
"""
import numpy as np


# Row chunks of the exchange pipeline, relative heights top to bottom.  The bottom chunk is the first window to arrive
# (nothing can start before it) and the top chunk's rows are the last to reach the image: both small; measured at 8 GPUs
# on 65536 x 8192 (profiles/r02m_exchange_variants_n8.txt): 4 equal chunks 36.3 ms, (1, 2, 2, 2, 1) 29.7, this 29.4.
DEFAULT_CHUNKS = (1, 2, 3, 3, 2, 1)
# Below this many samples the chunked pipeline loses to one chunk (every chunk costs its own table-schedule, d/dt and tile
# launches with their tails): 4096 x 16384 = 6.7e7 samples took 3.3 / 4.0 / 6.7 ms in one chunk against 4.4 / 5.2 / 7.8 ms in six
# on 8 / 4 / 2 GPUs (profiles/r02[opr]_check_sharded_n*.txt); 65536 x 8192 = 5.4e8 samples gains 7 ms from it at 8 GPUs.
CHUNKING_MIN_SAMPLES = 1 << 28


def default_chunks(snum, tnum):
    """pipeline_chunks=None: the row-chunk pattern for an image of this size."""
    return DEFAULT_CHUNKS if int(snum) * int(tnum) >= CHUNKING_MIN_SAMPLES else 1


def profiles_for_rank(n_profiles, rank, world):
    """Indices of the profiles rank `rank` owns (p mod world == rank, process.py:151-193's serial loop split)."""
    return list(range(rank, n_profiles, world))


def kirchhoff_trace_cost(travel_time_us, dist_km, vel, n_depths=32, n_traces=2048):
    """Relative work per output trace: number of in-aperture input traces summed over a subsample of depths.

    The count is a smooth (piecewise linear) function of the trace position, so for monotone trace positions it is
    evaluated at `n_traces` evenly spaced traces and interpolated: O(n_depths * n_traces * log tnum) host work,
    well under a millisecond, instead of a searchsorted over every trace per depth.  `vel`: a scalar or one RMS
    velocity per sample."""
    tt = np.asarray(travel_time_us, dtype=np.float64) / 1e6
    dist = np.asarray(dist_km, dtype=np.float64) * 1e3
    T = len(dist)
    tmax = tt.max()
    v = np.broadcast_to(np.asarray(vel, dtype=np.float64), tt.shape)
    zs = v * tt / 2.0
    idx = np.unique(np.linspace(0, len(tt) - 1, min(n_depths, len(tt))).astype(int))
    a2 = (v[idx] * tmax / 2.0) ** 2 - zs[idx] ** 2
    a = np.sqrt(a2[a2 >= 0])
    if T < 2 or not np.all(np.diff(dist) >= 0):
        return np.full(T, float(len(a) * T) + 1.0)
    pick = np.unique(np.linspace(0, T - 1, min(n_traces, T)).astype(int))
    d = dist[pick]
    hi = np.searchsorted(dist, (d[None, :] + a[:, None]).ravel(), side='right')
    lo = np.searchsorted(dist, (d[None, :] - a[:, None]).ravel(), side='left')
    cost = (hi - lo).reshape(len(a), len(pick)).sum(axis=0).astype(np.float64)
    if len(pick) == T:
        return cost + 1.0
    return np.interp(np.arange(T), pick, cost) + 1.0


_range_cache = {}


def kirchhoff_output_ranges(tnum, world, travel_time_us, dist_km, vel, align=8):
    """[(x_begin, x_end)] per rank: contiguous, covering [0, tnum).  Uniform trace spacing (the table path): equal
    trace counts; any other geometry (the general kernel, which loops over the exact aperture): balanced by pair count,
    boundaries aligned to the kernel's 8-trace CTA tile."""
    tt = np.ascontiguousarray(travel_time_us, dtype=np.float64)
    dk = np.ascontiguousarray(dist_km, dtype=np.float64)
    vkey = float(vel) if np.ndim(vel) == 0 else hash(np.ascontiguousarray(vel, dtype=np.float64).tobytes())
    key = (int(tnum), int(world), vkey, int(align), hash(tt.tobytes()), hash(dk.tobytes()))
    hit = _range_cache.get(key)
    if hit is not None:
        return list(hit)
    if _spacing_is_uniform(tt, dk, vel):
        # table / tile kernels (uniform trace spacing): every output trace walks the same table rows - traces near
        # the ends of the profile sum zero padding instead of skipping it - so the cost is per TRACE, not per pair;
        # whole 256-trace CTA tiles per rank where the ranges are wide enough for that not to unbalance them
        tile = 256 if tnum >= 8 * 256 * world else align
        bounds = [min(int(round(tnum * r / world / tile)) * tile, tnum) for r in range(world)]
        bounds = [int(b) for b in np.maximum.accumulate(bounds)]
    else:
        cost = kirchhoff_trace_cost(tt, dk, vel)
        cum = np.concatenate([[0.0], np.cumsum(cost)])
        bounds = [0]
        for r in range(1, world):
            x = int(np.searchsorted(cum, cum[-1] * r / world))
            x = int(round(x / align)) * align
            x = min(max(x, bounds[-1]), tnum)
            bounds.append(x)
    bounds.append(tnum)
    ranges = [(bounds[r], bounds[r + 1]) for r in range(world)]
    if len(_range_cache) > 64:
        _range_cache.clear()
    _range_cache[key] = tuple(ranges)
    return ranges


def kirchhoff_output_range(tnum, rank, world, travel_time_us, dist_km, vel):
    return kirchhoff_output_ranges(tnum, world, travel_time_us, dist_km, vel)[rank]


def row_chunks(snum, nchunks):
    """[(r0, r1)] of the bottom-up row pipeline, listed top-down.  `nchunks` is a count (chunk j = rows
    [snum j / n, snum (j+1) / n)) or a sequence of relative chunk heights, top to bottom (e.g. (1, 2, 2, 1): the first
    window to arrive and the last rows to ship are half-size chunks)."""
    if hasattr(nchunks, "__len__"):
        w = np.asarray(nchunks, dtype=np.float64)
        b = np.concatenate([[0.0], np.cumsum(w)]) / w.sum() * snum
        b = np.round(b).astype(int)
        b[0], b[-1] = 0, snum
        return [(int(b[j]), int(b[j + 1])) for j in range(len(w)) if b[j + 1] > b[j]]
    n = max(1, min(int(nchunks), int(snum)))
    return [(snum * j // n, snum * (j + 1) // n) for j in range(n)]


def _kirchhoff_sharded_pipelined(x, travel_time_us, dist_km, vel, nearfield, rank, world, group, src, ranges,
                                 nchunks, compute_rows):
    """The exchange steps overlapped with the diffraction sum.  An output row only reads input rows at or below it
    (minus one for the d/dt stencil), so the input is broadcast bottom-up in row chunks, every chunk of this rank's
    output range is computed as soon as its rows have arrived, and its all-gather runs while the next chunk is
    computed.  Returns the assembled (snum, tnum) image, or None when `compute_rows` reports irregular trace spacing
    on the first chunk (nothing has been computed then; the input is completely broadcast on return)."""
    import torch
    import torch.distributed as dist
    S, T = x.shape
    xb, xe = ranges[rank]
    wmax = max(e - b for b, e in ranges)
    chunks = row_chunks(S, nchunks)
    # 1. every broadcast is enqueued up front, bottom-up; the collective stream runs them back to back
    arrive = {}
    u_hi = S
    for j in reversed(range(len(chunks))):
        u0 = max(chunks[j][0] - 1, 0)
        arrive[j] = dist.broadcast(x[u0:u_hi], src=src, group=group, async_op=True) if u0 < u_hi else None
        u_hi = min(u_hi, u0)
    # 2. chunk by chunk: wait for its rows, compute, start its all-gather
    block = torch.empty((S, max(xe - xb, 0)), dtype=x.dtype, device=x.device)
    padded = torch.zeros((S, wmax), dtype=x.dtype, device=x.device)
    stages, gathers = {}, {}
    g_hi = S
    for j in reversed(range(len(chunks))):
        r0, r1 = chunks[j]
        if arrive[j] is not None:
            arrive[j].wait()                       # the compute stream waits; the host does not
        if xe > xb:
            try:
                compute_rows(x, travel_time_us, dist_km, vel, nearfield, xb, xe, r0, r1, g_hi, block)
            except ValueError:
                if g_hi != S:
                    raise
                for w in arrive.values():          # irregular spacing: finish the broadcast, let the caller fall back
                    if w is not None:
                        w.wait()
                return None
            g_hi = r0
            padded[r0:r1, :xe - xb] = block[r0:r1]
        stages[j] = torch.empty((world, r1 - r0, wmax), dtype=x.dtype, device=x.device)
        gathers[j] = dist.all_gather_into_tensor(stages[j].view(world * (r1 - r0), wmax), padded[r0:r1], group=group,
                                                 async_op=True)
    # 3. assemble: (rank, rows, wmax) stages -> column blocks of the image
    out = torch.empty((S, T), dtype=x.dtype, device=x.device)
    for j in reversed(range(len(chunks))):
        r0, r1 = chunks[j]
        gathers[j].wait()
        for r, (b, e) in enumerate(ranges):
            if e > b:
                out[r0:r1, b:e] = stages[j][r, :, :e - b]
    return out


def kirchhoff_input_windows(snum, tnum, ranges, travel_time_us, dist_km, vel, window_fn=None):
    """[(col0, col1)] per rank: the input columns each output range can read (range + one aperture each side)."""
    if window_fn is None:
        from .migrationlib import kirchhoff_input_window as window_fn
    return [window_fn(snum, travel_time_us, dist_km, vel, b, e) if e > b else (0, 0) for b, e in ranges]


def _kirchhoff_sharded_halo(x, travel_time_us, dist_km, vel, nearfield, rank, world, group, src, ranges, windows,
                            nchunks, compute_window, gather, peer=None, peer_in=None):
    """Halo exchange: rank `src` holds the radargram; every other rank receives ONLY the columns its output range can
    read (its window), bottom-up in row chunks, computes each chunk of its range as soon as the rows are there and
    ships the finished rows to `src` (gather == 'src') while the next chunk runs.  Both exchanges are one
    all_to_all_single per chunk with empty splits everywhere except from / to `src`.  Rank `src` computes straight
    from its own image into the final one.  With `peer` (a _PeerImage: rank src's persistent image mapped into every
    rank) nothing is shipped at all: the kernels of the other ranks store their blocks into src's memory over NVLink
    as they run, a one-element all_reduce per chunk tells src that the chunk's rows are complete everywhere, and src
    copies them into the image it returns on its side stream.  With `peer_in` (a _PeerWindows: every rank's window
    buffer mapped into rank src) the input windows are not packed and sent either: src pushes them as strided 2-D
    copies over NVLink, one stream per destination, and broadcasts one element per chunk as the "landed" signal.
    Returns the (snum, tnum) image on `src` (None elsewhere) for gather == 'src', or this rank's (snum, range) block
    for gather False."""
    import torch
    import torch.distributed as dist
    S, T = x.shape
    xb, xe = ranges[rank]
    c0, c1 = windows[rank]
    chunks = row_chunks(S, nchunks)
    dev, dt = x.device, x.dtype
    empty = torch.empty(0, dtype=dt, device=dev)
    is_src = rank == src
    import os
    trace = [] if (os.environ.get("IMPDAR_TRACE_SHARDED") and x.is_cuda) else None

    def mark(label, stream=None):
        if trace is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(stream) if stream is not None else ev.record()
            trace.append((label, ev))

    mark("start")
    # ---- 1. input windows, every chunk enqueued up front (the collective stream runs them back to back).  On `src` the
    # packing of the other ranks' column slabs and, later, the filing of their finished rows run on a side stream: the
    # compute stream of `src` only ever waits for the kernels of its own range.
    use_side = x.is_cuda
    side = None
    if use_side:
        main = torch.cuda.current_stream(dev)
        side = _side_stream(dev)
        side.wait_stream(main)

    def on_side():
        import contextlib
        return torch.cuda.stream(side) if use_side else contextlib.nullcontext()

    use_peer_in = peer_in is not None and peer is not None and bool(gather)
    if is_src:
        win = x[:, c0:c1]
    elif use_peer_in:
        win = peer_in.window()                     # this rank's own buffer; rank src writes it through its mapping
    else:
        win = _halo_buffer("win", (S, c1 - c0), dt, dev)
    if use_peer_in and is_src:
        lanes = _peer_streams(dev, world)
        for r in range(world):
            if r != src and windows[r][1] > windows[r][0]:
                lanes[r].wait_stream(main)
    arrive = {}
    u_hi = S
    for j in reversed(range(len(chunks))):
        u0 = max(chunks[j][0] - 1, 0)
        if u0 >= u_hi:
            arrive[j] = None
            continue
        rows = u_hi - u0
        if use_peer_in:
            landed = _halo_buffer(("landed", j), (1,), dt, dev, zero=True)
            if is_src:
                for r in range(world):
                    if r != src and windows[r][1] > windows[r][0]:
                        with torch.cuda.stream(lanes[r]):
                            peer_in.push(x, u0, u_hi, windows[r][0], windows[r][1], r)
                        side.wait_stream(lanes[r])
                mark("window %d pushed" % j, side)
                with on_side():                    # stream order: the chunk's copies are complete before the signal leaves
                    arrive[j] = dist.broadcast(landed, src=src, group=group, async_op=True)
            else:
                arrive[j] = dist.broadcast(landed, src=src, group=group, async_op=True)
        elif is_src:
            sizes = [0 if r == src else rows * (windows[r][1] - windows[r][0]) for r in range(world)]
            with on_side():
                send = _halo_buffer(("send", j), (sum(sizes),), dt, dev)
                off = 0
                for r in range(world):
                    if sizes[r]:
                        send[off:off + sizes[r]].view(rows, -1).copy_(x[u0:u_hi, windows[r][0]:windows[r][1]])
                        off += sizes[r]
                arrive[j] = dist.all_to_all_single(empty, send, [0] * world, sizes, group=group, async_op=True)
        else:
            recv = win[u0:u_hi].view(-1)
            osz = [rows * (c1 - c0) if r == src else 0 for r in range(world)]
            arrive[j] = dist.all_to_all_single(recv, empty, osz, [0] * world, group=group, async_op=True)
        u_hi = u0
    # ---- 2. chunk by chunk: wait for its rows, compute, ship the finished rows
    use_peer = peer is not None and bool(gather)
    out = torch.empty((S, T), dtype=dt, device=dev) if (is_src and gather) else None
    if out is not None:
        block = out[:, xb:xe]
    elif use_peer:
        block = peer.block(xb, xe)                 # this rank's columns of src's image, through the peer mapping
    elif gather:
        block = _halo_buffer("block", (S, max(xe - xb, 0)), dt, dev)
    else:
        block = torch.empty((S, max(xe - xb, 0)), dtype=dt, device=dev)
    ship, stages = {}, {}
    g_hi = S
    for j in reversed(range(len(chunks))):
        r0, r1 = chunks[j]
        if arrive[j] is not None and not is_src:
            arrive[j].wait()                       # the compute stream waits; the host does not (src reads its own image)
        mark("window %d here" % j)
        if xe > xb:
            compute_window(win, c0, T, travel_time_us, dist_km, vel, nearfield, xb, xe, block, (r0, r1, g_hi))
            g_hi = r0
        mark("chunk %d computed" % j)
        if use_peer:
            # stream order: this rank's kernels of chunk j (and their peer stores) are complete before it joins
            ship[j] = dist.all_reduce(_halo_buffer(("done", j), (1,), dt, dev, zero=True), group=group, async_op=True)
        elif gather:
            rows = r1 - r0
            if is_src:
                sizes = [0 if r == src else rows * (ranges[r][1] - ranges[r][0]) for r in range(world)]
                stages[j] = _halo_buffer(("stage", j), (sum(sizes),), dt, dev)
                ship[j] = dist.all_to_all_single(stages[j], empty, sizes, [0] * world, group=group, async_op=True)
            else:
                isz = [rows * (xe - xb) if r == src else 0 for r in range(world)]
                ship[j] = dist.all_to_all_single(empty, block[r0:r1].reshape(-1), [0] * world, isz, group=group,
                                                 async_op=True)
    if not gather:
        return block
    # ---- 3. rank src files the received rows into the image (side stream: overlaps the kernels of later chunks)
    with on_side():
        for j in reversed(range(len(chunks))):
            ship[j].wait()
            if is_src and use_peer:
                r0, r1 = chunks[j]
                for a, b in ((0, xb), (xe, T)):    # the other ranks' columns, either side of this rank's own
                    if b > a:
                        peer.copy_rows_to(out, r0, r1, a, b)
                mark("chunk %d filed" % j, side)
            elif is_src:
                r0, r1 = chunks[j]
                off = 0
                for r in range(world):
                    n = 0 if r == src else (r1 - r0) * (ranges[r][1] - ranges[r][0])
                    if n:
                        out[r0:r1, ranges[r][0]:ranges[r][1]] = stages[j][off:off + n].view(r1 - r0, -1)
                        off += n
        for w in arrive.values():                  # src never waited for its sends on the compute stream
            if w is not None and is_src:
                w.wait()
    if use_side:
        main.wait_stream(side)
    mark("image assembled")
    if trace is not None:
        torch.cuda.synchronize()
        print("[rank %d] " % rank + "  ".join("%s %.2f" % (lab, trace[0][1].elapsed_time(ev)) for lab, ev in trace[1:]),
              flush=True)
    return out


class _RawBlock(object):
    """A (rows, cols) float32 block at a raw device address with row stride `ld` - a region of a peer-mapped image:
    what kirchhoff_window_device needs of its `out` argument."""

    def __init__(self, address, shape, ld):
        self.address, self.shape, self.ld = int(address), tuple(shape), int(ld)

    def data_ptr(self):
        return self.address

    def stride(self, i):
        return (self.ld, 1)[i]


class _PeerImage(object):
    """One persistent (snum, tnum) float32 image in the memory of rank `src`, mapped into the address space of every
    other rank of the node (csrc/peer.cu: cudaMalloc + CUDA IPC, peer access over NVLink / NVSwitch).  The other
    ranks' diffraction-sum kernels store their output blocks straight into it while they run; rank `src` copies the
    finished rows into the image it returns (a side-stream copy per row chunk), so the caller owns its result as with
    the unsharded call.  Building one is a collective over `group` (once per image shape); `ok` is the same on every
    rank."""

    def __init__(self, S, T, rank, src, world, group, dev):
        import ctypes
        import torch
        import torch.distributed as dist
        from . import _lib
        lib = _lib.load()
        self.S, self.T, self.src, self.is_src, self.lib = S, T, src, rank == src, lib
        self.address = 0
        good = 1
        handle = torch.zeros(64, dtype=torch.uint8, device=dev)
        if self.is_src:
            h = (ctypes.c_ubyte * 64)()
            p = ctypes.c_void_p(0)
            if lib.impdar_peer_alloc(ctypes.c_size_t(S * T * 4), ctypes.byref(p), h) == 0:
                self.address = int(p.value)
                handle.copy_(torch.frombuffer(bytearray(h), dtype=torch.uint8))
            else:
                good = 0
        dist.broadcast(handle, src=src, group=group)
        if not self.is_src:
            h = (ctypes.c_ubyte * 64).from_buffer_copy(bytes(handle.cpu().numpy().tobytes()))
            p = ctypes.c_void_p(0)
            if lib.impdar_peer_open(h, ctypes.byref(p)) == 0:
                self.address = int(p.value)
            else:
                good = 0
        flag = torch.tensor([good], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        self.ok = bool(int(flag.item()))

    def block(self, xb, xe):
        """Columns [xb, xe) of the image as the `out` of kirchhoff_window_device (any rank)."""
        return _RawBlock(self.address + 4 * int(xb), (self.S, int(xe) - int(xb)), self.T)

    def copy_rows_to(self, out, r0, r1, c0, c1):
        """out[r0:r1, c0:c1] = image[r0:r1, c0:c1] on the current stream (rank src)."""
        import ctypes
        from . import _lib, device
        if r1 <= r0 or c1 <= c0:
            return
        r0, r1, c0, c1 = int(r0), int(r1), int(c0), int(c1)
        off = 4 * (r0 * self.T + c0)
        dst = int(out.data_ptr()) + out.element_size() * (r0 * int(out.stride(0)) + c0)
        _lib.check(self.lib.impdar_copy2d_f32(ctypes.c_void_p(self.address + off), self.T, ctypes.c_void_p(dst),
                                              int(out.stride(0)), r1 - r0, c1 - c0, device.current_stream_ptr()))

    def close(self):
        import ctypes
        if self.address and not self.is_src:
            self.lib.impdar_peer_close(ctypes.c_void_p(self.address))
            self.address = 0

    def free(self):
        import ctypes
        if self.address and self.is_src:
            self.lib.impdar_peer_free(ctypes.c_void_p(self.address))
            self.address = 0


class _PeerWindows(object):
    """The input side of the same idea: every rank but `src` owns one persistent (snum, window width) float32 buffer in
    cudaMalloc memory and rank `src` maps them all.  The radargram's column windows then travel as strided 2-D copies
    from src's image straight into the owners' buffers (copy engines over NVLink, one stream per destination, no
    packing pass, no SMs), a one-element broadcast per row chunk telling the owners that the chunk has landed.
    Building one is a collective over `group`; `ok` is the same on every rank."""

    def __init__(self, S, widths, rank, src, world, group, dev):
        import ctypes
        import torch
        import torch.distributed as dist
        from . import _lib
        lib = _lib.load()
        self.S, self.widths, self.rank, self.src, self.is_src, self.lib = S, [int(w) for w in widths], rank, src, rank == src, lib
        self.address = 0                  # this rank's own buffer (not on src)
        self.mapped = {}                  # on src: rank -> address of that rank's buffer in this process
        good = 1
        handle = torch.zeros(64, dtype=torch.uint8, device=dev)
        if not self.is_src and self.widths[rank] > 0:
            h = (ctypes.c_ubyte * 64)()
            p = ctypes.c_void_p(0)
            if lib.impdar_peer_alloc(ctypes.c_size_t(S * self.widths[rank] * 4), ctypes.byref(p), h) == 0:
                self.address = int(p.value)
                handle.copy_(torch.frombuffer(bytearray(h), dtype=torch.uint8))
            else:
                good = 0
        handles = torch.zeros((world, 64), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(handles, handle, group=group)
        if self.is_src:
            hh = handles.cpu().numpy()
            for r in range(world):
                if r == src or self.widths[r] <= 0 or not hh[r].any():
                    good = good if (r == src or self.widths[r] <= 0) else 0
                    continue
                h = (ctypes.c_ubyte * 64).from_buffer_copy(hh[r].tobytes())
                p = ctypes.c_void_p(0)
                if lib.impdar_peer_open(h, ctypes.byref(p)) == 0:
                    self.mapped[r] = int(p.value)
                else:
                    good = 0
        flag = torch.tensor([good], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        self.ok = bool(int(flag.item()))

    def window(self):
        """This rank's window buffer as the `win` of kirchhoff_window_device."""
        w = self.widths[self.rank]
        return _RawBlock(self.address, (self.S, w), w)

    def push(self, x, u0, u1, c0, c1, r):
        """Rows [u0, u1) of columns [c0, c1) of src's image `x` into rank r's window buffer, on the current stream."""
        import ctypes
        from . import _lib, device
        u0, u1, c0, c1 = int(u0), int(u1), int(c0), int(c1)
        w = self.widths[r]
        assert c1 - c0 == w and x.stride(1) == 1 and x.element_size() == 4
        src_addr = int(x.data_ptr()) + 4 * (u0 * int(x.stride(0)) + c0)
        _lib.check(self.lib.impdar_copy2d_f32(ctypes.c_void_p(src_addr), int(x.stride(0)),
                                              ctypes.c_void_p(self.mapped[r] + 4 * u0 * w), w, u1 - u0, w,
                                              device.current_stream_ptr()))

    def close(self):
        import ctypes
        for a in self.mapped.values():
            self.lib.impdar_peer_close(ctypes.c_void_p(a))
        self.mapped = {}

    def free(self):
        import ctypes
        if self.address:
            self.lib.impdar_peer_free(ctypes.c_void_p(self.address))
            self.address = 0


_peer_images = {}


def _peer_windows(S, T, windows, rank, src, world, group, dev):
    """The cached peer-mapped window buffers for this shape and window layout (None: unavailable / switched off with
    IMPDAR_PEER_INPUT=0; the windows then travel by all_to_all).  Same decision on every rank."""
    import os
    widths = tuple(int(b - a) for a, b in windows)
    key = ("win", S, T, widths, src, world, id(group) if group is not None else None, str(dev))
    if key not in _peer_images:
        pw = None
        if os.environ.get("IMPDAR_PEER_INPUT", "1") != "0":
            try:
                pw = _PeerWindows(S, widths, rank, src, world, group, dev)
            except (RuntimeError, OSError, AttributeError) as e:
                import warnings
                warnings.warn("impdar_b200: peer-mapped window buffers unavailable (%s); using all_to_all" % e)
                pw = None
            if pw is not None and not pw.ok:
                pw.close()
                pw.free()
                pw = None
        _peer_images[key] = pw
    return _peer_images[key]


def _peer_image(S, T, rank, src, world, group, dev):
    """The cached peer-mapped image for this shape, or None when peer mapping is switched off (IMPDAR_PEER_OUTPUT=0)
    or did not work on some rank (the halo exchange then ships the rows with all_to_all as before).  Every rank takes
    the same decision: the environment switch is reduced over the group with the mapping outcome."""
    import os
    key = (S, T, src, world, id(group) if group is not None else None, str(dev))
    if key not in _peer_images:
        if os.environ.get("IMPDAR_PEER_OUTPUT", "1") == "0":
            _peer_images[key] = None
        else:
            try:
                img = _PeerImage(S, T, rank, src, world, group, dev)
            except (RuntimeError, OSError, AttributeError) as e:      # collective state is unknown: do not retry
                import warnings
                warnings.warn("impdar_b200: peer-mapped output image unavailable (%s); using the all_to_all gather" % e)
                img = None
            if img is not None and not img.ok:
                img.close()
                img.free()
                img = None
            _peer_images[key] = img
    return _peer_images[key]


_side_streams = {}
_halo_buffers = {}
_lane_streams = {}


def _peer_streams(dev, world):
    """One copy stream per destination rank (rank src's pushes to different ranks run on different copy engines)."""
    import torch
    key = (torch.device(dev).index if torch.device(dev).index is not None else torch.cuda.current_device(), world)
    if key not in _lane_streams:
        _lane_streams[key] = [torch.cuda.Stream(device=dev) for _ in range(world)]
    return _lane_streams[key]



def _halo_buffer(key, shape, dtype, device, zero=False):
    """Persistent exchange buffers (send slabs, receive stages, input window, output block), one per role and shape:
    a step allocates nothing, so tensors that cross streams never wait for the caching allocator's cross-stream events
    (a fresh cudaMalloc per step cost ~6 ms at 8 GPUs).  Stream order makes the reuse safe: a step's side-stream and
    collective work is joined into the caller's stream before the call returns."""
    import torch
    k = (key, tuple(shape), dtype, str(device))
    t = _halo_buffers.get(k)
    if t is None:
        if len(_halo_buffers) > 256:
            _halo_buffers.clear()
        t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=device)
        _halo_buffers[k] = t
    return t


def peer_output_active():
    """True when some sharded call of this process went through a peer-mapped output image."""
    return any(isinstance(v, _PeerImage) for v in _peer_images.values())


def peer_input_active():
    """True when some sharded call of this process pushed its input windows through peer-mapped buffers."""
    return any(isinstance(v, _PeerWindows) for v in _peer_images.values())


def free_exchange_buffers():
    """Drop the persistent exchange buffers.  With peer-mapped images alive this is a collective over the default
    group (mappings are closed before the holder frees): call it on every rank at the same point."""
    _halo_buffers.clear()
    if any(v is not None for v in _peer_images.values()):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        for img in _peer_images.values():
            if img is not None:
                img.close()
        if dist.is_initialized():
            dist.barrier()
        for img in _peer_images.values():
            if img is not None:
                img.free()
    _peer_images.clear()


def _side_stream(dev):
    import torch
    key = torch.device(dev).index if torch.device(dev).index is not None else torch.cuda.current_device()
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=dev)
    return _side_streams[key]


def _spacing_is_uniform(travel_time_us, dist_km, vel):
    """The table path's own criterion (csrc/kirchhoff.cu: uniform_ok), evaluated on the host from vectors every rank
    has, so that all ranks take the same branch before any collective is issued.  A per-sample velocity enters through
    its smallest value, as in the kernel."""
    tt = np.asarray(travel_time_us, dtype=np.float64) / 1e6
    d = np.asarray(dist_km, dtype=np.float64) * 1e3
    T, S = len(d), len(tt)
    if T < 2 or S < 2 or not np.all(np.diff(d) >= 0):
        return False
    dxm = (d[-1] - d[0]) / (T - 1)
    tmax = tt.max()
    if not (dxm > 0 and tmax > 0):
        return False
    dev = np.max(np.abs(d - (d[0] + np.arange(T) * dxm)))
    dt_eff = (tt[-1] - tt[0]) / (S - 1)
    eps_t = (2.0 / float(np.min(vel))) * (2.0 * dev) + 1e-15 * (abs(tmax) + abs(tt[0]))
    return bool(eps_t / dt_eff < 1e-5)


def kirchhoff_sharded_device(x, travel_time_us, dist_km, vel, nearfield, rank=None, world=None, gather=True,
                             compute=None, group=None, src=0, pipeline_chunks=None, compute_rows=None, exchange=None,
                             compute_window=None, window_fn=None, peer_image=None):
    """Kirchhoff migration of one radargram over all ranks of the process group.

    x : (snum, tnum) float32 tensor on this rank's device; only rank `src`'s content matters.
    vel : a scalar, or one RMS velocity per sample (length snum, see migrationlib.rms_velocity).
    exchange = 'halo' (default with gather in ('src', False)): every rank receives only the input columns its output
        range can read, and the output blocks go to rank `src` only (gather='src': returns the image there, None
        elsewhere) or stay put (gather=False: returns (block, range)).  `x` is not written on the other ranks.
    exchange = 'broadcast' (default with gather=True, the round-1 scheme): the whole input is broadcast into `x` and
        the padded blocks are all-gathered, so every rank returns the full image.
    compute(x, travel_time_us, dist_km, vel, nearfield, x_begin, x_end) -> (snum, x_end-x_begin) tensor;
    defaults to the CUDA kernel (tests on CPU/gloo inject their own), likewise compute_rows (row-range entry) and
    compute_window(win, col0, tnum, tt, dist, vel, nearfield, x_begin, x_end, out, rows) (column-window entry).
    pipeline_chunks: None = by image size (default_chunks: DEFAULT_CHUNKS from 2^28 samples, one chunk below);
    > 1 (a count, or a sequence of relative chunk heights top to bottom): the exchanges and the
    kernels overlap in bottom-up row chunks (uniform trace spacing; decided on the host identically on every rank -
    irregular spacing runs the phases back to back).
    peer_image (halo exchange with gather='src'): None = automatic - float32 CUDA images computed by the default
    kernels go through a peer-mapped image (_PeerImage: the other ranks' kernels store their blocks straight into
    rank src's memory, no output collective) when the mapping works on every rank; False = off (all_to_all gather);
    or an object with block(xb, xe) / copy_rows_to(out, r0, r1, c0, c1) (tests)."""
    import torch
    import torch.distributed as dist
    default_compute = compute is None
    if compute is None:
        from .migrationlib import kirchhoff_device
        compute = kirchhoff_device
    if compute_rows is None and default_compute:
        from .migrationlib import kirchhoff_rows_device
        compute_rows = kirchhoff_rows_device
    if compute_window is None and default_compute:
        from .migrationlib import kirchhoff_window_device
        compute_window = kirchhoff_window_device
    if world is None:
        world = dist.get_world_size(group) if dist.is_initialized() else 1
    if rank is None:
        rank = dist.get_rank(group) if dist.is_initialized() else 0
    S, T = x.shape
    if pipeline_chunks is None:
        pipeline_chunks = default_chunks(S, T)
    ranges = kirchhoff_output_ranges(T, world, travel_time_us, dist_km, vel)
    xb, xe = ranges[rank]
    if exchange is None:
        exchange = 'broadcast' if gather is True else 'halo'
    if exchange not in ('halo', 'broadcast'):
        raise ValueError("exchange must be 'halo' or 'broadcast'")
    if exchange == 'halo' and gather is True:
        raise ValueError("exchange='halo' delivers the image to rank src only: pass gather='src' (or False)")
    uniform = _spacing_is_uniform(travel_time_us, dist_km, vel)
    if world > 1 and exchange == 'halo' and compute_window is not None:
        windows = kirchhoff_input_windows(S, T, ranges, travel_time_us, dist_km, vel, window_fn)
        many = hasattr(pipeline_chunks, "__len__") or pipeline_chunks > 1
        nchunks = pipeline_chunks if (uniform and many) else 1
        peer = peer_image if peer_image not in (None, False) else None
        if peer_image is None and gather and default_compute and x.is_cuda and x.dtype == torch.float32:
            peer = _peer_image(S, T, rank, src, world, group, x.device)
        peer_in = None
        if peer is not None and peer_image is None:
            peer_in = _peer_windows(S, T, windows, rank, src, world, group, x.device)
            if peer_in is not None and rank == src and x.stride(1) != 1:
                x = x.contiguous()
        res = _kirchhoff_sharded_halo(x, travel_time_us, dist_km, vel, nearfield, rank, world, group, src, ranges,
                                      windows, nchunks, compute_window, gather, peer, peer_in)
        return res if gather else (res, (xb, xe))
    broadcast_done = False
    if world > 1 and gather is True and (hasattr(pipeline_chunks, "__len__") or pipeline_chunks > 1) and \
            compute_rows is not None and uniform:
        out = _kirchhoff_sharded_pipelined(x, travel_time_us, dist_km, vel, nearfield, rank, world, group, src, ranges,
                                           pipeline_chunks, compute_rows)
        if out is not None:
            return out
        broadcast_done = True
    if world > 1 and not broadcast_done:
        dist.broadcast(x, src=src, group=group)          # the one exchange step on the input side
    block = compute(x, travel_time_us, dist_km, vel, nearfield, xb, xe) if xe > xb else \
        torch.empty((S, 0), dtype=x.dtype, device=x.device)
    if not gather:
        return block, (xb, xe)
    if world == 1:
        return block
    wmax = max(e - b for b, e in ranges)
    padded = torch.zeros((S, wmax), dtype=x.dtype, device=x.device)
    padded[:, :xe - xb] = block
    allb2 = torch.empty((world * S, wmax), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(allb2, padded, group=group)      # (S, range) blocks, concatenated along rows
    allb = allb2.view(world, S, wmax)
    out = torch.empty((S, T), dtype=x.dtype, device=x.device)
    for r, (b, e) in enumerate(ranges):
        if e > b:
            out[:, b:e] = allb[r, :, :e - b]
    return out


def kirchhoff_sharded_host(data, snum, tnum, travel_time_us, dist_km, vel, nearfield, rank=None, world=None, group=None,
                           src=0, pipeline_chunks=None):
    """Host-to-host form of the sharded migration (what a torchrun script calls with the radargram loaded on rank
    `src`): `data` is the (snum, tnum) host array on `src` (None elsewhere); returns the float64 migrated image as a
    host array on `src` (page-locked, like RadarData.migrate's result), None elsewhere."""
    import torch
    from . import device
    if rank == src:
        x = device.to_device(data)
    else:
        x = torch.empty((1, 1), dtype=torch.float32, device="cuda").expand(snum, tnum)   # shape carrier: never read
    out = kirchhoff_sharded_device(x, travel_time_us, dist_km, vel, nearfield, rank=rank, world=world, gather='src',
                                   group=group, src=src, pipeline_chunks=pipeline_chunks)
    if rank != src:
        torch.cuda.current_stream().synchronize()
        return None
    return device.to_host(out, np.float64)
