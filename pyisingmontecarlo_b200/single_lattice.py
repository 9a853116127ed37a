"""One large 2D Ising lattice domain-decomposed in row strips (BASELINE config 5).

The reference cannot express this workload (one experiment = one rayon task, lattice.rs:197-212,
and a 65536^2 edge list would need 206 GB); it is the "one lattice too big for one thread"
analogue of SURVEY.md 5.7.  Spins are bit-packed along x, every rank owns a block of rows, and
per colour phase one boundary row (Lx/64 words, 8 KiB at Lx = 65536) goes to each neighbour:
NCCL send/recv over NVLink between GPUs (gloo in the CPU tests), a device copy when one strip
holds the whole lattice.
"""
import numpy as np

from . import _native as nat
from .tempering import shard_range


def exchange_halos(strip, colour, rank, world, dist=None, group=None, device=None):
    """Boundary rows of `colour` -> the neighbouring strips' ghost rows (periodic ring).

    strip: .get_boundary(colour, which, dst), .set_ghost(colour, which, src), .wrap_local(colour),
    .words.  With world == 1 the strip wraps onto itself."""
    if world == 1:
        strip.wrap_local(colour)
        return
    import torch

    up, down = (rank - 1) % world, (rank + 1) % world
    on_gpu = device is not None and device.type == "cuda"
    kw = dict(dtype=torch.int32, device=device if on_gpu else "cpu")
    send_top, send_bot = torch.empty(strip.words, **kw), torch.empty(strip.words, **kw)
    recv_top, recv_bot = torch.empty(strip.words, **kw), torch.empty(strip.words, **kw)
    if on_gpu:
        strip.get_boundary(colour, 0, send_top.data_ptr())
        strip.get_boundary(colour, 1, send_bot.data_ptr())
    else:
        send_top.copy_(torch.from_numpy(strip.get_boundary(colour, 0).view(np.int32)))
        send_bot.copy_(torch.from_numpy(strip.get_boundary(colour, 1).view(np.int32)))
    if world == 2:
        # both neighbours are the same peer: order the four messages explicitly
        ops = [dist.P2POp(dist.isend, send_top, up, group=group, tag=0),
               dist.P2POp(dist.isend, send_bot, down, group=group, tag=1),
               dist.P2POp(dist.irecv, recv_bot, down, group=group, tag=0),   # peer's top row
               dist.P2POp(dist.irecv, recv_top, up, group=group, tag=1)]     # peer's bottom row
    else:
        ops = [dist.P2POp(dist.isend, send_top, up, group=group),
               dist.P2POp(dist.isend, send_bot, down, group=group),
               dist.P2POp(dist.irecv, recv_top, up, group=group),
               dist.P2POp(dist.irecv, recv_bot, down, group=group)]
    for req in dist.batch_isend_irecv(ops):
        req.wait()
    if on_gpu:
        torch.cuda.synchronize(device)
        strip.set_ghost(colour, 0, recv_top.data_ptr())
        strip.set_ghost(colour, 1, recv_bot.data_ptr())
    else:
        strip.set_ghost(colour, 0, recv_top.numpy().view(np.uint32))
        strip.set_ghost(colour, 1, recv_bot.numpy().view(np.uint32))


def exchange_deep(strip, depth, rank, world, dist=None, group=None, device=None, bufs=None):
    """The first / last `depth` rows of BOTH colours -> the neighbouring strips' ghost rows, in
    one message per neighbour.  After it a strip can run depth // 2 sweeps on its own
    (Strip.phase_ext), so the per-message latency is paid once per batch instead of per phase.

    strip: .halo_deep(direction, depth, buf[, sync]), .wrap_deep(depth), .words.  bufs: optional
    (send, recv) int32 device tensors of >= 4 * depth * words elements (enqueue-only path)."""
    if world == 1:
        strip.wrap_deep(depth)
        return
    import torch

    up, down = (rank - 1) % world, (rank + 1) % world
    n = 4 * depth * strip.words
    half = n // 2
    on_gpu = bufs is not None
    if on_gpu:
        send, recv = bufs[0][:n], bufs[1][:n]
        strip.halo_deep(0, depth, send.data_ptr(), sync=False)
    else:
        host = np.empty(n, dtype=np.uint32)
        strip.halo_deep(0, depth, host)
        send = torch.from_numpy(host.view(np.int32))
        recv = torch.empty(n, dtype=torch.int32)
    if world == 2:   # both neighbours are the same peer: match the messages by order / tag
        ops = [dist.P2POp(dist.isend, send[:half], up, group=group, tag=0),
               dist.P2POp(dist.isend, send[half:], down, group=group, tag=1),
               dist.P2POp(dist.irecv, recv[half:], down, group=group, tag=0),   # peer's first rows
               dist.P2POp(dist.irecv, recv[:half], up, group=group, tag=1)]     # peer's last rows
    else:
        ops = [dist.P2POp(dist.isend, send[:half], up, group=group),
               dist.P2POp(dist.isend, send[half:], down, group=group),
               dist.P2POp(dist.irecv, recv[:half], up, group=group),
               dist.P2POp(dist.irecv, recv[half:], down, group=group)]
    for req in dist.batch_isend_irecv(ops):
        req.wait()                      # NCCL: a stream-side wait, the host does not block
    if on_gpu:
        strip.halo_deep(1, depth, recv.data_ptr(), sync=False)
    else:
        strip.halo_deep(1, depth, np.ascontiguousarray(recv.numpy()).view(np.uint32))


def sweep_batches(strip, betas, k, rank, world, dist=None, group=None, device=None, bufs=None, sync=True,
                  fields=None):
    """One checkerboard sweep per beta in batches of at most k sweeps: one deep exchange of 2 nb
    rows, then 2 nb colour phases that update 2 nb - 1 - q ghost rows next to the local ones
    (phase q), so that the valid ghost region shrinks by one row per phase and is used up
    exactly when the batch ends.  strip needs .phase_ext and the interface of exchange_deep.
    fields: one field h per beta (strip.set_field before the first sweep and wherever h changes),
    None = the strip's field."""
    betas = np.atleast_1d(np.asarray(betas, dtype=np.float64))
    cur = None
    i = 0
    while i < len(betas):
        nb = min(int(k), len(betas) - i)          # sweeps in this batch
        exchange_deep(strip, 2 * nb, rank, world, dist, group, device, bufs)
        for q in range(2 * nb):
            if fields is not None and fields[i + q // 2] != cur:
                cur = fields[i + q // 2]
                strip.set_field(cur)
            strip.phase_ext(q & 1, betas[i + q // 2], 2 * nb - 1 - q, advance=bool(q & 1), sync=sync)
        i += nb


def _finite_field(h):
    h = float(h)
    if not np.isfinite(h):
        raise ValueError(f"field must be finite, got {h}")
    return h


class SingleLattice2D:
    """Periodic Lx x Ly lattice with uniform coupling j (j < 0 ferromagnetic, README.md:45-46) in a
    uniform longitudinal field h (E = sum J s s' - h sum s, s = +1 for an up spin)."""

    def __init__(self, Lx, Ly=None, j=-1.0, seed=0, *, device=None, process_group=None, planes=0, rounds=0,
                 exchange_every=8, field=0.0):
        """exchange_every = k > 0: strips exchange 2k boundary rows once per k sweeps and update
        the ghost rows redundantly in between (same bits, 1/(2k) of the messages);
        exchange_every = 0: one boundary row per colour phase, overlapped with the interior.
        field: the field h of the sweeps until set_field or a schedule changes it."""
        import torch.distributed as dist

        field = _finite_field(field)

        self.Lx, self.Ly, self.j = int(Lx), int(Lx if Ly is None else Ly), float(j)
        self._dist, self._group = dist, process_group
        active = dist.is_available() and dist.is_initialized() and dist.get_world_size(process_group) > 1
        self.rank = dist.get_rank(process_group) if active else 0
        self.world = dist.get_world_size(process_group) if active else 1
        self.row_lo, self.row_hi = shard_range(self.Ly, self.rank, self.world)
        self._torch_device = None
        self._async = False
        self._comm = None
        self._native_comm = (active and dist.get_backend(process_group) == "nccl" and int(exchange_every) > 0)
        if self._native_comm:
            # multi-GPU, batched exchange: the halo send/recv are the library's own NCCL calls on
            # its stream (ising_strip_sweeps); torch.distributed only carries the NCCL id
            ctx = nat.Context.get(device)
            self._comm = nat.Comm.from_torch(ctx, process_group)
        elif active and dist.get_backend(process_group) == "nccl":
            # multi-GPU: run the library on torch's current stream, so that halo copies, NCCL
            # send/recv and the sweep kernels are ordered on the device without host waits
            import torch

            dev = int(device) if device is not None else int(torch.cuda.current_device())
            self._torch_device = torch.device("cuda", dev)
            ctx = nat.Context(dev, stream=torch.cuda.current_stream(self._torch_device).cuda_stream)
            self._async = True
        else:
            ctx = nat.Context.get(device)
            if active:
                import torch

                self._torch_device = torch.device("cpu")
        # 2k ghost rows must come from the direct neighbour: k <= (rows of the smallest strip) / 2
        self._k = max(0, min(int(exchange_every), (self.Ly // self.world) // 2))
        ghost = max(1, 2 * self._k)
        self.strip = nat.Strip(ctx, self.Lx, self.Ly, self.row_lo, self.row_hi, j, seed, planes, rounds,
                               ghost=ghost)
        self.nsites = self.Lx * self.Ly
        self._field = 0.0
        if field != 0.0:
            self.set_field(field)
        self._bufs = None
        if self._async:
            import torch

            w = self.strip.words
            self._send = torch.empty(4 * ghost * w, dtype=torch.int32, device=self._torch_device)
            self._recv = torch.empty(4 * ghost * w, dtype=torch.int32, device=self._torch_device)
            self._bufs = (self._send, self._recv)

    def _exchange(self, colour):
        exchange_halos(self.strip, colour, self.rank, self.world, self._dist, self._group, self._torch_device)

    def set_all(self, up=True):
        self.strip.set_all(up)

    @property
    def field(self):
        """the uniform longitudinal field h of the next sweeps"""
        return self._field

    def set_field(self, h):
        self._field = _finite_field(h)
        self.strip.set_field(self._field)

    def _phase_overlapped(self, colour, beta):
        """Stage the boundary rows, start the NCCL exchange, update the interior rows while it
        is in flight, then the two boundary rows once the ghosts have arrived.  Everything is
        enqueued on one stream; the host never waits."""
        dist, w, other = self._dist, self.strip.words, 1 - colour
        rows = self.row_hi - self.row_lo
        up, down = (self.rank - 1) % self.world, (self.rank + 1) % self.world
        self.strip.halo_async(other, 0, self._send.data_ptr())
        send_top, send_bot = self._send[:w], self._send[w:2 * w]
        recv_top, recv_bot = self._recv[:w], self._recv[w:2 * w]
        if self.world == 2:   # both neighbours are the same peer: match messages by order
            ops = [dist.P2POp(dist.isend, send_top, up, group=self._group),
                   dist.P2POp(dist.isend, send_bot, down, group=self._group),
                   dist.P2POp(dist.irecv, recv_bot, down, group=self._group),
                   dist.P2POp(dist.irecv, recv_top, up, group=self._group)]
        else:
            ops = [dist.P2POp(dist.isend, send_top, up, group=self._group),
                   dist.P2POp(dist.isend, send_bot, down, group=self._group),
                   dist.P2POp(dist.irecv, recv_top, up, group=self._group),
                   dist.P2POp(dist.irecv, recv_bot, down, group=self._group)]
        reqs = dist.batch_isend_irecv(ops)
        last = colour == 1
        if rows > 2:
            self.strip.phase_rows(colour, beta, 1, rows - 1)           # interior: no ghost rows read
        for r in reqs:
            r.wait()                                                    # stream-side wait for NCCL
        self.strip.halo_async(other, 1, self._recv.data_ptr())
        if rows > 2:
            self.strip.phase_rows(colour, beta, 0, 1)
            self.strip.phase_rows(colour, beta, rows - 1, rows, advance=last)
        else:
            self.strip.phase_rows(colour, beta, 0, rows, advance=last)

    def sweeps(self, betas, fields=None):
        """One checkerboard sweep per beta: exchange the rows of the colour about to be read,
        update the other colour.  fields: the field h of each sweep (a scalar or one value per
        beta; the last one stays set), None = the current field."""
        betas = np.atleast_1d(np.asarray(betas, dtype=np.float64))
        if fields is not None:
            fields = np.asarray(fields, dtype=np.float64)
            fields = np.full(len(betas), float(fields)) if fields.ndim == 0 else fields
            if fields.shape != betas.shape:
                raise ValueError(f"fields: a scalar or one value per beta ({len(betas)}), got shape {fields.shape}")
            if not np.isfinite(fields).all():
                raise ValueError("fields must be finite")
            if len(fields) == 0:
                fields = None
        if self._native_comm or (self.world == 1 and self._k > 0):
            self.strip.sweeps(betas, self._comm, max(self._k, 1), fields=fields)   # whole loop inside the library
        elif self._k == 0:
            for t, beta in enumerate(betas):
                if fields is not None and fields[t] != self._field:
                    self.set_field(fields[t])
                for colour in (0, 1):
                    if self._async:
                        self._phase_overlapped(colour, beta)
                    else:
                        self._exchange(1 - colour)
                        self.strip.phase(colour, beta)
        else:
            sweep_batches(self.strip, betas, self._k, self.rank, self.world, self._dist, self._group,
                          self._torch_device, self._bufs, sync=not self._async, fields=fields)
        if fields is not None:
            self._field = float(fields[-1])

    def _global_sums(self):
        if self._native_comm:
            return self.strip.global_sums(self._comm)
        if self._async:
            import torch

            torch.cuda.current_stream(self._torch_device).synchronize()
        self._exchange(1)
        nsat, up = self.strip.observables()
        if self.world > 1:
            import torch

            t = torch.tensor([nsat, up], dtype=torch.int64, device=self._torch_device)
            self._dist.all_reduce(t, group=self._group)
            nsat, up = int(t[0]), int(t[1])
        return nsat, up

    def energy(self):
        """E = sum J s s' over the 2 Lx Ly bonds - h M in the current field h."""
        nsat, up = self._global_sums()
        if self._field == 0.0:
            return abs(self.j) * (2 * self.nsites - 2 * nsat)
        return abs(self.j) * (2 * self.nsites - 2 * nsat) - self._field * (2 * up - self.nsites)

    def magnetization(self):
        _, up = self._global_sums()
        return 2 * up - self.nsites

    def local_rows(self):
        """bool[row_hi - row_lo, Lx] of this rank's rows."""
        return self.strip.rows()
