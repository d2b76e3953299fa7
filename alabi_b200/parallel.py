"""Multi-GPU layer: one process per GPU, ``torch.distributed`` (NCCL over
NVLink / NVSwitch) for the plumbing (SURVEY 8e).

The GP is trained once on rank 0; the Cholesky factor L and alpha are broadcast
(``ncclBroadcast``); after that every unit of work is independent:

* query points and candidate batches are split by contiguous row ranges,
* the utility argmin is an ``all_gather`` of one (value, index) pair per rank
  reduced with the single-GPU tie rule (lowest global index),
* walkers are split into independent sub-ensembles whose chain blocks are
  ``all_gather``-ed.

There is no data-path collective inside predict / utility / the sampler.  The
host logic (ranges, pair reduction, chain gathering) works on CPU tensors with
the ``gloo`` backend as well, which is how the CPU test-suite covers world
size 2.
"""
import os

import numpy as np

__all__ = ["init_distributed", "shard_range", "broadcast_gp", "argmin_allgather", "allgather_rows", "allgather_walkers",
           "sharded_predict", "sharded_utility_argmin", "sharded_ensemble", "sharded_restarts",
           "broadcast_object", "world_size", "sharded_rows", "NativeComm"]


def init_distributed(backend=None):
    """Initialise torch.distributed from RANK / WORLD_SIZE / LOCAL_RANK /
    MASTER_* (torchrun).  Returns (rank, world_size, local_rank)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    elif torch.cuda.is_available():
        torch.cuda.set_device(local)
    return rank, world, local


def _dist():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized()) else None


def shard_range(m, rank, world):
    """Contiguous row range [lo, hi) of shard ``rank``; sizes differ by at most one."""
    base, rem = divmod(int(m), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class NativeComm:
    """NCCL communicator owned by libalabi_b200 (``ab_nccl_*``, include/alabi_b200.h): the factor state
    moves between the handles' own buffers without staging copies and without torch tensors.  The
    128-byte NCCL id is made on rank 0 and handed to the other ranks through whatever channel the
    application has — here ``torch.distributed``'s object broadcast, which is only used for that."""

    def __init__(self, device=None):
        import ctypes
        import torch
        from . import _lib
        dist = _dist()
        self._lib, self.lib = _lib, _lib.load()
        self.rank = dist.get_rank() if dist else 0
        self.world = dist.get_world_size() if dist else 1
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.stream = torch.cuda.current_stream(self.device)
        idb = (ctypes.c_ubyte * 128)()
        if self.rank == 0:
            _lib.check(self.lib.ab_nccl_unique_id(idb), "ab_nccl_unique_id")
        raw = broadcast_object(bytes(idb), src=0)
        idb = (ctypes.c_ubyte * 128).from_buffer_copy(raw)
        h = ctypes.c_void_p()
        _lib.check(self.lib.ab_nccl_init(ctypes.byref(h), self.world, self.rank, idb, self.device,
                                         ctypes.c_void_p(self.stream.cuda_stream)), "ab_nccl_init")
        self.h = h

    def broadcast(self, t, root=0):
        self._lib.check(self.lib.ab_nccl_broadcast(self.h, self._lib.ptr(t), t.numel() * t.element_size(), root), "ab_nccl_broadcast")
        return t

    def allgather(self, t):
        import torch
        t = t.contiguous()
        out = torch.empty((self.world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
        self._lib.check(self.lib.ab_nccl_allgather(self.h, self._lib.ptr(t), self._lib.ptr(out), t.numel() * t.element_size()),
                        "ab_nccl_allgather")
        return out

    def sync(self):
        self._lib.check(self.lib.ab_nccl_sync(self.h), "ab_nccl_sync")

    def broadcast_gp(self, gp, root=0):
        """``broadcast_gp`` through the library's own communicator: hyper-parameters, inputs and
        targets as a pickled object, then L / D^-1 / alpha handle to handle (``ab_nccl_broadcast_gp``)."""
        meta = None
        if self.rank == root:
            meta = dict(vector=gp.get_parameter_vector(include_frozen=True), x=gp._x, y=gp._y, yerr2=gp._yerr2)
        m = broadcast_object(meta, src=root)
        if self.rank != root:
            gp.set_parameter_vector(m["vector"], include_frozen=True)
            gp._x = gp.parse_samples(m["x"])
            gp._yerr2 = float(m["yerr2"])
            gp._inputs_pushed = False
            gp._mark_dirty()
            gp._push()
        self._lib.check(self.lib.ab_nccl_broadcast_gp(self.h, gp._hd.h, root), "ab_nccl_broadcast_gp")
        if self.rank != root:
            gp._y = np.ascontiguousarray(np.asarray(m["y"], dtype=np.float64).reshape(-1))
            gp.computed = True
            gp._factor_key = gp._spec_key()
            gp._targets_pushed = True
            gp._alpha_np = None
        return gp

    def close(self):
        if getattr(self, "h", None):
            self.lib.ab_nccl_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


def broadcast_gp(gp, x=None, y=None, src=0, stats=None):
    """Make every rank hold the GP trained on ``src``: hyper-parameters, inputs
    and targets travel as a pickled object, L (npad x npad), the diagonal-block inverses and
    alpha as device tensors over NCCL.  Returns the (imported) GP on every rank.  ``stats``
    (a dict) receives ``bytes`` and ``seconds`` of the three device broadcasts (CUDA events on
    the current stream around them; the first NCCL call of a process also pays the communicator
    set-up, so time a second broadcast for a bandwidth figure)."""
    import torch
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return gp
    rank = dist.get_rank()
    meta = [None]
    if rank == src:
        L, alpha = gp.export_state()
        Dinv = gp.export_block_inverses()
        meta = [dict(vector=gp.get_parameter_vector(include_frozen=True), x=gp._x, y=gp._y, yerr2=gp._yerr2,
                     npad=int(L.shape[0]), n=int(alpha.shape[0]))]
    dist.broadcast_object_list(meta, src=src)
    m = meta[0]
    on_gpu = dist.get_backend() == "nccl"
    dev = torch.device("cuda", torch.cuda.current_device()) if on_gpu else torch.device("cpu")
    if rank != src:
        L = torch.empty((m["npad"], m["npad"]), dtype=torch.float64, device=dev)
        alpha = torch.empty(m["n"], dtype=torch.float64, device=dev)
        Dinv = torch.empty((m["npad"] // 128, 128, 128), dtype=torch.float64, device=dev)
    if on_gpu:
        if stats is not None:
            torch.cuda.synchronize()       # timing requested: buffers allocated and exported on every rank first
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    dist.broadcast(L, src=src)
    dist.broadcast(Dinv, src=src)          # same diagonal-block inverses => same L^-1 bits everywhere
    dist.broadcast(alpha, src=src)
    if on_gpu:
        e1.record()
        e1.synchronize()
        if stats is not None:
            stats["bytes"] = int(8 * (L.numel() + Dinv.numel() + alpha.numel()))
            stats["seconds"] = e0.elapsed_time(e1) * 1e-3
    if rank != src:
        gp.set_parameter_vector(m["vector"], include_frozen=True)
        gp.import_state(m["x"], m["y"], L, alpha, yerr=np.sqrt(m["yerr2"]), Dinv=Dinv)
    return gp


def argmin_allgather(value, index, device=None):
    """Global (value, index) of the smallest finite value over all ranks; ties go
    to the lowest global index (what a single-GPU argmin over the concatenated
    candidates returns).  index < 0 means "no finite value on this rank"."""
    import torch
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return float(value), int(index)
    world = dist.get_world_size()
    dev = device if device is not None else (torch.device("cuda", torch.cuda.current_device())
                                             if dist.get_backend() == "nccl" else torch.device("cpu"))
    # one 16-byte record per rank: the value's bit pattern and the index, both as int64 (an index
    # carried as a float64 would be exact only below 2^53)
    mine = torch.empty(2, dtype=torch.int64)
    mine[0] = int(np.float64(value).view(np.int64))
    mine[1] = int(index)
    mine = mine.to(dev)
    out = torch.empty(2 * world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(out, mine)
    rec = out.cpu().numpy().reshape(world, 2)
    best_v, best_i = float("inf"), -1
    for r in range(world):
        v, i = float(rec[r, :1].view(np.float64)[0]), int(rec[r, 1])
        if i >= 0 and (best_i < 0 or v < best_v or (v == best_v and i < best_i)):
            best_v, best_i = v, i
    return best_v, best_i


def allgather_rows(t, dim=0):
    """Concatenate per-rank tensors that may differ in length along ``dim``."""
    import torch
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return t
    world = dist.get_world_size()
    n = torch.tensor([t.shape[dim]], dtype=torch.int64, device=t.device)
    sizes = [torch.empty_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(s) for s in sizes]
    mx = max(sizes)
    t = t.movedim(dim, 0).contiguous()
    pad = torch.zeros((mx,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[:t.shape[0]] = t
    bufs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad)
    return torch.cat([b[:s] for b, s in zip(bufs, sizes)], dim=0).movedim(0, dim)


def sharded_predict(gp, y, xq, return_var=True, gather=False):
    """Predict this rank's contiguous slice of ``xq`` (a CUDA tensor holding
    the full or the local query set is the caller's choice: pass the full set
    and the slice is taken here)."""
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    lo, hi = shard_range(xq.shape[0], rank, world)
    out = gp.predict(y, xq[lo:hi], return_var=return_var, return_cov=False)
    if not gather:
        return out, (lo, hi)
    if return_var:
        return (allgather_rows(out[0]), allgather_rows(out[1])), (lo, hi)
    return allgather_rows(out), (lo, hi)


def sharded_utility_argmin(gp, y, candidates, bounds, algorithm="bape", y_best=0.0, zeta=0.01):
    """Each rank evaluates its slice of the candidate set; one all_gather of
    (value, global index) pairs picks the winner, bit-identical to a
    single-GPU argmin over the whole set."""
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    lo, hi = shard_range(candidates.shape[0], rank, world)
    idx, val = gp.utility_argmin(y, candidates[lo:hi], bounds, algorithm=algorithm, y_best=y_best, zeta=zeta)
    return argmin_allgather(val, idx + lo if idx >= 0 else -1)


class PeerChainBuffers:
    """Gathered chain buffers of one shape in peer memory: every rank owns a (nsteps, nwalkers_total,
    ndim) chain and a (nsteps, nwalkers_total) log-probability buffer (one cudaMalloc, exported with
    CUDA IPC) and maps the buffers of all other ranks, so that the sampler kernel of rank r can write
    its columns into all of them (``ab_ensemble_config.chain_peers``).  Built collectively (one
    ``all_gather_object`` of the 64-byte handles); the two most recent shapes stay cached (an older one
    is released collectively, every rank evicting in the same order).  ``get`` returns None on EVERY
    rank when any rank could not allocate or map (no peer access, out of memory): the caller then takes
    the NCCL route."""
    _cache = {}                     # insertion ordered: least recently used first
    MAX_CACHED = 2

    @classmethod
    def get(cls, lib, device, nsteps, nwalkers_total, ndim):
        key = (int(device), int(nsteps), int(nwalkers_total), int(ndim))
        if key in cls._cache:
            cls._cache[key] = cls._cache.pop(key)                # most recently used last
            return cls._cache[key]
        while len(cls._cache) >= cls.MAX_CACHED:
            cls._cache.pop(next(iter(cls._cache))).release()
        bufs = cls(lib, *key)
        if not bufs.ok:
            bufs.release()
            return None
        cls._cache[key] = bufs
        return bufs

    def __init__(self, lib, device, nsteps, nwalkers_total, ndim):
        import ctypes
        import torch
        from . import _lib
        dist = _dist()
        self._lib, self._device = lib, device
        self.shape = (nsteps, nwalkers_total, ndim)
        nchain = nsteps * nwalkers_total * ndim * 8
        self._lp_off = (nchain + 255) // 256 * 256
        nbytes = self._lp_off + nsteps * nwalkers_total * 8
        own, hnd = ctypes.c_void_p(), (ctypes.c_ubyte * _lib.PEER_HANDLE_BYTES)()
        good = lib.ab_peer_alloc(device, nbytes, ctypes.byref(own), hnd) == 0
        self.own = own.value if good else None
        handles = [None] * dist.get_world_size()
        dist.all_gather_object(handles, bytes(hnd) if good else None)
        self.peers = []                                          # base pointers of the other ranks' buffers, by rank order
        good = good and all(hb is not None for hb in handles)
        if good:
            for r, hb in enumerate(handles):
                if r == dist.get_rank():
                    continue
                p = ctypes.c_void_p()
                buf = (ctypes.c_ubyte * _lib.PEER_HANDLE_BYTES).from_buffer_copy(hb)
                if lib.ab_peer_open(device, buf, ctypes.byref(p)) != 0:
                    good = False
                    break
                self.peers.append(p.value)
        flag = torch.tensor([1.0 if good else 0.0], device=f"cuda:{device}")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)              # usable only if every rank mapped every buffer
        self.ok = bool(flag.item() == 1.0)
        if self.ok:
            self.chain = _tensor_at(self.own, (nsteps, nwalkers_total, ndim), device)
            self.log_prob = _tensor_at(self.own + self._lp_off, (nsteps, nwalkers_total), device)

    def release(self):
        """Collective: unmap the peers' buffers, then (after everybody has) free the own one."""
        import torch
        dist = _dist()
        torch.cuda.synchronize(self._device)
        self.chain = self.log_prob = None
        for p in self.peers:
            self._lib.ab_peer_close(self._device, p)
        self.peers = []
        dist.barrier()
        if self.own is not None:
            self._lib.ab_peer_free(self._device, self.own)
            self.own = None

    def spec(self, column, row0=0, rows=None, keep_local=True):
        """What ``EnsembleSampler.run_mcmc(gather=...)`` takes: this rank's walkers are columns
        [column, column + nwalkers_local) of every row.  ``row0`` / ``rows``: the stored rows a piece of a
        longer run writes; ``keep_local=False``: the sampler keeps no copy of its own columns."""
        rows = self.shape[0] - row0 if rows is None else int(rows)
        c_off = row0 * self.shape[1] * self.shape[2] * 8
        l_off = self._lp_off + row0 * self.shape[1] * 8
        peers = list(self.peers)
        return {"chain": self.chain[row0:row0 + rows], "log_prob": self.log_prob[row0:row0 + rows],
                "nwalkers_total": self.shape[1], "column": int(column), "keep_local": bool(keep_local),
                "peer_chain_ptrs": [p + c_off for p in peers], "peer_log_prob_ptrs": [p + l_off for p in peers]}


def _tensor_at(ptr, shape, device):
    """float64 torch tensor over device memory this package owns (zero copy)."""
    import torch

    class _Mem:
        __cuda_array_interface__ = {"shape": tuple(int(v) for v in shape), "typestr": "<f8", "data": (int(ptr), False),
                                    "version": 2, "strides": None}
    return torch.as_tensor(_Mem(), device=f"cuda:{device}")


def sharded_ensemble(sampler_factory, p0, nsteps, gather=True, to_host=True, fused=True, pieces=None, **run_kwargs):
    """Independent sub-ensembles: rank r advances walkers [lo, hi) of ``p0`` with
    RNG counters offset by ``lo`` (statistically independent streams), then the
    chain blocks are all_gather-ed along the walker axis — on the device when the backend is nccl
    (the stored chain never leaves HBM before the collective).

    ``fused`` (nccl, equal shards, at most 16 ranks): the collective is fused into the sampler
    kernel — every rank's kernel stores its rows into the gathered buffer of every rank (peer memory
    over NVLink / NVSwitch, :class:`PeerChainBuffers`) while it samples, so nothing of the all_gather
    is left after the run but a barrier.  The gathered tensor then aliases a buffer that the next
    fused gather of the same shape overwrites (``to_host=True`` copies it; large chains are then sampled
    in ``pieces`` whose rows travel to the host while the next piece runs).  ``fused=False``: one NCCL
    ``all_gather_into_tensor`` after the run.

    ``sampler_factory(nwalkers_local)`` builds the rank-local EnsembleSampler.  Returns
    (sampler, chain): the gathered (nsteps, nwalkers, ndim) chain as a NumPy array
    (``to_host=True``) or as a tensor on the collective's device."""
    import torch
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    lo, hi = shard_range(len(p0), rank, world)
    s = sampler_factory(hi - lo)
    if not gather or world == 1:
        s.run_mcmc(np.asarray(p0)[lo:hi], nsteps, walker_offset=lo, **run_kwargs)
        return s, s.get_chain()
    from . import _lib
    if (fused and dist.get_backend() == "nccl" and len(p0) % world == 0 and world - 1 <= _lib.MAX_PEERS
            and not run_kwargs.get("record_proposals")):
        hd = s.log_prob_fn.gp._hd
        bufs = PeerChainBuffers.get(hd.lib, hd.device, int(nsteps), len(p0), s.ndim)
        if bufs is not None:
            # Where any rank wants the chain in host memory and it is large, the run is cut into pieces: after
            # the barrier that closes piece b its rows are complete in every rank's buffer and travel to the
            # host on a copy stream while piece b + 1 samples (the random streams are counter based: same chain)
            want = torch.tensor([1.0 if to_host else 0.0], device=f"cuda:{hd.device}")
            dist.all_reduce(want, op=dist.ReduceOp.MAX)          # also: nobody still reads the buffers of an earlier gather
            nbytes = int(nsteps) * len(p0) * s.ndim * 8
            npieces = min(4, int(nsteps)) if (want.item() > 0 and nbytes >= (128 << 20)) else 1
            if pieces is not None:
                npieces = max(1, min(int(pieces), int(nsteps)))   # (the same on every rank)
            host, copy_stream = None, None
            if to_host:
                try:
                    host = torch.empty(tuple(bufs.chain.shape), dtype=torch.float64, pin_memory=True)
                except RuntimeError:
                    host = torch.empty(tuple(bufs.chain.shape), dtype=torch.float64)
                copy_stream = torch.cuda.Stream(device=hd.device)
            per, row0 = -(-int(nsteps) // npieces), 0
            while row0 < int(nsteps):
                rows = min(per, int(nsteps) - row0)
                s.run_mcmc(np.asarray(p0)[lo:hi] if row0 == 0 else None, rows, walker_offset=lo, store="device",
                           gather=bufs.spec(lo, row0, rows, keep_local=False), **run_kwargs)
                torch.cuda.synchronize(hd.device)
                dist.barrier()                                   # every rank's kernel of this piece has finished
                if to_host:
                    with torch.cuda.stream(copy_stream):
                        host[row0:row0 + rows].copy_(bufs.chain[row0:row0 + rows], non_blocking=True)
                row0 += rows
            # the sampler's own record of the run: its columns of the gathered buffers
            s.device_chain = bufs.chain[:, lo:hi].clone()
            s.device_log_prob = bufs.log_prob[:, lo:hi].clone()
            s._device_rows_pending = True
            s.iteration += int(nsteps)
            if to_host:
                copy_stream.synchronize()
                return s, host.numpy()
            return s, bufs.chain
    if dist.get_backend() == "nccl":
        s.run_mcmc(np.asarray(p0)[lo:hi], nsteps, walker_offset=lo, store="device", **run_kwargs)
        local = s.device_chain
    else:
        s.run_mcmc(np.asarray(p0)[lo:hi], nsteps, walker_offset=lo, **run_kwargs)
        local = torch.from_numpy(np.ascontiguousarray(s.get_chain()))
    chain = allgather_walkers(local, len(p0))
    return s, (_to_host(chain) if to_host else chain)


def _to_host(t):
    """NumPy copy of a tensor; CUDA tensors land in page-locked memory (torch caches the block, so
    repeated gathers reuse locked, touched pages) unless that allocation fails."""
    import torch
    if t.device.type != "cuda":
        return t.numpy()
    try:
        h = torch.empty(tuple(t.shape), dtype=t.dtype, pin_memory=True)
    except RuntimeError:
        return t.cpu().numpy()
    h.copy_(t)
    return h.numpy()


def allgather_walkers(local, nwalkers_total):
    """all_gather of per-rank chain blocks (nsteps, nwalkers_local, ...) along the walker axis.
    Equal shards take ONE ``all_gather_into_tensor`` (rank-major) followed by a local
    re-interleave; ragged shards go through :func:`allgather_rows`."""
    import torch
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return local
    world = dist.get_world_size()
    if nwalkers_total % world != 0:
        return allgather_rows(local, dim=1)
    local = local.contiguous()
    out = torch.empty((world * local.shape[0],) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, local)                  # rank-major concatenation along dim 0
    out = out.view((world,) + tuple(local.shape))
    # (world, steps, nwl, ...) -> (steps, world * nwl, ...)
    return out.movedim(0, 1).reshape((local.shape[0], world * local.shape[1]) + tuple(local.shape[2:]))


def world_size():
    dist = _dist()
    return dist.get_world_size() if dist else 1


def broadcast_object(obj, src=0):
    """Every rank returns ``src``'s object (restart seeds, candidate sets)."""
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return obj
    box = [obj]
    dist.broadcast_object_list(box, src=src)
    return box[0]


def sharded_restarts(optimize_fn, starts):
    """Hyper-parameter optimiser restarts sharded over ranks (SURVEY 8e): restart r
    runs on rank r mod world (its own K1 + K2 per objective evaluation, no
    communication), then ONE all_gather of (fun, restart index, x) and every rank
    picks the same winner: smallest finite ``fun``, lowest restart index on ties —
    the serial ``min(results, key=fun)`` of alabi/core.py:1309-1311.

    ``optimize_fn(x0)`` returns a scipy ``OptimizeResult``; ``starts`` must be the
    same on every rank (use :func:`broadcast_object`).  Returns (best, all results
    sorted by restart index) as ``OptimizeResult`` / list of tuples."""
    from scipy.optimize import OptimizeResult
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    local = []
    for r in range(rank, len(starts), world):
        res = optimize_fn(starts[r])
        local.append((float(res.fun), r, np.asarray(res.x, dtype=np.float64), int(getattr(res, "nit", 0)),
                      bool(getattr(res, "success", True))))
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, local)
        allr = [t for g in gathered for t in g]
    else:
        allr = local
    allr.sort(key=lambda t: t[1])
    best = min(allr, key=lambda t: (t[0] if np.isfinite(t[0]) else np.inf, t[1]))
    return OptimizeResult(x=best[2], fun=best[0], nit=best[3], success=best[4], restart=best[1]), allr


def sharded_rows(eval_fn, nrows):
    """Row-sharded evaluation with one all_gather (k-fold CV candidates, SURVEY 8f-1): rank r calls
    ``eval_fn(indices)`` for the rows r, r + world, ... and gets a (len(indices), ...) float array;
    every rank returns the full (nrows, ...) array in row order.  ``eval_fn`` must depend on the
    global row index only (e.g. fold splits seeded by candidate index), so the result equals a
    single-rank evaluation."""
    import torch
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    mine = np.arange(rank, nrows, world)
    local = np.asarray(eval_fn(mine), dtype=np.float64)
    if world == 1:
        return local
    tail = tuple(local.shape[1:])
    per = (nrows + world - 1) // world
    pad = np.full((per,) + tail, np.nan)
    pad[:len(mine)] = local
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.from_numpy(pad).to(dev)
    out = torch.empty((world * per,) + tail, dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(out, t)
    out = out.cpu().numpy().reshape((world, per) + tail)
    full = np.empty((nrows,) + tail)
    for r in range(world):
        idx = np.arange(r, nrows, world)
        full[idx] = out[r, :len(idx)]
    return full
