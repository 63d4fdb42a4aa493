"""`ModelBuffer` with the reference's contract (buffers/modelbuffer.py:18-226), backed by
time-major device buffers.  GAE / cost-GAE run in cmbpo_gae_paths, the advantage statistics,
normalisation and the populated-mask flatten of get() in cmbpo_adv_* / cmbpo_compact_field.
"""
import numpy as np

from . import _lib as L
from .dist import Ranks
from .rollout import RolloutBuffers

EPS = 1e-8

# The 12 arrays of get() in the reference's order (modelbuffer.py:184-226; log_std and mu are the sorted pi_info
# keys): the RolloutBuffers field and the ModelBuffer attribute that gives its row width, None for one scalar
# per row (a 1-D array).
FIELDS = (("obs", "obs_dim"), ("act", "act_dim"), ("adv", None), ("cadv", None), ("ret", None), ("cret", None),
          ("logp", None), ("val", None), ("cval", None), ("cost", None), ("log_std", "act_dim"), ("mu", "act_dim"))
LOG_STD = [name for name, _ in FIELDS].index("log_std")


class ModelBuffer:
    def __init__(self, batch_size, obs_dim, act_dim, max_path_length, engine=None, *args, **kwargs):
        if engine is None:
            raise L.CmbpoError("ModelBuffer needs the Engine that owns the device buffers")
        self.engine = engine
        self.max_path_length = int(max_path_length)
        self.batch_size = int(batch_size)
        self.obs_shape, self.act_shape = obs_dim, act_dim
        self.obs_dim = int(np.prod(obs_dim))
        self.act_dim = int(np.prod(act_dim))
        self.pi_info_shapes = None
        self.gamma, self.lam, self.cost_gamma, self.cost_lam = 0.99, 0.95, 0.99, 0.95
        self.reduce_fn = None        # set by the multi-GPU wrapper: all-reduce of the statistics
        self._ranks = Ranks()        # the ranks get() gathers the batch from: this process alone until distribute()
        self.reset()

    def initialize(self, pi_info_shapes, gamma=0.99, lam=0.95, cost_gamma=0.99, cost_lam=0.95):
        """modelbuffer.py:41-51."""
        self.pi_info_shapes = dict(pi_info_shapes)
        self.sorted_pi_info_keys = sorted(self.pi_info_shapes)
        assert self.sorted_pi_info_keys == ["log_std", "mu"], "Gaussian policy pi_info expected"
        self.gamma, self.lam = gamma, lam
        self.cost_gamma, self.cost_lam = cost_gamma, cost_lam

    def reset(self, batch_size=None):
        """modelbuffer.py:53-98: fresh zeroed buffers sized to the batch."""
        if batch_size is not None:
            self.batch_size = int(batch_size)
        self.bufs = RolloutBuffers(self.engine, self.batch_size, self.max_path_length,
                                   self.obs_dim, self.act_dim)
        self.ptr, self.path_start_idx = 0, 0
        self.max_size = np.ones(self.batch_size) * self.max_path_length
        self.terminated_paths_mask = np.zeros(self.batch_size, dtype=bool)
        self._length = np.zeros(self.batch_size, dtype=np.int32)   # host mirror (step-wise mode)
        self._device_lengths = False     # True once a fused rollout owns length/last_val on device
        self._log_std_row = None

    # ---- properties of the reference -------------------------------------------------------
    @property
    def populated_mask(self):
        if self._device_lengths:
            return self.bufs.populated_mask()
        return np.arange(self.max_path_length)[None, :] < self._length[:, None]

    @property
    def size(self):
        # number of populated cells = sum of the path lengths (no [B, T] mask is materialised)
        if self._device_lengths:
            return int(self.bufs.length.sum().item())
        return int(self._length.sum())

    @property
    def has_room(self):
        return bool((self.ptr < self.max_size).all())

    @property
    def alive_paths(self):
        return np.logical_not(self.terminated_paths_mask)

    @property
    def holds_batch(self):
        """True from a rollout into this buffer until get() / get_async() returns it and resets."""
        return self._device_lengths or self.ptr > 0

    def __getattr__(self, name):
        # reference attribute names, e.g. obs_buf / adv_buf / term_buf, as [B, T, ...] numpy copies
        table = {"obs_buf": "obs", "act_buf": "act", "nextobs_buf": "nextobs", "rew_buf": "rew",
                 "val_buf": "val", "cost_buf": "cost", "cval_buf": "cval", "logp_buf": "logp",
                 "dyn_error_buf": "dyn_error", "adv_buf": "adv", "ret_buf": "ret",
                 "cadv_buf": "cadv", "cret_buf": "cret", "term_buf": "term"}
        if name in table and "bufs" in self.__dict__:
            return self.bufs.host(table[name])
        raise AttributeError(name)

    # ---- step-wise interface (external policy) ------------------------------------------------
    def store_multiple(self, obs, act, next_obs, rew, val, cost, cval, dyn_error, logp, pi_info, term):
        """modelbuffer.py:114-135: row i of every argument goes to the i-th alive path, column ptr."""
        assert (self.ptr < self.max_size).all()
        e, t = self.engine, self.engine.torch
        alive_idx = np.flatnonzero(self.alive_paths).astype(np.int32)
        n = len(alive_idx)
        idx = e.to_device(alive_idx, t.int32)
        B, b = self.batch_size, self.bufs

        def put(dst, src, width):
            src = e.to_device(np.asarray(src, np.float32).reshape(n, width), t.float32)
            e.scatter_rows(dst, B, width, self.ptr, idx, src)

        put(b.obs, obs, self.obs_dim); put(b.act, act, self.act_dim)
        put(b.nextobs, next_obs, self.obs_dim); put(b.mu, pi_info["mu"], self.act_dim)
        for dst, src in ((b.rew, rew), (b.val, val), (b.cost, cost), (b.cval, cval),
                         (b.logp, logp), (b.dyn_error, dyn_error)):
            put(dst, src, 1)
        tcol = b.term[self.ptr]
        tcol[idx.long()] = e.to_device(np.asarray(term, bool).astype(np.uint8).reshape(n), t.uint8)
        if n:
            self._log_std_row = np.asarray(pi_info["log_std"], np.float32).reshape(n, -1)[0].copy()
        self._length[alive_idx] = self.ptr + 1
        self.ptr += 1

    def finish_path_multiple(self, term_mask, last_val=0, last_cval=0):
        """modelbuffer.py:138-182: GAE + cost-GAE for the paths being closed, at close time."""
        term_mask = np.asarray(term_mask, dtype=bool)
        if not term_mask.any():
            return
        assert self.alive_paths.sum() == len(term_mask)
        alive_idx = np.flatnonzero(self.alive_paths)
        fin = alive_idx[term_mask]
        if self.ptr > 0:
            e, t = self.engine, self.engine.torch
            len_now = np.zeros(self.batch_size, np.int32)
            len_now[fin] = self.ptr
            lv = np.zeros(self.batch_size, np.float32)
            lc = np.zeros(self.batch_size, np.float32)
            lv[fin] = np.asarray(last_val, np.float32)
            lc[fin] = np.asarray(last_cval, np.float32)
            b = self.bufs
            e.gae_paths(b.rew, b.val, b.cost, b.cval, e.to_device(len_now, t.int32),
                        e.to_device(lv), e.to_device(lc), self.gamma, self.lam, self.cost_gamma,
                        self.cost_lam, self.batch_size, self.max_path_length, 1, self.batch_size,
                        out=(b.adv, b.ret, b.cadv, b.cret))
        # a path closed before its first store contributes nothing (modelbuffer.py:160)
        self.terminated_paths_mask[fin] = True

    # ---- fused interface --------------------------------------------------------------------
    def adopt_device_rollout(self, log_std_row):
        """Called by ModelSampler after a fused rollout filled `self.bufs` on the device."""
        self._device_lengths = True
        self._log_std_row = np.asarray(log_std_row, np.float32)

    def finish_all_device(self):
        """GAE for every path from the device-resident (length, last_val, last_cval)."""
        self.bufs.gae(self.gamma, self.lam, self.cost_gamma, self.cost_lam)
        self.terminated_paths_mask[:] = True

    # ---- multi-GPU ---------------------------------------------------------------------------
    def distribute(self, group=None, root=0):
        """Every rank of `group` holds a contiguous block of one batch's paths (rank order = path order):
        the advantage statistics are all-reduced, and get() / get_device() / get_async() return the rows of the
        WHOLE batch, in global path order, on rank `root` (group rank) and arrays with zero rows on the other
        ranks.  The diagnostics are the batch's on every rank.  Without distribute() the same code gathers from
        this process alone.  Called by ModelSampler.distribute."""
        from .dist import make_reduce_fn
        self.reduce_fn = make_reduce_fn(group)
        self._ranks = Ranks.of(group, root)

    def _gather_rows(self, off, n_rows, staging_gen):
        """The compacted rows of the FIELDS (log_std aside) of every rank, in rank order, as [N_total, ...] tensors
        on the root: persistent staging of generation `staging_gen` when given, else fresh tensors.  The root
        compacts its own rows straight into its slice of them; the other ranks compact into their persistent
        staging and send it; the root receives straight into the final slices (one batch of point-to-point
        operations: no padding, no reassembly copy).  Over gloo (ranks that share a GPU) the messages are host
        copies.  A single rank compacts its rows and exchanges nothing.
        Every write into the returned tensors is ordered before what the caller queues next on the current
        stream: the compaction runs on it, req.wait() of an NCCL receive makes it wait for NCCL's stream, and the
        gloo messages land through copies on it.  The NCCL operations themselves start only after what the
        current stream had queued before this call.  A non-root rank reuses its single "send" staging in its
        next compaction, which is ordered after the send: by req.wait() over NCCL, and over gloo because the
        message is a synchronous host copy of it.
        Returns (the tensors -- zero rows off the root, None at LOG_STD --, the row count of the whole batch)."""
        import torch.distributed as dist
        e, b, r = self.engine, self.bufs, self._ranks
        counts = r.gather(np.array([n_rows], np.int64), e.device)[:, 0]
        starts = np.concatenate([[0], np.cumsum(counts)])
        root = r.rank == r.root
        n_out = int(starts[-1]) if root else 0
        nccl = r.world > 1 and dist.get_backend(r.group) == "nccl"
        out, ops, landed = [], [], []       # landed (gloo): (device slice, host message)
        for i, (name, dim) in enumerate(FIELDS):
            if i == LOG_STD:
                out.append(None)
                continue
            width, vector = (getattr(self, dim), True) if dim else (1, False)

            def compact(dst):
                return e.compact(getattr(b, name), self.batch_size, self.max_path_length, width, b.length, off,
                                 n_rows, dst)
            if staging_gen is not None and root:
                full = self._staging(staging_gen, i, n_out, width, vector)
            else:
                full = e.empty(n_out, width) if vector else e.empty(n_out)
            if root:
                compact(full[starts[r.rank]:starts[r.rank + 1]])
                for g in range(r.world):
                    if g != r.rank and counts[g]:
                        dst = full[starts[g]:starts[g + 1]]
                        msg = dst if nccl else e.torch.empty(dst.shape, dtype=dst.dtype)
                        ops.append(dist.P2POp(dist.irecv, msg, group=r.group, group_peer=g))
                        if not nccl:
                            landed.append((dst, msg))
            elif n_rows:
                msg = compact(self._staging("send", i, n_rows, width, vector))
                ops.append(dist.P2POp(dist.isend, msg if nccl else msg.cpu(), group=r.group, group_peer=r.root))
            out.append(full)
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        for dst, msg in landed:
            dst.copy_(msg)
        return out, int(starts[-1])

    # ---- get ---------------------------------------------------------------------------------
    def _staging(self, gen, i, n_rows, width, vector):
        """Persistent compaction target (generation `gen`, field `i`), sized for a full buffer of this rank and
        grown when `n_rows` is more (the root of a sharded block holds the rows of every rank): no allocator
        traffic per batch (a fresh 500 MB of tensors per batch makes the caching allocator call cudaMalloc /
        cudaFree, which synchronise the device at unpredictable moments)."""
        pool = self.__dict__.setdefault("_compact_pool", {})
        need = max(self.batch_size * self.max_path_length, n_rows) * width
        buf = pool.get((gen, i))
        if buf is None or buf.numel() < need:
            buf = self.engine.empty(need)
            pool[(gen, i)] = buf
        flat = buf[:n_rows * width]
        return flat.view(n_rows, width) if vector else flat

    def _log_std_host(self):
        """A [1, A] float32 copy of the row every row of log_std repeats (one variable, ac_network.py:119):
        this batch's policy row, zeros before anything was stored."""
        row = self._log_std_row if self._log_std_row is not None else np.zeros(self.act_dim, np.float32)
        return np.array(row, np.float32).reshape(1, self.act_dim)

    def get_device(self, staging_gen=None):
        """get() without the device->host copy: (list of the 12 device tensors of FIELDS, diagnostics).  With
        `staging_gen` (0 | 1) the tensors are views of persistent buffers of that generation, valid
        until the second next call with the same generation.  After distribute(), the root's tensors hold the
        whole batch and the other ranks' have zero rows (never staging)."""
        assert self.terminated_paths_mask.all()
        e, t, b = self.engine, self.engine.torch, self.bufs
        B, T = self.batch_size, self.max_path_length
        if not self._device_lengths:
            b.length.copy_(e.to_device(self._length, t.int32))
        # statistics and normalisation are queued without a host round trip (device-resident sums); the first
        # synchronisation is the row count below, by which time everything is in flight
        sums = e.adv_statistics_device(b.adv, b.cadv, b.ret, b.cret, B, T, 1, B, b.length, self.reduce_fn)
        e.adv_normalise_device(b.adv, b.cadv, B, T, 1, B, b.length, sums)
        off = e.path_offsets(b.length)
        n_rows = int(off[-1].item())
        st = e.stats_from_sums(sums.cpu().numpy())
        out, n_rows = self._gather_rows(off, n_rows, staging_gen)
        n_out = out[0].shape[0]
        # every row of log_std is the same [A] variable: a stride-0 view
        out[LOG_STD] = e.to_device(self._log_std_host(), t.float32).expand(n_out, self.act_dim)
        diag = dict(poolm_batch_size=n_rows, poolm_ret_mean=st["ret_mean"],
                    poolm_cret_mean=st["cret_mean"])
        return out, diag

    def get(self, pinned=True):
        """modelbuffer.py:184-226.  Returns caller-owned numpy arrays and resets, like the reference.

        The 12 arrays are copied with one asynchronous D2H each and a single synchronisation into FRESH
        page-locked host tensors; the numpy arrays returned are views that own those tensors, so nothing here is
        recycled under the caller.  When the caller drops an array its block goes back to torch's caching host
        allocator, so in steady state (cmbpo.py:270 concatenates the arrays and drops them) no page is pinned or
        faulted again: ~50 GB/s instead of the ~3 GB/s of fresh pageable arrays.  `pinned=False`: plain pageable
        host tensors."""
        out, diag = self.get_device()
        res = self.to_host(out, pinned)
        self.reset()
        return res, diag

    def to_host(self, out, pinned=True):
        """The device->host half of get(): the 12 device tensors of get_device() as numpy arrays.  Call it
        before the next reset(): log_std comes from this batch's host row."""
        t = self.engine.torch
        host = _copy_to_host(out, lambda i, x: t.empty(tuple(x.shape), dtype=x.dtype, pin_memory=pinned))
        t.cuda.current_stream(self.engine.device).synchronize()
        return _numpy_arrays(host, self._log_std_host())

    def get_async(self):
        """`get()` split in two so that the device->host copy of this batch overlaps the NEXT
        rollout batch (algorithms/cmbpo.py:251-270 rolls several batches per epoch and only
        concatenates their sample lists): statistics / normalisation / compaction run now on the
        engine's stream, the copies into page-locked buffers are queued on a side stream, the buffer
        resets.  Returns a handle whose `result()` waits for the copies and returns exactly what
        `get()` returns.  At most two handles may be outstanding (two pinned buffer sets).

        After distribute() the root's handle returns the whole batch in global path order, the other ranks' return
        zero-row arrays at once (they copy nothing and wait for nothing of the root), and the diagnostics are the
        same on every rank.  Like get(), this is a sequence of collectives (the statistics all-reduces, the row
        count gather, the point-to-point batch): every rank calls get_async() and the rest of the block in the same
        order."""
        self._pin_gen = getattr(self, "_pin_gen", 0) ^ 1
        t, dev = self.engine.torch, self.engine.device
        # the staging / pinned buffers of this generation may still be read by the copy of the handle
        # issued two calls ago: the compaction kernels and the receives below (NCCL's stream waits for the
        # current stream when they are queued) must not start before that copy finished
        prev = self.__dict__.setdefault("_gen_done", {}).get(self._pin_gen)
        if prev is not None:
            t.cuda.current_stream(dev).wait_event(prev)
        out, diag = self.get_device(staging_gen=self._pin_gen)
        if self._ranks.rank != self._ranks.root:
            host = [None if i == LOG_STD else t.empty(tuple(x.shape), dtype=x.dtype) for i, x in enumerate(out)]
            res = PendingGet(None, host, self._log_std_host(), diag, None)
            self.reset()
            return res
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = t.cuda.Stream(device=dev)
        pool = self.__dict__.setdefault("_pin_pool", {})

        def pinned(i, x):                           # the page-locked buffer of this generation and field
            key = (self._pin_gen, i)
            buf = pool.get(key)
            if buf is None or buf.numel() < x.numel() or buf.dtype != x.dtype:
                buf = t.empty(max(x.numel(), 1), dtype=x.dtype, pin_memory=True)
                pool[key] = buf
            return buf[:x.numel()].view(x.shape)

        main = t.cuda.current_stream(dev)
        # recorded after get_device() returned: behind this batch's compaction kernels and, on the root of a
        # sharded block, behind the receives of the other ranks' rows (NCCL: req.wait() made the current stream
        # wait for them; gloo: they landed through copies on it), so the copies below read complete rows
        ready = t.cuda.Event(enable_timing=True)
        ready.record(main)
        with t.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(ready)
            host = _copy_to_host(out, pinned)       # out: persistent staging buffers of this generation
            done = t.cuda.Event(enable_timing=True)
            done.record(self._copy_stream)
        self._gen_done[self._pin_gen] = done
        res = PendingGet(done, host, self._log_std_host(), diag, out, ready)
        self.reset()
        return res


def _copy_to_host(out, host_like):
    """Queue on the current stream one device->host copy of each of get_device()'s tensors but log_std, into
    `host_like(i, x)` (a host tensor of x's shape and dtype).  Returns the host tensors, None at LOG_STD."""
    host = [None] * len(out)
    for i, x in enumerate(out):
        if i != LOG_STD:
            host[i] = host_like(i, x)
            host[i].copy_(x, non_blocking=True)
    return host


def _numpy_arrays(host, log_std_row):
    """get()'s 12 numpy arrays from the host tensors of _copy_to_host: log_std is the [1, A] row as a read-only
    broadcast view (values, shape and dtype as the reference's array; it crossed PCIe once, as an upload)."""
    rows = host[0].shape[0]
    return [np.broadcast_to(log_std_row, (rows, log_std_row.shape[1])) if i == LOG_STD else h.numpy()
            for i, h in enumerate(host)]


class PendingGet:
    """Handle of `ModelBuffer.get_async()`.  `done` None: nothing was copied (a non-root rank of a sharded block)."""

    def __init__(self, done, host, log_std_row, diag, keep_alive, ready=None):
        self._done, self._host, self._ls, self._diag, self._keep = done, host, log_std_row, diag, keep_alive
        self._ready = ready

    def result(self):
        if self._done is not None:
            self._done.synchronize()
        self._keep = None
        return _numpy_arrays(self._host, self._ls), self._diag

    def copy_ms(self):
        """Device time (ms) from the end of the batch's compaction and receives to the end of its device->host
        copy, None when nothing was copied.  Call after result()."""
        if self._done is None:
            return None
        return self._ready.elapsed_time(self._done)
