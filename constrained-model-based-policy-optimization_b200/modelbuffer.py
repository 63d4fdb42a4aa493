"""`ModelBuffer` with the reference's contract (buffers/modelbuffer.py:18-226), backed by
time-major device buffers.  GAE / cost-GAE run in cmbpo_gae_paths, the advantage statistics,
normalisation and the populated-mask flatten of get() in cmbpo_adv_* / cmbpo_compact_field.
"""
import numpy as np

from . import _lib as L
from .rollout import RolloutBuffers

EPS = 1e-8


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
        self._dist = None            # distribute(): get() gathers the whole batch on one rank
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
        self._last_val = np.zeros(self.batch_size, dtype=np.float32)
        self._last_cval = np.zeros(self.batch_size, dtype=np.float32)
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
            self._last_val[fin], self._last_cval[fin] = lv[fin], lc[fin]
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
        the advantage statistics are all-reduced, and get() / get_device() return the rows of the WHOLE batch,
        in global path order, on rank `root` (group rank) and arrays with zero rows on the other ranks.  The
        diagnostics are the batch's on every rank.  Called by ModelSampler.distribute."""
        import torch.distributed as dist
        from .dist import make_reduce_fn
        self.reduce_fn = make_reduce_fn(group)
        self._dist = dict(group=group, root=int(root), rank=dist.get_rank(group))

    def _gather_rows(self, fields, off, n_rows):
        """The compacted `fields` ((field, width, vector) as get_device compacts them) of every rank, in rank
        order, into fresh [N_total, ...] tensors on the root: the root compacts its own rows straight into its
        slice of them; the other ranks compact into their persistent staging and send it; the root receives
        straight into the final slices (one batch of point-to-point operations: no padding, no reassembly copy).
        Over gloo (ranks that share a GPU) the messages are host copies.
        Returns (the tensors -- zero rows off the root --, the row count of the whole batch)."""
        import torch.distributed as dist
        from .dist import all_gather_host
        e, ds, b = self.engine, self._dist, self.bufs
        group, root, rank = ds["group"], ds["root"], ds["rank"]
        nccl = dist.get_backend(group) == "nccl"
        landed = []                         # gloo: (device slice, host message)
        counts = all_gather_host(np.array([n_rows], np.int64), group, e.device)[:, 0]
        starts = np.concatenate([[0], np.cumsum(counts)])
        n_out = int(starts[-1]) if rank == root else 0
        out, ops = [], []
        for i, (f, width, vector) in enumerate(fields):
            def compact(dst):
                return e.compact(f, self.batch_size, self.max_path_length, width, b.length, off, n_rows, dst)
            if rank == root:
                full = e.empty(n_out, width) if vector else e.empty(n_out)
                compact(full[starts[rank]:starts[rank + 1]])
                for g in range(len(counts)):
                    if g != rank and counts[g]:
                        dst = full[starts[g]:starts[g + 1]]
                        msg = dst if nccl else e.torch.empty(dst.shape, dtype=dst.dtype)
                        ops.append(dist.P2POp(dist.irecv, msg, group=group, group_peer=g))
                        if not nccl:
                            landed.append((dst, msg))
            else:
                full = e.empty(0, width) if vector else e.empty(0)
                if n_rows:
                    msg = compact(self._staging("send", i, n_rows, width, vector))
                    ops.append(dist.P2POp(dist.isend, msg if nccl else msg.cpu(), group=group, group_peer=root))
            out.append(full)
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        for dst, msg in landed:
            dst.copy_(msg)
        return out, int(starts[-1])

    # ---- get ---------------------------------------------------------------------------------
    def _staging(self, gen, i, n_rows, width, vector):
        """Persistent compaction target (generation `gen`, field `i`), sized for a full buffer: no
        allocator traffic per batch (a fresh 500 MB of tensors per batch makes the caching allocator
        call cudaMalloc / cudaFree, which synchronise the device at unpredictable moments)."""
        pool = self.__dict__.setdefault("_compact_pool", {})
        cap = self.batch_size * self.max_path_length
        buf = pool.get((gen, i))
        if buf is None or buf.numel() < cap * width:
            buf = self.engine.empty(cap * width)
            pool[(gen, i)] = buf
        flat = buf[:n_rows * width]
        return flat.view(n_rows, width) if vector else flat

    def get_device(self, staging_gen=None):
        """get() without the device->host copy: (list of 12 device tensors, diagnostics).  With
        `staging_gen` (0 | 1) the tensors are views of persistent buffers of that generation, valid
        until the second next call with the same generation."""
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
        O, A = self.obs_dim, self.act_dim
        if self._dist is not None:
            if staging_gen is not None:
                raise L.CmbpoError("the persistent staging of get_async() is for one rank only; after "
                                   "distribute() use get()")
            vec, sc = (lambda f, w: (f, w, True)), (lambda f: (f, 1, False))
            fields = [vec(b.obs, O), vec(b.act, A)] + [sc(f) for f in (b.adv, b.cadv, b.ret, b.cret, b.logp, b.val,
                                                                       b.cval, b.cost)] + [vec(b.mu, A)]
            full, n_rows = self._gather_rows(fields, off, n_rows)
            out, mu = full[:10], full[10]
            n_out = mu.shape[0]
        else:
            def tgt(i, width, vector):
                return None if staging_gen is None else self._staging(staging_gen, i, n_rows, width, vector)

            out = [e.compact(b.obs, B, T, O, b.length, off, n_rows, tgt(0, O, True)),
                   e.compact(b.act, B, T, A, b.length, off, n_rows, tgt(1, A, True))]
            for i, f in enumerate((b.adv, b.cadv, b.ret, b.cret, b.logp, b.val, b.cval, b.cost)):
                out.append(e.compact(f, B, T, 1, b.length, off, n_rows, tgt(2 + i, 1, False)))
            mu = e.compact(b.mu, B, T, A, b.length, off, n_rows, tgt(11, A, True))
            n_out = n_rows
        ls_row = self._log_std_row if self._log_std_row is not None else np.zeros(A, np.float32)
        # every row of log_std is the same [A] variable (ac_network.py:119): a stride-0 view
        log_std = e.to_device(ls_row, t.float32).reshape(1, A).expand(n_out, A)
        out += [log_std, mu]                       # sorted pi_info keys: log_std, mu
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
        `.cpu()` copies."""
        out, diag = self.get_device()
        res = self.to_host(out, pinned)
        self.reset()
        return res, diag

    def to_host(self, out, pinned=True):
        """The device->host half of get(): the 12 device tensors of get_device() as numpy arrays."""
        # log_std (index 10) is one [A] row repeated: it crosses PCIe once and is returned as a
        # read-only broadcast view (values, shape and dtype as the reference's array)
        ls_host = np.broadcast_to(out[10][:1].cpu().numpy().reshape(1, -1) if out[10].shape[0] else
                                  np.zeros((1, self.act_dim), np.float32), tuple(out[10].shape))
        if not pinned:
            return [ls_host if i == 10 else x.cpu().numpy() for i, x in enumerate(out)]
        t = self.engine.torch
        host = []
        for i, x in enumerate(out):
            if i == 10:
                host.append(None)
                continue
            h = t.empty(tuple(x.shape), dtype=x.dtype, pin_memory=True)
            h.copy_(x, non_blocking=True)
            host.append(h)
        t.cuda.current_stream(self.engine.device).synchronize()
        return [ls_host if h is None else h.numpy() for h in host]

    def get_async(self):
        """`get()` split in two so that the device->host copy of this batch overlaps the NEXT
        rollout batch (algorithms/cmbpo.py:251-270 rolls several batches per epoch and only
        concatenates their sample lists): statistics / normalisation / compaction run now on the
        engine's stream, the copies into page-locked buffers are queued on a side stream, the buffer
        resets.  Returns a handle whose `result()` waits for the copies and returns exactly what
        `get()` returns.  At most two handles may be outstanding (two pinned buffer sets).  One rank only."""
        if self._dist is not None:
            raise L.CmbpoError("get_async() runs on one rank only; after distribute() use get()")
        self._pin_gen = getattr(self, "_pin_gen", 0) ^ 1
        t, dev = self.engine.torch, self.engine.device
        # the staging / pinned buffers of this generation may still be read by the copy of the handle
        # issued two calls ago: the compaction kernels below must not start before that copy finished
        prev = self.__dict__.setdefault("_gen_done", {}).get(self._pin_gen)
        if prev is not None:
            t.cuda.current_stream(dev).wait_event(prev)
        out, diag = self.get_device(staging_gen=self._pin_gen)
        ls_row = out[10][:1].cpu().numpy().reshape(1, -1) if out[10].shape[0] else np.zeros((1, self.act_dim), np.float32)
        ls_host = np.broadcast_to(ls_row, tuple(out[10].shape))
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = t.cuda.Stream(device=dev)
        pool = self.__dict__.setdefault("_pin_pool", {})
        main = t.cuda.current_stream(dev)
        ready = t.cuda.Event()
        ready.record(main)                          # compaction kernels of this batch are queued
        host = []
        with t.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(ready)
            for i, x in enumerate(out):
                if i == 10:
                    host.append(None)
                    continue
                key = (self._pin_gen, i)
                buf = pool.get(key)
                if buf is None or buf.numel() < x.numel() or buf.dtype != x.dtype:
                    buf = t.empty(max(x.numel(), 1), dtype=x.dtype, pin_memory=True)
                    pool[key] = buf
                h = buf[:x.numel()].view(x.shape)
                h.copy_(x, non_blocking=True)       # x: persistent staging buffer of this generation
                host.append(h)
            done = t.cuda.Event()
            done.record(self._copy_stream)
        self._gen_done[self._pin_gen] = done
        self.reset()
        return PendingGet(done, host, ls_host, diag, out)


class PendingGet:
    """Handle of `ModelBuffer.get_async()`."""

    def __init__(self, done, host, ls_host, diag, keep_alive):
        self._done, self._host, self._ls, self._diag, self._keep = done, host, ls_host, diag, keep_alive

    def result(self):
        self._done.synchronize()
        self._keep = None
        return [self._ls if h is None else h.numpy() for h in self._host], self._diag
