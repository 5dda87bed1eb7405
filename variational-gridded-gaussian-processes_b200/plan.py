"""Host-side wrapper of one libvggp plan + the autograd bridge used by the model classes.

The three C-ABI calls of a step (grid forward -> per-observation forward+backward -> grid backward) run
asynchronously on torch's current CUDA stream; with a process group, the single all-reduce(sum) of the
per-observation gradient buffer sits between the second and third call (SURVEY.md section 8e)."""
import ctypes as C
from typing import List, Optional, Sequence

import torch

from . import _lib

_TORCH_DTYPE = {_lib.F32: torch.float32, _lib.F64: torch.float64}
_OBS_CODE = {torch.float32: _lib.F32, torch.float64: _lib.F64}


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class GridPlan:
    """Grid descriptor (family, per-dimension float32 meshes) + device workspace."""

    def __init__(self, family: int, meshes: Sequence[torch.Tensor], obs_dtype: torch.dtype, device):
        lib = _lib.load()
        self.lib = lib
        self.family = int(family)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("GridPlan needs a CUDA device: this package has no CPU path")
        self.obs_dtype = obs_dtype
        self.D = len(meshes)
        self.meshes = [m.detach().to("cpu", torch.float32).contiguous() for m in meshes]
        n_knots = (C.c_int * self.D)(*[int(m.numel()) for m in self.meshes])
        ptrs = (C.POINTER(C.c_float) * self.D)(
            *[C.cast(m.data_ptr(), C.POINTER(C.c_float)) for m in self.meshes])
        handle = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", dev_index)
        _lib.check(lib.vggp_plan_create(C.byref(handle), self.family, self.D, n_knots, ptrs,
                                        _OBS_CODE[obs_dtype], dev_index))
        self.handle = handle
        dims = (C.c_int * 3)()
        M = C.c_int64()
        Dd = C.c_int()
        _lib.check(lib.vggp_plan_dims(handle, C.byref(Dd), dims, C.byref(M)))
        self.m_per_dim = [int(dims[d]) for d in range(self.D)]
        self.M = int(M.value)
        self.L_sizes = [n * n for n in self.m_per_dim]
        self.L_total = sum(self.L_sizes)
        ne, so, ns, tot = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        _lib.check(lib.vggp_gbuf_layout(handle, C.byref(ne), C.byref(so), C.byref(ns), C.byref(tot)))
        self.gbuf_obs_elems, self.gbuf_scalar_offset = int(ne.value), int(so.value)
        self.gbuf_scalars, self.gbuf_bytes = int(ns.value), int(tot.value)
        self.gbuf = torch.zeros(self.gbuf_bytes, dtype=torch.uint8, device=self.device)
        self.last_out = None                   # [ELBO, scaled ELL, KL, n_obs] of the last step (device tensor)

    def __del__(self):
        h = getattr(self, "handle", None)
        if h is not None and h.value:
            try:
                self.lib.vggp_plan_destroy(h)
            except Exception:
                pass
            self.handle = None

    # -- views of the gradient buffer (what gets all-reduced) ------------------------------------------------
    def gbuf_views(self, gbuf: Optional[torch.Tensor] = None):
        g = self.gbuf if gbuf is None else gbuf
        esz = 4 if self.obs_dtype == torch.float32 else 8
        obs = g[: self.gbuf_obs_elems * esz].view(self.obs_dtype)
        scal = g[self.gbuf_scalar_offset: self.gbuf_scalar_offset + 8 * self.gbuf_scalars].view(torch.float64)
        return obs, scal

    # -- the three calls -------------------------------------------------------------------------------------
    def grid_forward(self, theta: torch.Tensor, m: torch.Tensor, L: torch.Tensor):
        self._check_f64(theta, 2 * self.D + 1, "theta")
        self._check_f64(m, self.M, "m")
        self._check_f64(L, self.L_total, "L")
        _lib.check(self.lib.vggp_grid_forward(self.handle, theta.data_ptr(), m.data_ptr(), L.data_ptr(),
                                              _stream_ptr(self.device)))

    def _check_obs(self, xs, y, n):
        if len(xs) != self.D:
            raise ValueError(f"expected {self.D} coordinate arrays")
        for t in list(xs) + [y]:
            if t.dtype != self.obs_dtype or t.device != self.device or not t.is_contiguous() or t.numel() != n:
                raise ValueError("observations must be contiguous 1-D tensors of the plan's dtype on the plan's device")

    def pack(self, xs: Sequence[torch.Tensor], y: torch.Tensor, sort_by_cell: bool = True) -> "PackedObs":
        """One-time layout pass (X is constant over optimisation steps): optional ordering by grid cell + the
        warp-transposed layout the fused kernel streams (include/vggp.h, vggp_obs_pack)."""
        n = int(y.numel())
        self._check_obs(xs, y, n)
        npk, run = C.c_int64(), C.c_int()
        _lib.check(self.lib.vggp_obs_pack_geometry(self.handle, n, C.byref(npk), C.byref(run)))
        xp = [torch.empty(int(npk.value), dtype=self.obs_dtype, device=self.device) for _ in range(self.D)]
        yp = torch.empty(int(npk.value), dtype=self.obs_dtype, device=self.device)
        if n > 0:
            src = (C.c_void_p * self.D)(*[t.data_ptr() for t in xs])
            dst = (C.c_void_p * self.D)(*[t.data_ptr() for t in xp])
            _lib.check(self.lib.vggp_obs_pack(self.handle, src, y.data_ptr(), n, 1 if sort_by_cell else 0, dst,
                                              yp.data_ptr(), _stream_ptr(self.device)))
        return PackedObs(xp, yp, n, int(run.value), bool(sort_by_cell))

    def bin(self, xs: Sequence[torch.Tensor], y: torch.Tensor, run_cap: int = 256) -> "BinnedObs":
        """One-time layout pass, second form (include/vggp.h, vggp_obs_bin_*): observations ordered by grid cell, cut
        into per-cell runs of at most `run_cap`, 32 equally long runs per warp task.  The hot-path layout of both
        families since round 2 (DESIGN.md sections 8 and 10); `pack` stays as the any-order cross-check."""
        n = int(y.numel())
        self._check_obs(xs, y, n)
        desc = _lib.BinnedDesc()
        src = (C.c_void_p * self.D)(*[t.data_ptr() for t in xs])
        _lib.check(self.lib.vggp_obs_bin_prepare(self.handle, src, n, int(run_cap), C.byref(desc),
                                                 _stream_ptr(self.device)))
        buf = torch.empty(int(desc.bytes), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.vggp_obs_bin_pack(self.handle, C.byref(desc), src, y.data_ptr(), buf.data_ptr(),
                                              _stream_ptr(self.device)))
        return BinnedObs(buf, desc, 4 if self.obs_dtype == torch.float32 else 8)

    def bin_epoch(self, xs: Sequence[torch.Tensor], y: torch.Tensor, batch_size: int, seed: int, epoch: int,
                  run_cap: int = 256, rank: int = 0, n_batches: int = 0) -> "EpochBins":
        """All minibatches of one epoch in the binned layout, binned in one device pass (include/vggp.h, vggp_epoch_bin_*).
        Epoch `epoch` of `rank` draws a pseudo-random permutation pi of the n observations (keyed by seed, epoch and rank);
        batch b is {i : pi(i) in [b B, (b + 1) B)} for b < P = n // B (or `n_batches`, which a sharded run sets to the
        smallest shard's count), the rest of the epoch is dropped.  Each batch is a BinnedBatch view of one buffer: a
        BinnedObs with n = B and scale = n / B, bit-identical to `bin` of its observations in ascending index order."""
        n = int(y.numel())
        self._check_obs(xs, y, n)
        B = int(batch_size)
        P = int(n_batches) or (n // B if B >= 1 else 0)
        desc = _lib.EpochDesc()
        totals = (C.c_int64 * max(1, _lib.EPOCH_TOTALS * P))()
        src = (C.c_void_p * self.D)(*[t.data_ptr() for t in xs])
        _lib.check(self.lib.vggp_epoch_bin_prepare(self.handle, src, n, B, int(n_batches), int(run_cap), int(seed), int(epoch),
                                                   int(rank), C.byref(desc), totals, _stream_ptr(self.device)))
        buf = torch.empty(int(desc.bytes), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.vggp_epoch_bin_pack(self.handle, C.byref(desc), totals, src, y.data_ptr(), buf.data_ptr(),
                                                _stream_ptr(self.device)))
        esz = 4 if self.obs_dtype == torch.float32 else 8
        batches = []
        for b in range(int(desc.n_batches)):
            bd, off = _lib.BinnedDesc(), C.c_int64()
            _lib.check(self.lib.vggp_epoch_batch(C.byref(desc), totals, b, C.byref(bd), C.byref(off)))
            batches.append(BinnedBatch(buf[int(off.value):], bd, esz, float(n) / float(B)))
        return EpochBins(buf, desc, batches)

    def meanopt_assemble(self, binned: "BinnedObs"):
        """Fill the stencil system of the optimal variational mean from a binned buffer of this plan
        (vggp_meanopt_assemble; B1 and SVGP_MARKOV families, the latter at the theta of the last grid_forward)."""
        if not isinstance(binned, BinnedObs):
            raise TypeError("meanopt_assemble takes the BinnedObs of GridPlan.bin")
        _lib.check(self.lib.vggp_meanopt_assemble(self.handle, C.byref(binned.desc), binned.buf.data_ptr(),
                                                  _stream_ptr(self.device)))

    MEANOPT_PRECONDITIONERS = {"jacobi": _lib.MEANOPT_JACOBI, "kronecker": _lib.MEANOPT_KRONECKER}

    def meanopt_solve(self, rtol: float, max_iter: int, preconditioner: str = "jacobi"):
        """Conjugate gradients on the assembled system from the state of the last grid_forward (vggp_meanopt_solve_pc;
        synchronises).  `preconditioner`: "jacobi" (vggp_meanopt_solve) or "kronecker" (kron_d (F_d + g I)^-1 of the
        per-dimension prior factors, applied exactly by tridiagonal sweeps).  Returns (m_star float64 [M], iterations,
        final relative residual); not converged when relres > rtol."""
        if preconditioner not in self.MEANOPT_PRECONDITIONERS:
            raise ValueError(f"preconditioner must be one of {sorted(self.MEANOPT_PRECONDITIONERS)}, not {preconditioner!r}")
        m = torch.empty(self.M, dtype=torch.float64, device=self.device)
        it, rr = C.c_int(0), C.c_double(0.0)
        _lib.check(self.lib.vggp_meanopt_solve_pc(self.handle, self.MEANOPT_PRECONDITIONERS[preconditioner], float(rtol),
                                                  int(max_iter), m.data_ptr(), C.byref(it), C.byref(rr),
                                                  _stream_ptr(self.device)))
        return m, int(it.value), float(rr.value)

    PROBES = {"rademacher": _lib.PROBE_RADEMACHER, "unit": _lib.PROBE_UNIT}

    def logdet_system(self, n_probes: int, seed: int = 0, preconditioner: str = "kronecker", probes: str = "rademacher",
                      max_steps: int = 1000, rtol: float = 1e-6, per_probe: bool = False) -> dict:
        """log det of the assembled optimal-mean system A by preconditioned stochastic Lanczos quadrature
        (vggp_logdet_system; synchronises).  `probes`: "rademacher" (signs hashed from `seed`) or "unit" (e_seed ..
        e_{seed + n_probes - 1}: with seed = 0 and n_probes = M the exact value).  Returns {"logdet", "stderr", "logdet_p",
        "steps", "converged", "probes"} and, with per_probe, the per-probe values (float64 CPU tensor)."""
        if preconditioner not in self.MEANOPT_PRECONDITIONERS:
            raise ValueError(f"preconditioner must be one of {sorted(self.MEANOPT_PRECONDITIONERS)}, not {preconditioner!r}")
        if probes not in self.PROBES:
            raise ValueError(f"probes must be one of {sorted(self.PROBES)}, not {probes!r}")
        out = (C.c_double * _lib.LOGDET_FIELDS)()
        pp = (C.c_double * int(n_probes))() if per_probe and n_probes > 0 else None
        _lib.check(self.lib.vggp_logdet_system(self.handle, self.MEANOPT_PRECONDITIONERS[preconditioner], self.PROBES[probes],
                                               int(n_probes), int(seed), int(max_steps), float(rtol), C.cast(out, C.c_void_p),
                                               C.cast(pp, C.c_void_p) if pp is not None else None,
                                               _stream_ptr(self.device)))
        res = {"logdet": out[0], "stderr": out[1], "logdet_p": out[2], "steps": int(out[3]), "converged": int(out[4]),
               "probes": int(out[5])}
        if pp is not None:
            res["per_probe"] = torch.tensor(pp[:], dtype=torch.float64)
        return res

    def collapsed_terms(self, binned: "BinnedObs") -> torch.Tensor:
        """{N, sum y^2, b^T x*, tr(F^-1 G), log det Kuu} (float64 device tensor; vggp_collapsed_terms, asynchronous) of the
        assembled and solved optimal-mean system; `binned` is the set given to meanopt_assemble."""
        if not isinstance(binned, BinnedObs):
            raise TypeError("collapsed_terms takes the BinnedObs of GridPlan.bin")
        out = torch.empty(_lib.CT_FIELDS, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.vggp_collapsed_terms(self.handle, C.byref(binned.desc), binned.buf.data_ptr(), out.data_ptr(),
                                                 _stream_ptr(self.device)))
        return out

    def covopt_update(self, dim: int, gbuf: torch.Tensor, ell_scale: float, L: torch.Tensor, change: torch.Tensor):
        """One coordinate update of the optimal Kronecker-factored covariance (vggp_covopt_update; B1 and SVGP_MARKOV):
        block `dim` of the float64 factors `L` (the L of the last grid_forward) is overwritten in place with the Cholesky
        factor of the S_dim that maximises the ELBO given the other factors, and the normalised factor change is added to
        the float64 device scalar `change`.  `gbuf` is the gradient buffer of a step at that forward, all-reduced when
        sharded.  Asynchronous."""
        self._check_f64(L, self.L_total, "L")
        self._check_f64(change, 1, "change")
        if gbuf.device != self.device or gbuf.numel() < self.gbuf_bytes:
            raise ValueError("gbuf must be a gradient buffer of this plan")
        _lib.check(self.lib.vggp_covopt_update(self.handle, int(dim), gbuf.data_ptr(), float(ell_scale), L.data_ptr(),
                                               L.data_ptr(), change.data_ptr(), _stream_ptr(self.device)))

    def predict(self, xs: Sequence[torch.Tensor]):
        """Marginal mean and variance of q(f(x*)) at test points, from the state of the last grid_forward."""
        n = int(xs[0].numel())
        xs = [t.to(self.device, self.obs_dtype).contiguous() for t in xs]
        if len(xs) != self.D or any(t.numel() != n for t in xs):
            raise ValueError(f"expected {self.D} coordinate arrays of equal length")
        mean = torch.empty(n, dtype=self.obs_dtype, device=self.device)
        var = torch.empty(n, dtype=self.obs_dtype, device=self.device)
        ptrs = (C.c_void_p * self.D)(*[t.data_ptr() for t in xs])
        _lib.check(self.lib.vggp_predict(self.handle, ptrs, n, mean.data_ptr(), var.data_ptr(),
                                         _stream_ptr(self.device)))
        return mean, var

    def predict_metrics(self, xs: Sequence[torch.Tensor], y: torch.Tensor) -> dict:
        """MSE, MAE, RMSE, R^2 (src/utils/evaluationmetrics.py:6-54) of the posterior mean at the test points against
        `y`, in one fused pass: the predictions are never written to memory (vggp_predict_metrics)."""
        from .utils.evaluationmetrics import finish
        n = int(y.numel())
        xs = [t.to(self.device, self.obs_dtype).contiguous() for t in xs]
        y = y.to(self.device, self.obs_dtype).contiguous()
        if len(xs) != self.D or any(t.numel() != n for t in xs):
            raise ValueError(f"expected {self.D} coordinate arrays of the length of y")
        out = torch.empty(4, dtype=torch.float64, device=self.device)
        ptrs = (C.c_void_p * self.D)(*[t.data_ptr() for t in xs])
        _lib.check(self.lib.vggp_predict_metrics(self.handle, ptrs, y.data_ptr(), n, out.data_ptr(),
                                                 _stream_ptr(self.device)))
        return finish(out, n)

    def cell_keys(self, xs: Sequence[torch.Tensor]) -> torch.Tensor:
        """Flat (row-major) cell id of every observation, n_cells for observations outside the mesh (B1 stencil)."""
        key = None
        inside = None
        for d in range(self.D):
            c, _, _ = self.b1_stencil(d, xs[d])
            ok = c >= 0
            c = c.clamp(min=0).to(torch.int64)
            cells = int(self.meshes[d].numel()) - 1
            key = c if key is None else key * cells + c
            inside = ok if inside is None else (inside & ok)
        return torch.where(inside, key, torch.full_like(key, self.n_cells))

    @property
    def n_cells(self) -> int:
        n = 1
        for m in self.meshes:
            n *= int(m.numel()) - 1
        return n

    def obs_fwd_bwd(self, xs, y: Optional[torch.Tensor] = None, gbuf: Optional[torch.Tensor] = None):
        """Fused per-observation forward+backward.  `xs` is either a PackedObs (hot path) or a list of plain
        coordinate arrays with targets `y` (any order; transposed into plan scratch first)."""
        g = self.gbuf if gbuf is None else gbuf
        if isinstance(xs, BinnedObs):
            _lib.check(self.lib.vggp_obs_fwd_bwd_binned(self.handle, C.byref(xs.desc), xs.buf.data_ptr(), g.data_ptr(),
                                                        _stream_ptr(self.device)))
            return
        if isinstance(xs, PackedObs):
            ptrs = (C.c_void_p * self.D)(*[t.data_ptr() for t in xs.xp])
            _lib.check(self.lib.vggp_obs_fwd_bwd_packed(self.handle, ptrs, xs.yp.data_ptr(), xs.n, g.data_ptr(),
                                                        _stream_ptr(self.device)))
            return
        n = int(y.numel())
        self._check_obs(xs, y, n)
        ptrs = (C.c_void_p * self.D)(*[t.data_ptr() for t in xs])
        _lib.check(self.lib.vggp_obs_fwd_bwd(self.handle, ptrs, y.data_ptr(), n, g.data_ptr(),
                                             _stream_ptr(self.device)))

    def grid_backward(self, theta, m, L, ell_scale: float, gbuf: Optional[torch.Tensor] = None):
        g = self.gbuf if gbuf is None else gbuf
        out = torch.empty(4, dtype=torch.float64, device=self.device)
        dtheta = torch.empty(2 * self.D + 1, dtype=torch.float64, device=self.device)
        dm = torch.empty(self.M, dtype=torch.float64, device=self.device)
        dL = torch.empty(self.L_total, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.vggp_grid_backward(self.handle, theta.data_ptr(), m.data_ptr(), L.data_ptr(),
                                               g.data_ptr(), float(ell_scale), out.data_ptr(), dtheta.data_ptr(),
                                               dm.data_ptr(), dL.data_ptr(), _stream_ptr(self.device)))
        return out, dtheta, dm, dL

    def enable_peer_allreduce(self, group=None) -> bool:
        """Make `allreduce_gbuf` the library's own one-kernel collective over NVLink peer memory (vggp_allreduce_gbuf,
        csrc/collective.cuh) instead of NCCL: the plan's gradient buffer is re-allocated as a SYMMETRIC buffer (same size on
        every rank, mapped into every process) together with a small signal pad.  torch.distributed._symmetric_memory does
        the allocation and the handle exchange (plumbing); the reduction kernel is ours.  Collective call: every rank of
        `group` (<= 8 ranks of one NVSwitch node) must make it.  Returns whether the multicast (in-switch reduction) path
        is available; without it the kernel uses peer loads / stores."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        grp = dist.group.WORLD if group is None else group
        world, rank = dist.get_world_size(grp), dist.get_rank(grp)
        if world > 8:
            raise ValueError("the peer-memory collective covers one NVSwitch node (<= 8 ranks)")
        with torch.cuda.device(self.device):
            buf = symm.empty(self.gbuf_bytes, dtype=torch.uint8, device=self.device)
            pad = symm.empty(576, dtype=torch.int32, device=self.device)     # VGGP_AR_PAD_WORDS
            buf.zero_()
            pad.zero_()
            hb = symm.rendezvous(buf, grp)
            hp = symm.rendezvous(pad, grp)
        desc = _lib.ArDesc()
        # the handle's pointers address the allocation block; the tensor sits `offset` bytes into it (0 for its own block)
        ob, op = int(getattr(hb, "offset", 0) or 0), int(getattr(hp, "offset", 0) or 0)
        mc = int(getattr(hb, "multicast_ptr", 0) or 0)
        desc.mc_ptr = (mc + ob) if mc else None
        for r in range(world):
            desc.buf_ptrs[r] = int(hb.buffer_ptrs[r]) + ob
            desc.pad_ptrs[r] = int(hp.buffer_ptrs[r]) + op
        if desc.buf_ptrs[rank] != buf.data_ptr() or desc.pad_ptrs[rank] != pad.data_ptr():
            raise RuntimeError("symmetric-memory handle does not address the local tensors")
        desc.rank, desc.world = rank, world
        self.gbuf = buf
        self._ar = {"desc": desc, "handles": (hb, hp), "pad": pad,
                    "err": torch.zeros(1, dtype=torch.int32, device=self.device)}
        torch.cuda.synchronize(self.device)
        dist.barrier(grp)                   # every pad is zeroed before the first signal arrives
        return bool(mc)

    def peer_allreduce_failed(self) -> bool:
        """True if a barrier of the peer-memory collective timed out (synchronises)."""
        ar = getattr(self, "_ar", None)
        return bool(ar is not None and int(ar["err"].item()) != 0)

    def allreduce_gbuf(self, group=None, gbuf: Optional[torch.Tensor] = None):
        """One sum-all-reduce of the per-observation gradient buffer: the library's peer-memory kernel after
        `enable_peer_allreduce`, otherwise one NCCL launch (two typed views of one allocation inside one group when the
        observation dtype is float32, a single float64 view otherwise)."""
        from .dist import allreduce_gbuf_views
        g = self.gbuf if gbuf is None else gbuf
        ar = getattr(self, "_ar", None)
        if ar is not None and g is self.gbuf:
            _lib.check(self.lib.vggp_allreduce_gbuf(self.handle, C.byref(ar["desc"]), ar["err"].data_ptr(),
                                                    _stream_ptr(self.device)))
            return
        obs, scal = self.gbuf_views(g)
        allreduce_gbuf_views(g, obs, scal, group)

    def step(self, theta, m, L, xs, y, ell_scale: float = 1.0, group=None):
        """ELBO and all gradients for one (sharded) minibatch.  Returns (out[4], dtheta, dm, dL).
        `group`: None = single process; "world" or a ProcessGroup = all-reduce the gradient buffer over it."""
        self.grid_forward(theta, m, L)
        self.obs_fwd_bwd(xs, y)
        if group is not None:
            self.allreduce_gbuf(None if isinstance(group, str) else group)
        res = self.grid_backward(theta, m, L, ell_scale)
        self.last_out = res[0]
        return res

    def graphed_step(self, theta, m, L, xs, y=None, ell_scale: float = 1.0, group=None, warmup: int = 3):
        """Capture the C-ABI launches of one step into CUDA graphs (opt-in; removes the launch gaps between the ~15
        small kernels).  `theta`, `m`, `L` and the observations are STATIC device buffers: write new parameter values
        into them (copy_) and call `.replay()`.  An NCCL all-reduce is NOT captured -- a round-1 run with NCCL inside the
        graph did not shut down cleanly -- so a sharded step over NCCL is two graphs around one eager all-reduce.  After
        `enable_peer_allreduce` the collective is this library's own kernel (no per-call argument) and the whole sharded
        step is ONE graph."""
        gs = GraphedStep(self, group)
        peer = group is not None and getattr(self, "_ar", None) is not None
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.step(theta, m, L, xs, y, ell_scale, group)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        gs.front = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gs.front):
            self.grid_forward(theta, m, L)
            self.obs_fwd_bwd(xs, y)
            if peer:
                self.allreduce_gbuf(None)
            if group is None or peer:
                gs.outs = self.grid_backward(theta, m, L, ell_scale)
        if group is not None and not peer:
            gs.back = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gs.back):
                gs.outs = self.grid_backward(theta, m, L, ell_scale)
        return gs

    def workspace_bytes(self) -> dict:
        """Device memory behind the plan (vggp_workspace_bytes): plan-owned, the caller-owned gradient buffer, opt-in scratch."""
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        _lib.check(self.lib.vggp_workspace_bytes(self.handle, C.byref(a), C.byref(b), C.byref(c)))
        return {"plan": int(a.value), "gbuf": int(b.value), "scratch": int(c.value)}

    def set_deterministic(self, on: bool = True):
        """Bitwise run-to-run reproducible steps (vggp_set_deterministic): B1 family, binned layout, M_d <= 512."""
        _lib.check(self.lib.vggp_set_deterministic(self.handle, 1 if on else 0))

    def k1_timing(self, enable: bool = True):
        """Start / stop the library's own device timing of the per-observation kernel (vggp_k1_timing)."""
        _lib.check(self.lib.vggp_k1_timing(self.handle, 1 if enable else 0))

    def k1_time_read(self):
        """(mean milliseconds, launches) of the per-observation kernel since k1_timing(True); synchronises."""
        ms, n = C.c_float(0.0), C.c_int(0)
        _lib.check(self.lib.vggp_k1_time_read(self.handle, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def k1_graph_time_read(self) -> float:
        """Milliseconds of the per-observation kernel in the most recent replay of a graph captured while k1_timing was on
        (external event-record nodes inside the graph); synchronises."""
        ms = C.c_float()
        _lib.check(self.lib.vggp_k1_graph_time_read(self.handle, C.byref(ms)))
        return float(ms.value)

    def arm_info_check(self):
        """Copy the factorisation flag of the last forward into pinned host memory in stream order, without synchronising
        (vggp_info_async), and record an event behind the copy; `poll_info` turns it into a value later."""
        if getattr(self, "_info_host", None) is None:
            self._info_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        _lib.check(self.lib.vggp_info_async(self.handle, self._info_host.data_ptr(), _stream_ptr(self.device)))
        self._info_event = torch.cuda.Event()
        self._info_event.record(torch.cuda.current_stream(self.device))

    def poll_info(self, wait: bool) -> Optional[int]:
        """Flag armed by `arm_info_check` (0 = ok, d + 1 = factor d not positive definite), or None if nothing is armed /
        the copy has not completed yet and `wait` is False."""
        ev = getattr(self, "_info_event", None)
        if ev is None:
            return None
        if wait:
            ev.synchronize()
        elif not ev.query():
            return None
        self._info_event = None
        return int(self._info_host[0])

    def read_info(self) -> int:
        info = C.c_int(0)
        _lib.check(self.lib.vggp_read_info(self.handle, C.byref(info), _stream_ptr(self.device)))
        return int(info.value)

    # -- feature evaluation ----------------------------------------------------------------------------------
    def b1_stencil(self, dim: int, x: torch.Tensor):
        x = x.to(self.device, self.obs_dtype).contiguous()
        n = x.numel()
        c = torch.empty(n, dtype=torch.int32, device=self.device)
        wl = torch.empty_like(x)
        wh = torch.empty_like(x)
        _lib.check(self.lib.vggp_b1_stencil(self.handle, dim, x.data_ptr(), n, c.data_ptr(), wl.data_ptr(),
                                            wh.data_ptr(), _stream_ptr(self.device)))
        return c, wl, wh

    def features_dense(self, dim: int, x: torch.Tensor, theta: Optional[torch.Tensor] = None):
        x = x.to(self.device, self.obs_dtype).contiguous()
        n = x.numel()
        phi = torch.empty(self.m_per_dim[dim], n, dtype=self.obs_dtype, device=self.device)
        tp = theta.data_ptr() if theta is not None else None
        _lib.check(self.lib.vggp_features_dense(self.handle, dim, x.data_ptr(), n, tp, phi.data_ptr(),
                                                _stream_ptr(self.device)))
        return phi

    # -- workspace views -------------------------------------------------------------------------------------
    def workspace(self, which: int, dim: int = 0) -> torch.Tensor:
        """Copy of a float64 workspace array of the last forward (tests / predictions)."""
        ptr, n = C.c_void_p(), C.c_int64()
        _lib.check(self.lib.vggp_workspace_ptr(self.handle, which, dim, C.byref(ptr), C.byref(n)))
        out = torch.as_tensor(_DevArray(ptr.value, int(n.value)), device=self.device).clone()
        if which in (_lib.WS_ALPHA, _lib.WS_SCAL, _lib.WS_QBAND):
            return out
        nd = self.m_per_dim[dim]
        return out.view(nd, nd)

    def mode_product(self, dim: int, A: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
        dst = torch.empty_like(src)
        _lib.check(self.lib.vggp_mode_product(self.handle, dim, A.data_ptr(), src.data_ptr(), dst.data_ptr(),
                                              _stream_ptr(self.device)))
        return dst

    def _check_f64(self, t: torch.Tensor, numel: int, name: str):
        if t.dtype != torch.float64 or t.device != self.device or not t.is_contiguous() or t.numel() != numel:
            raise ValueError(f"{name} must be a contiguous float64 tensor with {numel} elements on {self.device}")


class PackedObs:
    """Observations in the packed (optionally cell-sorted, warp-transposed) layout of vggp_obs_pack."""

    def __init__(self, xp, yp, n: int, run_len: int, sorted_by_cell: bool):
        self.xp, self.yp, self.n, self.run_len, self.sorted_by_cell = xp, yp, n, run_len, sorted_by_cell

    def numel(self) -> int:
        return self.n


class GraphedStep:
    """One step as CUDA graph replays (GridPlan.graphed_step).  `.replay()` returns (out, dtheta, dm, dL); the tensors
    are overwritten by every replay."""

    def __init__(self, plan: "GridPlan", group):
        self.plan, self.group = plan, group
        self.front = self.back = None
        self.outs = None

    def replay(self):
        self.front.replay()
        if self.back is not None:
            self.plan.allreduce_gbuf(None if isinstance(self.group, str) else self.group)
            self.back.replay()
        return self.outs


class BinnedObs:
    """Observations in the binned layout of vggp_obs_bin_pack: one device buffer + its host descriptor."""

    def __init__(self, buf: torch.Tensor, desc, elem_size: int = 4):
        self.buf, self.desc, self.elem_size = buf, desc, elem_size
        self.n, self.n_inside = int(desc.n), int(desc.n_inside)
        self.n_tasks, self.n_runs, self.run_cap = int(desc.n_tasks), int(desc.n_runs), int(desc.run_cap)

    def numel(self) -> int:
        return self.n

    @property
    def streamed_bytes(self) -> int:
        """Bytes of observation data the fused kernel reads per launch (padding included)."""
        return int(self.desc.data_elems) * self.elem_size


class BinnedBatch(BinnedObs):
    """One minibatch of an epoch (GridPlan.bin_epoch): a view into the epoch's buffer that every binned entry point takes,
    plus `scale` = n / B, the ell_scale that makes its expected log-likelihood an unbiased estimate of the full one."""

    def __init__(self, buf: torch.Tensor, desc, elem_size: int, scale: float):
        super().__init__(buf, desc, elem_size)
        self.scale = scale


class EpochBins:
    """The binned minibatches of one epoch: one device buffer (`buf`), its descriptor and the P BinnedBatch views."""

    def __init__(self, buf: torch.Tensor, desc, batches):
        self.buf, self.desc, self.batches = buf, desc, batches

    def __len__(self) -> int:
        return len(self.batches)

    def __iter__(self):
        return iter(self.batches)

    def __getitem__(self, b: int) -> BinnedBatch:
        return self.batches[b]


class _DevArray:
    """float64 device array seen through __cuda_array_interface__ (zero-copy view of plan workspace)."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}


def gemm_f64(A: torch.Tensor, B: torch.Tensor, use_mma: bool = True, splitk: int = 1,
             alpha: float = 1.0, beta: float = 0.0, C_in: Optional[torch.Tensor] = None) -> torch.Tensor:
    """C = alpha * A @ B + beta * C through vggp_gemm_f64 (arbitrary strides; optional leading batch dim)."""
    lib = _lib.load()
    if A.dim() == 2:
        A = A.unsqueeze(0)
        B = B.unsqueeze(0)
        squeeze = True
    else:
        squeeze = False
    batch, m, k = A.shape
    n = B.shape[2]
    Cm = torch.zeros(batch, m, n, dtype=torch.float64, device=A.device) if C_in is None else C_in.reshape(batch, m, n)
    _lib.check(lib.vggp_gemm_f64(1 if use_mma else 0, batch, m, n, k, float(alpha),
                                 A.data_ptr(), A.stride(1), A.stride(2), A.stride(0) if batch > 1 else 0,
                                 B.data_ptr(), B.stride(1), B.stride(2), B.stride(0) if batch > 1 else 0,
                                 float(beta), Cm.data_ptr(), Cm.stride(1), Cm.stride(2), Cm.stride(0),
                                 int(splitk), _stream_ptr(A.device)))
    return Cm[0] if squeeze else Cm


class _GriddedELBO(torch.autograd.Function):
    """ELBO(theta, m, L_1..L_D) with the reverse pass computed in the same fused step."""

    @staticmethod
    def forward(ctx, plan: GridPlan, xs, y, ell_scale, group, lengthscale, outputscale, noise, m, *Ls):
        theta = torch.cat([lengthscale.reshape(-1), outputscale.reshape(-1), noise.reshape(-1)]).to(torch.float64).contiguous()
        m64 = m.detach().to(torch.float64).contiguous()
        L64 = torch.cat([L.detach().to(torch.float64).reshape(-1) for L in Ls]).contiguous()
        out, dtheta, dm, dL = plan.step(theta.detach(), m64, L64, xs, y, ell_scale, group)
        D = plan.D
        ctx.D = D
        ctx.shapes = (lengthscale.shape, outputscale.shape, noise.shape, m.shape, [L.shape for L in Ls])
        ctx.dtypes = (lengthscale.dtype, outputscale.dtype, noise.dtype, m.dtype, [L.dtype for L in Ls])
        ctx.L_sizes = plan.L_sizes
        ctx.save_for_backward(dtheta, dm, dL)
        ctx.aux = out
        return out[0].to(m.dtype)

    @staticmethod
    def backward(ctx, grad_out):
        dtheta, dm, dL = ctx.saved_tensors
        D = ctx.D
        go = grad_out.to(torch.float64)
        sl, ss, sn, sm, sL = ctx.shapes
        tl, ts, tn, tm, tL = ctx.dtypes
        g_l = (go * dtheta[:D]).reshape(sl).to(tl)
        g_s = (go * dtheta[D:2 * D]).reshape(ss).to(ts)
        g_n = (go * dtheta[2 * D]).reshape(sn).to(tn)
        g_m = (go * dm).reshape(sm).to(tm)
        gLs = []
        off = 0
        for shp, dt, sz in zip(sL, tL, ctx.L_sizes):
            gLs.append((go * dL[off:off + sz]).reshape(shp).to(dt))
            off += sz
        return (None, None, None, None, None, g_l, g_s, g_n, g_m, *gLs)


def gridded_elbo(plan: GridPlan, xs: List[torch.Tensor], y: torch.Tensor, lengthscale, outputscale, noise, m,
                 Ls: Sequence[torch.Tensor], ell_scale: float = 1.0, group=None) -> torch.Tensor:
    return _GriddedELBO.apply(plan, xs, y, ell_scale, group, lengthscale, outputscale, noise, m, *Ls)
