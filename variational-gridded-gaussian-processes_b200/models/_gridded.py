"""Shared implementation of the gridded sparse variational GP models (D = 1, 2, 3).

What the reference does in `_elbo()` (kronecker_structure.py:249-278): builds dense Kuu = torch.kron(K_1, K_2),
dense Kuf (Khatri-Rao) and N x N evidence matrices for the *collapsed* bound.  Here `_elbo()` is the uncollapsed
bound with explicit variational parameters q(u) = N(m, kron_d L_d L_d^T) (SURVEY.md appendix A) evaluated by
libvggp: per-dimension Cholesky / inverse / Kronecker mode-n products on the grid side and one fused
per-observation kernel; at the optimal q(u) the two bounds coincide (tests/test_oracle_identities.py).

Training-loop API kept from the notebooks (5_gridded_kronecker_structure_models.ipynb:438-446):
    opt = torch.optim.Adam(model.parameters()); loss = -model._elbo(); loss.backward(); opt.step()
"""
import os
from typing import List, Optional, Sequence

import torch
from torch import nn

from .. import _lib
from ..params import DenseNormal, GaussianLikelihood, GriddedMarginals, GriddedNormal, MaternKernel, ScaleKernel
from ..plan import BinnedObs, GridPlan, gridded_elbo
from ..dist import shard_bounds


class GriddedVariationalGP(nn.Module):
    family: int = _lib.B1_ASVGP

    def __init__(self, X: torch.Tensor, y: torch.Tensor, meshes: Sequence[torch.Tensor]):
        super().__init__()
        self.train_inputs = (X,)
        self.train_targets = y
        self.likelihood = GaussianLikelihood()
        self.D = len(meshes)
        self._meshes = [m.detach().to(torch.float32).cpu() for m in meshes]
        if self.D == 1:
            # univariate_structure.py:563-571: a single `kernel`
            self.kernel = ScaleKernel(MaternKernel(nu=0.5))
            self._kernels = [self.kernel]
        else:
            # kronecker_structure.py:30-32: kernel_1, kernel_2 (kernel_3 for the 3-D generalisation)
            self._kernels = []
            for d in range(self.D):
                k = ScaleKernel(MaternKernel(nu=0.5, active_dims=[d]))
                setattr(self, f"kernel_{d + 1}", k)
                self._kernels.append(k)
        self.m_per_dim = [m.numel() - 1 if self.family == _lib.B0_GRIDDED else m.numel() for m in self._meshes]
        M = 1
        for n in self.m_per_dim:
            M *= n
        self.M = M
        # variational parameters: q(u) = N(m, kron_d L_d L_d^T)
        self.variational_mean = nn.Parameter(torch.zeros(M))
        self._chol_names = []
        for d, n in enumerate(self.m_per_dim):
            name = f"variational_chol_{d + 1}"
            setattr(self, name, nn.Parameter(torch.eye(n)))
            self._chol_names.append(name)
        self._plan: Optional[GridPlan] = None
        self._obs = None
        self._packed = None
        self._group = None
        self._n_total = int(y.numel())
        self._terms = None                      # [ELBO, scaled ELL, KL, n_obs] of the last _elbo() (device tensor)
        self.strict_checks = bool(int(os.environ.get("VGGP_STRICT", "0")))   # synchronise and check after every _elbo()

    # ---- parameters as the kernels see them -----------------------------------------------------------------
    def _chols(self) -> List[torch.Tensor]:
        return [getattr(self, n) for n in self._chol_names]

    def _hyper(self):
        ls = torch.cat([k.base_kernel.lengthscale.reshape(-1) for k in self._kernels])
        os_ = torch.cat([k.outputscale.reshape(-1) for k in self._kernels])
        return ls, os_, self.likelihood.noise.reshape(-1)

    # ---- data placement -------------------------------------------------------------------------------------
    def set_train_data(self, X: torch.Tensor, y: torch.Tensor):
        self.train_inputs = (X,)
        self.train_targets = y
        self._n_total = int(y.numel())
        self._obs = None

    def shard_observations(self, rank: int, world: int, group="world"):
        """Keep this rank's contiguous slice of the observations; `_elbo()` then all-reduces the per-observation
        gradient buffer over `group` (SURVEY.md section 8e).  Call on every rank with the same full data set."""
        X, y = self.train_inputs[0], self.train_targets
        lo, hi = shard_bounds(y.numel(), rank, world)
        self._n_total = int(y.numel())
        self.train_inputs = (X[lo:hi],)
        self.train_targets = y[lo:hi]
        self._group = group if world > 1 else None
        self._obs = None

    def _device_dtype(self):
        p = self.variational_mean
        if p.device.type != "cuda":
            raise RuntimeError("the ELBO path runs only on CUDA (sm_100a): move the model with .to('cuda'); "
                               "there is no CPU fallback")
        return p.device, p.dtype

    def _ensure_plan(self):
        device, dtype = self._device_dtype()
        if self._plan is None or self._plan.device != device or self._plan.obs_dtype != dtype:
            self._plan = GridPlan(self.family, self._meshes, dtype, device)
            self._obs = None
        if self._obs is None:
            X = self.train_inputs[0]
            X = X.reshape(X.shape[0], -1) if X.dim() > 1 else X.reshape(-1, 1)
            if X.shape[1] != self.D:
                raise ValueError(f"X must have {self.D} columns")
            Xd = X.to(device=device, dtype=dtype)
            xs = [Xd[:, d].contiguous() for d in range(self.D)]       # structure of arrays, made once
            y = self.train_targets.reshape(-1).to(device=device, dtype=dtype).contiguous()
            self._obs = (xs, y)
            # one-time layout pass (setup, X is constant over optimisation steps).  Default: per-cell runs grouped into warp
            # tasks (B1: k_obs_b1_binned; B0, D <= 2: scan form of the cell-integrated features), DESIGN.md sections 8 and 10.
            # VGGP_OBS_LAYOUT=packed selects the round-1 layouts (B1: cell-sorted packed runs, B0: plain arrays through the
            # dense-feature kernel), kept as cross-checks.
            layout = os.environ.get("VGGP_OBS_LAYOUT", "binned")
            if self.family == _lib.SVGP_MARKOV:
                self._packed = self._plan.bin(xs, y)        # the only observation layout of the Markov form
            elif self.family in (_lib.SVGP_GRID, _lib.VFF_GRID):
                self._packed = None                 # dense-feature kernel: plain arrays
            elif layout == "binned" and not (self.family != _lib.B1_ASVGP and self.D > 2):
                self._packed = self._plan.bin(xs, y)
            elif self.family != _lib.B1_ASVGP:
                self._packed = None
            else:
                self._packed = self._plan.pack(xs, y, sort_by_cell=True)
        return self._plan

    # ---- the hot path ---------------------------------------------------------------------------------------
    def _raise_if_failed(self, wait: bool):
        """The reference raises LinAlgError where a covariance stops being positive definite (gpytorch's Cholesky;
        61_envisat_gulfstream_experiment.ipynb:746 catches it).  The library sets a device flag instead of synchronising
        the step; it is copied to pinned memory behind every step and turned into the exception here -- at the next
        `_elbo()` that finds the copy complete, or immediately with `strict_checks` / `check_factorisation()`."""
        if self._plan is None:
            return
        flag = self._plan.poll_info(wait)
        if flag is None:
            return
        if flag != 0:
            raise torch.linalg.LinAlgError(
                f"the per-dimension factor K_{flag} = Kuu along dimension {flag} is not positive definite at the current "
                "hyper-parameters (Cholesky / pivot recurrence failed); the ELBO of that step is invalid")

    def set_deterministic(self, on: bool = True) -> None:
        """Bitwise run-to-run reproducible `_elbo()` values and gradients (vggp_set_deterministic; B1 family over the default
        binned layout, full batch).  The reference is deterministic only because it is single-threaded CPU code."""
        self._ensure_plan().set_deterministic(on)

    def check_factorisation(self) -> None:
        """Synchronise and raise torch.linalg.LinAlgError if the last `_elbo()` hit a non-positive-definite factor."""
        self._raise_if_failed(wait=True)

    def _elbo(self, batch: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Evidence lower bound (0-dim tensor with grad_fn).  `batch`: optional index tensor / slice selecting a
        minibatch of this rank's observations; the expected log-likelihood is rescaled by N / B."""
        self._raise_if_failed(wait=False)
        plan = self._ensure_plan()
        if self._packed is not None:
            xs, y = self._packed, None
        else:
            xs, y = self._obs
        scale = 1.0
        if batch is not None:
            if self.family == _lib.SVGP_MARKOV:
                raise NotImplementedError("minibatches of the Markov SVGP form need the plain-array per-observation path, which "
                                          "this family does not have yet: call _elbo() on the full (sharded) data set")
            xs = [x[batch].contiguous() for x in self._obs[0]]
            y = self._obs[1][batch].contiguous()
            n_local = self._obs[1].numel()
            scale = float(n_local) / float(max(1, y.numel()))
        ls, os_, noise = self._hyper()
        elbo = gridded_elbo(plan, xs, y, ls, os_, noise, self.variational_mean, self._chols(),
                            ell_scale=scale, group=self._group)
        self._terms = plan.last_out
        plan.arm_info_check()
        if self.strict_checks:
            self._raise_if_failed(wait=True)
        return elbo

    def elbo_terms(self) -> torch.Tensor:
        """[ELBO, scaled expected log-likelihood, KL, n_obs over all ranks] of the last `_elbo()` call (float64 device
        tensor, no synchronisation)."""
        if self._terms is None:
            raise RuntimeError("elbo_terms() needs a previous _elbo() call")
        return self._terms

    # ---- variational distribution ---------------------------------------------------------------------------
    def q_u(self, optimal: bool = False):
        """q(u).  Default: the *learned* variational distribution N(m, kron_d L_d L_d^T) (GriddedNormal).  `optimal=True`:
        the reference's closed form (its `q_u()`, gridded_kronecker_structure.py:903-916), dense -- see `q_u_optimal`.
        The two agree where the learned q(u) has converged (tests/test_oracle_identities.py)."""
        if optimal:
            return self.q_u_optimal()
        Ss = []
        for L in self._chols():
            Lt = torch.tril(L.detach())
            Ss.append(Lt @ Lt.T)
        return GriddedNormal(self.variational_mean.detach(), Ss)

    MEANOPT_MAX_ITER = 20000

    @torch.no_grad()
    def set_optimal_mean(self, rtol: float = 1e-10, max_iter: Optional[int] = None, preconditioner: str = "jacobi") -> dict:
        """Load the optimal variational mean at the current hyper-parameters into `variational_mean`: the m that maximises
        the ELBO for fixed theta and S, which is the mean of the reference's q_u() (m* = Kuu Sigma^-1 Kuf y / noise), at any
        grid size.  One pass over the binned observations assembles a 3^D-stencil system, preconditioned conjugate
        gradients solve it from the current mean (include/vggp.h, vggp_meanopt_*).  B1 and Markov SVGP families.
        `max_iter` defaults to MEANOPT_MAX_ITER = 20000.  `preconditioner`:
          "jacobi"     (default) measured on one B200 to rtol 1e-8 from m = 0 (float32 track observations,
                       profiles/optimal_mean/): 512 x 512 points, 2^26 observations: B1 678, Markov 59 iterations; 2^22
                       observations: B1 3054, Markov 283; 64 x 64 x 16 points, 2^20 observations: Markov 16046, B1 not
                       converged after 60000.
          "kronecker"  kron_d (F_d + g I)^-1 of the per-dimension prior factors, applied exactly by D tridiagonal sweeps;
                       it converges on 3-D B1 grids.  Same data on one B200 (profiles/optimal_mean_kron/):
                       512 x 512 points, 2^26 observations: B1 100 iterations (7.1 ms, Jacobi 15.8 ms), Markov 37 (3.1 ms,
                       Jacobi 1.4 ms); 256 x 256 x 64 points: B1 7855 iterations (6.0 s), Markov relres 2.1e-7 after 20000.
                       Float64 oracle counts with 2^22 / 2^20 observations: 512 x 512 B1 196, Markov 66; 64 x 64 x 16 B1 990.
        Any other value raises ValueError.  Returns {"iterations", "relres"}; raises RuntimeError, leaving
        `variational_mean` unchanged, if the solve stops above `rtol`."""
        if preconditioner not in ("jacobi", "kronecker"):
            raise ValueError(f"preconditioner must be 'jacobi' or 'kronecker', not {preconditioner!r}")
        if self.family not in (_lib.B1_ASVGP, _lib.SVGP_MARKOV):
            raise NotImplementedError("set_optimal_mean() needs the 3^D-stencil system of the B1 and Markov SVGP families; "
                                      "for this family use set_optimal_q() (dense, M <= 4096)")
        if self._group is not None:
            raise NotImplementedError("set_optimal_mean() on a sharded model would need the rank sum of the assembled "
                                      "system, which is not implemented")
        plan = self._ensure_plan()
        plan.grid_forward(self._theta(), self.variational_mean.detach().to(torch.float64).contiguous(),
                          torch.cat([c.detach().to(torch.float64).reshape(-1) for c in self._chols()]).contiguous())
        binned = self._binned_for_optimal_q(plan)
        # the B1 system does not depend on theta: assembled once per plan and data set; the Markov one on every call
        if self.family != _lib.B1_ASVGP or getattr(plan, "_mo_obs", None) is not self._obs:
            plan.meanopt_assemble(binned)
            plan._mo_obs = self._obs if self.family == _lib.B1_ASVGP else None
        m, iters, relres = plan.meanopt_solve(rtol, self.MEANOPT_MAX_ITER if max_iter is None else max_iter, preconditioner)
        if not relres <= rtol:
            raise RuntimeError(f"set_optimal_mean(): conjugate gradients stopped after {iters} iterations at relative residual "
                               f"{relres:.3e} > rtol = {rtol:.1e}; variational_mean is unchanged")
        self.variational_mean.copy_(m.to(self.variational_mean.dtype))
        return {"iterations": iters, "relres": relres}

    def _binned_for_optimal_q(self, plan):
        """The binned layout of the observations (VGGP_OBS_LAYOUT=packed: binned once, for the optimal-q methods only)."""
        if isinstance(self._packed, BinnedObs):
            return self._packed
        if getattr(plan, "_mo_binned", (None,))[0] is not self._obs:
            plan._mo_binned = (self._obs, plan.bin(*self._obs))
        return plan._mo_binned[1]

    @torch.no_grad()
    def set_optimal_covariance(self, rtol: float = 1e-8, max_sweeps: int = 100) -> dict:
        """Load the ELBO-optimal Kronecker-factored covariance S = kron_d tril(L_d) tril(L_d)^T at the current
        hyper-parameters and variational mean into the `variational_chol_*` factors, at any grid size.  With everything
        else fixed the ELBO is strictly concave in one S_d and its maximiser has a closed form built from a tridiagonal matrix
        (include/vggp.h, vggp_covopt_update; DESIGN.md section 4, K1s); this method cycles d = 0..D-1 (coordinate ascent,
        the ELBO cannot decrease), each update after a grid forward and one pass over the binned observations, all-reduced
        over the model's process group when sharded.  It stops after the first sweep whose summed normalised factor change
        ||L_new / ||L_new|| - L_old / ||L_old||||_F is <= rtol.  B1 and Markov SVGP families.

        The result is the optimum within the Kronecker family, exact for D = 1 (the reference's S* = Kuu Sigma^-1 Kuu).
        `set_optimal_q()` instead loads the Kronecker product nearest in the Frobenius norm to the unconstrained S* (dense,
        M <= 4096, D <= 2), which is not the ELBO's optimum in this family for D = 2.  m and S separate in the bound, so
        `set_optimal_mean()` followed by this method gives the ELBO-optimal q(u) of the family.

        Sweeps to rtol 1e-8 from L_d = I, float64 oracle (Markov features, 4000 - 20000 observations): D = 1 one update,
        D = 2 11 - 18 sweeps, D = 3 15 - 25 sweeps.  One B200 (1000 W), 2^26 float32 track observations
        (profiles/optimal_cov/): 512 x 512 points B1 15 sweeps (28 ms), 256 x 256 x 64 B1 19 sweeps (35 ms); the Markov
        change stalls near 3e-8 (reached after 11 and 17 sweeps): with float32 observations the band sums change in their last
        bits from one data pass to the next, so use rtol >= 1e-7 there (DESIGN.md section 4, K1s).
        Returns {"sweeps", "change" (of the last sweep), "elbo" (after the update)}.  Raises RuntimeError after `max_sweeps`
        sweeps above `rtol`, and torch.linalg.LinAlgError if an update meets a matrix that is not positive definite; both
        leave the factors as they were."""
        if self.family not in (_lib.B1_ASVGP, _lib.SVGP_MARKOV):
            raise NotImplementedError("set_optimal_covariance() needs the tridiagonal update of the B1 and Markov SVGP "
                                      "families; for this family use set_optimal_q() (dense, M <= 4096)")
        plan = self._ensure_plan()
        binned = self._binned_for_optimal_q(plan)
        group = None if self._group is None or isinstance(self._group, str) else self._group
        theta = self._theta()
        m = self.variational_mean.detach().to(torch.float64).contiguous()
        L = torch.cat([c.detach().to(torch.float64).reshape(-1) for c in self._chols()]).contiguous()
        change = torch.zeros(1, dtype=torch.float64, device=plan.device)
        sweeps, last = 0, float("inf")
        while sweeps < max_sweeps:
            change.zero_()
            for d in range(self.D):
                plan.grid_forward(theta, m, L)
                plan.obs_fwd_bwd(binned)
                if self._group is not None:
                    plan.allreduce_gbuf(group)
                plan.covopt_update(d, plan.gbuf, 1.0, L, change)
            sweeps += 1
            last = float(change.item())
            if not last < float("inf"):
                raise torch.linalg.LinAlgError(
                    "set_optimal_covariance(): an update met a tridiagonal matrix that is not positive definite (is a "
                    "factor L_d singular?); the variational factors are unchanged")
            if last <= rtol:
                break
        else:
            raise RuntimeError(f"set_optimal_covariance(): the factor change is {last:.3e} > rtol = {rtol:.1e} after "
                               f"{sweeps} sweeps; the variational factors are unchanged")
        out = plan.step(theta, m, L, binned, None, 1.0, self._group)[0]
        off = 0
        for c in self._chols():
            n = c.numel()
            c.copy_(L[off:off + n].reshape(c.shape).to(c.dtype))
            off += n
        return {"sweeps": sweeps, "change": last, "elbo": float(out[0].item())}

    # ---- the reference's closed-form (collapsed) quantities: dense M x M algebra, small problems only -------------
    DENSE_LIMIT = 4096          # largest M for which dense M x M matrices are formed (128 MiB in float64)

    def _dense_guard(self, what: str) -> None:
        if self.M > self.DENSE_LIMIT:
            raise RuntimeError(f"{what} forms dense {self.M} x {self.M} matrices (the reference's algorithm); it is offered up to "
                               f"M = {self.DENSE_LIMIT}.  Use the structured path instead: _elbo(), q_u(), posterior(), q_v()")

    def _X2d(self) -> torch.Tensor:
        X = self.train_inputs[0]
        return X.reshape(X.shape[0], -1) if X.dim() > 1 else X.reshape(-1, 1)

    def _gram_and_moment(self, chunk: int = 1 << 16):
        """A = Kuf Kuf^T (M x M) and b = Kuf y (M), accumulated over chunks of observations (Kuf itself is M x N)."""
        plan = self._ensure_plan()
        X, y = self._X2d(), self.train_targets.reshape(-1)
        A = torch.zeros(self.M, self.M, dtype=torch.float64, device=plan.device)
        b = torch.zeros(self.M, dtype=torch.float64, device=plan.device)
        for lo in range(0, X.shape[0], chunk):
            Kuf = self._Kuf(X[lo:lo + chunk]).to(torch.float64)
            A += Kuf @ Kuf.T
            b += Kuf @ y[lo:lo + chunk].to(device=plan.device, dtype=torch.float64)
        return A, b

    def _sigma(self) -> torch.Tensor:
        """Sigma = Kuu + Kuf Kuf^T / noise (kronecker_structure.py:134-150, univariate_structure.py:104-120), dense."""
        self._dense_guard("_sigma()")
        A, _ = self._gram_and_moment()
        noise = self.likelihood.noise.detach().to(torch.float64).reshape(()).to(A.device)
        return self._Kuu() + A / noise

    def q_u_optimal(self) -> DenseNormal:
        """The analytically optimal q(u) = N(m*, S*) of the collapsed bound, as the reference's `q_u()` / `q_v()` return it
        (gridded_kronecker_structure.py:903-916, 1409-1433; univariate_structure.py:693-717):
            m* = Kuu Sigma^-1 Kuf y / noise,   S* = Kuu Sigma^-1 Kuu   (symmetrised)
        Raises torch.linalg.LinAlgError if Sigma is not positive definite, like the reference's Cholesky."""
        self._dense_guard("q_u_optimal()")
        A, b = self._gram_and_moment()
        noise = self.likelihood.noise.detach().to(torch.float64).reshape(()).to(A.device)
        Kuu = self._Kuu()
        Ls = torch.linalg.cholesky(Kuu + A / noise)
        mean = Kuu @ torch.cholesky_solve(b.unsqueeze(-1), Ls).squeeze(-1) / noise
        cov = Kuu @ torch.cholesky_solve(Kuu, Ls)
        return DenseNormal(mean, 0.5 * (cov + cov.T))

    @torch.no_grad()
    def set_optimal_q(self) -> None:
        """Load the reference's closed-form q(u) into the variational parameters: m <- m*, and L_d <- Cholesky factors of
        the Kronecker product nearest to S* in the Frobenius norm (Van Loan & Pitsianis; exact for D = 1, where the
        uncollapsed bound then equals the reference's collapsed `_elbo()`).  D <= 2."""
        if self.D > 2:
            raise NotImplementedError("set_optimal_q() is offered for D <= 2, the dimensions the reference has")
        q = self.q_u_optimal()
        self.variational_mean.copy_(q.mean.to(self.variational_mean.dtype))
        S = q.covariance_matrix
        if self.D == 1:
            factors = [S]
        else:
            n1, n2 = self.m_per_dim
            R = S.reshape(n1, n2, n1, n2).permute(0, 2, 1, 3).reshape(n1 * n1, n2 * n2)
            v = torch.eye(n2, dtype=S.dtype, device=S.device).reshape(-1)
            for _ in range(30):                  # power iteration for the leading singular pair of the rearrangement
                u = R @ v
                u = u / u.norm()
                v = R.T @ u
                sig = v.norm()
                v = v / sig
            S1, S2 = u.reshape(n1, n1), v.reshape(n2, n2)
            if torch.trace(S1) < 0:
                S1, S2 = -S1, -S2
            S1 = 0.5 * (S1 + S1.T) * sig.sqrt()
            S2 = 0.5 * (S2 + S2.T) * sig.sqrt()
            factors = [S1, S2]
        for name, Sd in zip(self._chol_names, factors):
            getattr(self, name).copy_(torch.linalg.cholesky(Sd).to(getattr(self, name).dtype))

    def prior(self, x: torch.Tensor) -> DenseNormal:
        """GP prior over f(x): zero mean, product Matern-1/2 kernel (kronecker_structure.py:90-104); dense N* x N*."""
        x = x.reshape(x.shape[0], -1) if x.dim() > 1 else x.reshape(-1, 1)
        ls, os_, _ = self._hyper()
        K = torch.ones(x.shape[0], x.shape[0], dtype=x.dtype, device=x.device)
        for d in range(self.D):
            dist = (x[:, d, None] - x[None, :, d]).abs()
            K = K * (os_[d].detach().to(x) * torch.exp(-dist / ls[d].detach().to(x)))
        return DenseNormal(torch.zeros(x.shape[0], dtype=x.dtype, device=x.device), K)

    def posterior_dense(self, x: torch.Tensor, optimal: bool = False) -> DenseNormal:
        """q(f(x*)) with its full N* x N* covariance (kronecker_structure.py:199-230), small problems only:
            mean = Kuf*^T Kuu^-1 m,   cov = K** - Kuf*^T Kuu^-1 Kuf* + Kuf*^T Kuu^-1 S Kuu^-1 Kuf*
        with (m, S) the learned q(u), or the reference's optimal one (`optimal=True`, its Sigma^-1 form)."""
        self._dense_guard("posterior_dense()")
        q = self.q_u_optimal() if optimal else self.q_u()
        Kuu = self._Kuu()
        Ks = self._Kuf(x).to(torch.float64)
        Lk = torch.linalg.cholesky(Kuu)
        B = torch.cholesky_solve(Ks, Lk)                                  # Kuu^-1 Kuf*
        S = q.covariance_matrix.to(torch.float64)
        mean = B.T @ q.mean.to(torch.float64)
        cov = self.prior(x.to(device=Kuu.device, dtype=torch.float64)).covariance_matrix - Ks.T @ B + B.T @ S @ B
        return DenseNormal(mean, cov)

    # ---- predictions (kronecker_structure.py:199-247, marginals only) --------------------------------------------
    def posterior(self, x: torch.Tensor) -> GriddedMarginals:
        """q(f(x*)): marginal mean and variance at the test points x (N*, D) under the current q(u) and
        hyper-parameters.  B1 family: 2^D-point stencil; B0 family: scan form of the cell-integrated features
        (csrc/b0scan.cuh), O(1) per point as well."""
        plan = self._ensure_plan()
        theta = self._theta()
        m = self.variational_mean.detach().to(torch.float64).contiguous()
        L = torch.cat([c.detach().to(torch.float64).reshape(-1) for c in self._chols()]).contiguous()
        plan.grid_forward(theta, m, L)
        x = x.reshape(x.shape[0], -1) if x.dim() > 1 else x.reshape(-1, 1)
        xs = [x[:, d].contiguous() for d in range(self.D)]
        mean, var = plan.predict(xs)
        return GriddedMarginals(mean, var)

    def posterior_predictive(self, x: torch.Tensor) -> GriddedMarginals:
        """p(y* | y): the posterior marginals pushed through the Gaussian likelihood (variance + noise)."""
        post = self.posterior(x)
        return GriddedMarginals(post.mean, post.variance + self.likelihood.noise.detach().to(post.variance.dtype).reshape(()))

    # ---- reference plug-in points (dense, small problems only) -------------------------------------------------
    def _theta(self) -> torch.Tensor:
        ls, os_, noise = self._hyper()
        return torch.cat([ls, os_, noise]).detach().to(torch.float64).contiguous()

    def _Kuu_along_dim(self, dim: int) -> torch.Tensor:
        plan = self._ensure_plan()
        theta = self._theta()
        m = self.variational_mean.detach().to(torch.float64).contiguous()
        L = torch.cat([c.detach().to(torch.float64).reshape(-1) for c in self._chols()]).contiguous()
        plan.grid_forward(theta, m, L)
        return plan.workspace(_lib.WS_KRAW, dim)

    def _Kuf_along_dim(self, dim: int, x: torch.Tensor) -> torch.Tensor:
        plan = self._ensure_plan()
        return plan.features_dense(dim, x, self._theta())

    def _Kuu(self) -> torch.Tensor:
        out = self._Kuu_along_dim(0)
        for d in range(1, self.D):
            out = torch.kron(out, self._Kuu_along_dim(d))
        return out

    def _Kuf(self, x: torch.Tensor) -> torch.Tensor:
        x = x.reshape(x.shape[0], -1) if x.dim() > 1 else x.reshape(-1, 1)
        feats = [self._Kuf_along_dim(d, x[:, d].contiguous()) for d in range(self.D)]
        out = feats[0]
        for f in feats[1:]:
            out = (out[:, None, :] * f[None, :, :]).reshape(-1, f.shape[-1])
        return out

    # ---- initialisers (kronecker_structure.py:34-88; evident intent, see SURVEY.md appendix B) ----------------
    def non_informative_initialise(self, lmbda: float, kappa: float) -> None:
        X = self.train_inputs[0]
        X = X.reshape(X.shape[0], -1) if X.dim() > 1 else X.reshape(-1, 1)
        y = self.train_targets
        for d, k in enumerate(self._kernels):
            k.outputscale = y.var()
            k.base_kernel.lengthscale = X[:, d].std() / lmbda
        mean_os = sum(k.outputscale for k in self._kernels) / len(self._kernels)
        self.likelihood.noise = mean_os / (kappa ** 2)

    def informative_initialise(self, prior_amplitude: float, lmbda: float) -> None:
        X = self.train_inputs[0]
        X = X.reshape(X.shape[0], -1) if X.dim() > 1 else X.reshape(-1, 1)
        y = self.train_targets
        for d, k in enumerate(self._kernels):
            k.outputscale = (torch.tensor(prior_amplitude) / 2) ** 2
            k.base_kernel.lengthscale = X[:, d].std() / lmbda
        mean_os = sum(k.outputscale for k in self._kernels) / len(self._kernels)
        self.likelihood.noise = y.var() - mean_os


def b0_cell_cov(delta32: torch.Tensor, m: int, lengthscale: torch.Tensor, outputscale: torch.Tensor) -> torch.Tensor:
    """Cov[v_i, v_j] of the B0 cell integrals of a Matern-1/2 process: the Toeplitz matrix of `_Kvv_along_dim`
    (gridded_kronecker_structure.py:847-885; gridded_univariate_structure.py:612-646), float64, with the reference's
    float32 rounding of (k +- 1) * delta (int64 tensor times 0-dim float32)."""
    k = torch.arange(m)
    d32 = delta32.detach().to("cpu", torch.float32)
    l = lengthscale.detach().to("cpu", torch.float64).reshape(())
    s2 = outputscale.detach().to("cpu", torch.float64).reshape(())
    km, kp, k0 = ((k - 1) * d32).to(torch.float64), ((k + 1) * d32).to(torch.float64), (k * d32).to(torch.float64)
    row = torch.exp(-km / l) + torch.exp(-kp / l) - 2 * torch.exp(-k0 / l)
    dl = d32.to(torch.float64) / l
    row[0] = 2 * (torch.exp(-dl) + dl - 1)
    idx = (k[:, None] - k[None, :]).abs()
    return row[idx] * (l * l * s2)


def linspace_mesh(lims, n_knots: int) -> torch.Tensor:
    """float32 torch.linspace without dtype, exactly as the reference builds its meshes."""
    return torch.linspace(lims[0], lims[1], n_knots)


def padded_b0_mesh(lims, n_b0_splines: int, padding_factor: int):
    """gridded_kronecker_structure.py:707-720: B0 mesh plus `padding_factor` extra knots each side, built from
    Python floats of float32 values."""
    b0 = torch.linspace(lims[0], lims[1], n_b0_splines + 1)
    d = b0[1] - b0[0]
    left = torch.tensor([(b0[0] - (i * d)).item() for i in range(padding_factor, 0, -1)])
    right = torch.tensor([(b0[-1] + (i * d)).item() for i in range(1, padding_factor + 1)])
    return b0, d, torch.cat((left, b0, right))
