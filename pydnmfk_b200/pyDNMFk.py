"""NMFk: automatic rank estimation from a perturbation ensemble of ``PyNMF`` fits.

Mirrors ``pyDNMFk/pyDNMFk.py``: ``sample`` (:8-67), ``PyNMFk.fit`` (:169-212), ``pynmfk_per_k`` (:214-258: perturbation
loop, result stacking, clustering + silhouettes, W-fixed regression fit, per-k results) and ``pvalueAnalysis`` (:261-299).
The data shard, the ensemble tensors and the clustering stay on the device; only k x P-sized statistics go to the host.
"""
import os

import numpy as np
import numpy
import torch

from . import config   # noqa: F401
from . import device as D
from .pyDNMF import *  # noqa: F401,F403
from .pyDNMF import PyNMF
from .sparse import is_sparse_input
from .utils import comm_timing, var_init, Checkpoint


class sample():
    """Perturbed copy of a data shard (pyDNMFk.py:8-67).

    ``uniform``: X * (1 + nv + 2 nv u), u ~ U[0,1) -- what the reference's code does (its docstring
    says (1-eps, 1+eps); the code wins, SURVEY A7).  The random field is drawn on the host from the
    process-global legacy numpy stream (seeded with ``seed`` exactly like the reference, so
    ``PyNMF.init_factors`` continues the same stream, SURVEY A8) and the multiply runs on the
    device, bit-identical to numpy's fp32/fp64 result.
    ``poisson``: host ``np.random.poisson`` (same stream), uploaded.
    """

    @comm_timing()
    def __init__(self, data, noise_var, method, seed=None):
        if isinstance(data, torch.Tensor) and data.dtype in (torch.float16, torch.bfloat16):
            raise ValueError('sample: a 16-bit data shard (params.a_storage) is not supported: the perturbed matrix would '
                             'need its own rounding rule; perturb the float32 data instead')
        self.X = data
        self.noise_var = noise_var
        self.seed = seed
        if self.seed != None:  # noqa: E711
            np.random.seed(self.seed)
        self.method = method
        self.X_per = 0

    def _np_dtype(self):
        return np.dtype(str(self.X.dtype).replace('torch.', ''))

    @comm_timing()
    def randM(self):
        ops = D.default_ops()
        dt = self._np_dtype()
        U = np.random.random_sample(tuple(self.X.shape)).astype(dt)
        Xd = D.to_device(self.X)
        self.X_per = ops.perturb_uniform(Xd, D.to_device(U), self.noise_var)

    @comm_timing()
    def poisson(self):
        Xh = self.X.cpu().numpy() if isinstance(self.X, torch.Tensor) else np.asarray(self.X)
        self.X_per = D.to_device(np.random.poisson(Xh).astype(Xh.dtype))

    @comm_timing()
    def fit(self):
        """Returns the perturbed shard: a CUDA tensor if the input was one, else a numpy array."""
        if self.method == 'uniform':
            self.randM()
        elif self.method == 'poisson':
            self.poisson()
        if isinstance(self.X_per, torch.Tensor) and not isinstance(self.X, torch.Tensor):
            return self.X_per.cpu().numpy()
        return self.X_per


class PyNMFk():
    r"""Automatic rank estimation (pyDNMFk.py:126-299).

    ``fit()`` sweeps ``k = start_k .. end_k``: per k a perturbation ensemble of ``PyNMF`` fits (``fit_ensemble``),
    clustering + silhouettes of the stacked factors (``dist_clustering.custom_clustering``), a W-fixed regression fit
    from the cluster medians (``fit_regression``) and the per-k statistics written under
    ``results_path/<fname>/<k>/``; then ``pvalueAnalysis`` picks the rank.  ``fit_ensemble`` returns the factors stacked
    exactly as the reference stacks them: ``Wall (m_loc, k, P)``, ``Hall (k, n_loc, P)``, ``recon_err [P]``.
    """

    @comm_timing()
    def __init__(self, A_ij, factors=None, params=None):
        if getattr(params, 'a_storage', None) is not None:
            raise ValueError('params.a_storage is not supported by PyNMFk: the perturbed ensemble would need its own '
                             'rounding rule; fit the rounded matrix in float32 instead')
        if is_sparse_input(A_ij):
            raise ValueError('PyNMFk does not take a sparse A_ij: its perturbations change every entry of the matrix, '
                             'zeros included, and their random stream is part of the reference parity; densify the shard')
        self.A_ij = A_ij
        self.local_m, self.local_n = self.A_ij.shape
        self.params = params
        self.comm1 = self.params.comm1
        self.rank = self.comm1.rank
        if getattr(self.params, 'grid', None):                       # pyDNMFk.py:132-135: params.grid wins over p_r / p_c
            self.params.p_r, self.params.p_c = self.params.grid[0], self.params.grid[1]
        if getattr(self.params, 'k_range', None):                    # pyDNMFk.py:156-160
            self.params.start_k, self.params.end_k = self.params.k_range[0], self.params.k_range[1]
        self.p_r, self.p_c = self.params.p_r, self.params.p_c
        self.fpath = var_init(self.params, 'fpath', default='data/')
        self.fname = var_init(self.params, 'fname', default='A_')
        self.p = self.p_r * self.p_c
        self.start_k = var_init(self.params, 'start_k', default=1)
        self.end_k = var_init(self.params, 'end_k', default=10)
        self.params.start_k, self.params.end_k = self.start_k, self.end_k      # pvalueAnalysis reads them back
        self.step_k = var_init(self.params, 'step_k', default=1)
        self.sill_thr = var_init(self.params, 'sill_thr', default=0.9)
        self.verbose = var_init(self.params, 'verbose', default=False)
        self.sampling = var_init(self.params, 'sampling', default='uniform')
        self.perturbations = var_init(self.params, 'perturbations', default=20)
        self.noise_var = var_init(self.params, 'noise_var', default=.03)
        self.params.results_path = var_init(self.params, 'results_path', default='results/')
        self.Hall = 0
        self.Wall = 0
        self.recon_err = 0
        self.AvgH = 0
        self.AvgG = 0
        self.col_err = 0
        self.clusterSilhouetteCoefficients, self.avgSilhouetteCoefficients = 0, 0
        self.L_errDist = 0
        self.avgErr = 0
        self.start_time = 0
        self.end_time = 0
        self.params.checkpoint = var_init(self.params, 'checkpoint', default=True)
        self.params.rank = self.rank
        self.params.flag = 0      # 1: all perturbations of a k done, 2: clustered, 3: results saved (pyDNMFk.py:165)
        self.cp = Checkpoint(self.params.checkpoint, self.params)
        # keep the shard on the device across all perturbations
        self._A_dev = D.to_device(self.A_ij)
        self._numpy_in = not isinstance(self.A_ij, torch.Tensor)

    def _spread(self):
        """Replica mode: ``params.ensemble_parallel`` and a world larger than the p_r x p_c factorization grid.  The
        world is cut into ``world.size / (p_r p_c)`` replica groups; every group holds the whole matrix on its own
        grid and takes every n_groups-th perturbation (no data-path collective between groups)."""
        world = self.comm1
        return (bool(getattr(self.params, 'ensemble_parallel', False)) and world.size > self.p
                and world.size % self.p == 0)

    def _enter_group(self):
        """Swap the communicators on ``params`` for this rank's replica group (a private p_r x p_c grid)."""
        from .dist_comm import MPI_comm, split_into_groups
        world = self.comm1
        saved = (self.params.comm1, self.params.comm, self.params.row_comm, self.params.col_comm)
        gcomm, self._group_index, self._n_groups = split_into_groups(world, self.p)
        grid = MPI_comm(gcomm, self.p_r, self.p_c)
        self.params.comm1, self.params.comm = gcomm, grid
        self.params.row_comm, self.params.col_comm = grid.cart_1d_row(), grid.cart_1d_column()
        return saved

    def _leave_group(self, saved):
        self.params.comm1, self.params.comm, self.params.row_comm, self.params.col_comm = saved

    def fit_ensemble(self, k):
        """pyDNMFk.py:226-238 for one k.

        The reference runs the perturbations one after another on the whole grid.  With ``params.ensemble_parallel``
        set and a 1x1 factorization grid inside a larger world (every rank holds the full matrix on its own GPU), the
        perturbations are independent replicas: rank r takes perturbations r, r+size, ... on a private size-1
        communicator (no data-path collective) and the factors are exchanged once at the end.  Results are identical to
        the sequential order because every perturbation re-seeds its own RNG stream (seed = 1000 * perturbation).
        """
        self.k = k
        self.params.k = k
        world = self.params.comm1
        spread = self._spread()
        todo = list(range(self.perturbations))
        saved = None
        if spread:
            saved = self._enter_group()
            todo = todo[self._group_index::self._n_groups]
        mine = {}
        pending = []
        for perturbation in todo:
            if self.rank == 0 and self.verbose:
                print('Current perturbation =', perturbation)
            data = sample(data=self._A_dev, noise_var=self.noise_var, method=self.sampling,
                          seed=perturbation * 1000).fit()
            self.params.W_update = True
            fit = PyNMF(data, factors=None, params=self.params)
            if self.sampling == 'uniform' and fit._resident_ok():
                # tiny shard: the update loops of all perturbations run as ONE launch, one CTA per fit (the
                # perturbations share A's zero pattern, hence the pruned shapes and the masks left on params)
                pending.append((perturbation, fit))
                continue
            mine[perturbation] = fit.fit()
            if not spread:
                self.cp._save_checkpoint(self.params.flag, perturbation, self.k)
        if pending:
            fits = [f for _, f in pending]
            shapes = {(tuple(f.A_ij.shape), f.A_ij.stride(0)) for f in fits}
            if len(shapes) == 1:
                D.default_ops().mu_fit_resident([f.A_ij for f in fits], [f._get_factors()[0] for f in fits],
                                                [f._get_factors()[1] for f in fits], fits[0].norm, True, 0, fits[0].itr,
                                                fits[0].eps)
            else:
                for f in fits:
                    f._run_loop()
            for perturbation, f in pending:
                mine[perturbation] = f._finish()
                if not spread:
                    self.cp._save_checkpoint(self.params.flag, perturbation, self.k)
        if spread:
            self._leave_group(saved)
            # every rank needs ITS block of every perturbation: take the parts of the ranks that sit at the same
            # position of their replica group
            pos = world.rank % self.p
            merged = {}
            parts = world.allgather((pos, {p: (W.cpu().numpy(), H.cpu().numpy(), e) for p, (W, H, e) in mine.items()}))
            for other_pos, part in parts:
                if other_pos == pos:
                    merged.update(part)
            mine = {p: (D.to_device(W), D.to_device(H), e) for p, (W, H, e) in merged.items()}
        results = [mine[p] for p in range(self.perturbations)]
        # Wall[:, :, p] = W_p (hstack + reshape(order='F'), pyDNMFk.py:234-235); Hall is the reference's vstack followed
        # by a C-order reshape to (k, n, P) (pyDNMFk.py:236-237) -- both kept on the device for the clustering
        self._Wall_dev = torch.stack([r[0] for r in results], dim=2).contiguous()
        Hs = torch.cat([r[1] for r in results], dim=0)
        self._Hall_dev = Hs.reshape(self.k, Hs.shape[1], self.perturbations).contiguous()
        self.Wall = self._Wall_dev.cpu().numpy()
        self.Hall = self._Hall_dev.cpu().numpy()
        self.recon_err = [r[2] for r in results]
        return self.Wall, self.Hall, self.recon_err

    def fit_regression(self, AvgW, AvgH):
        """W-fixed fit from the cluster medians (pyDNMFk.py:245-248): only the H half-step runs.  In replica mode
        every rank runs the same (deterministic) fit on its own copy."""
        self.params.W_update = False
        saved = self._enter_group() if self._spread() else None
        reg = PyNMF(self._A_dev, factors=[AvgW, AvgH], params=self.params)
        W, H, err = reg.fit()
        self.col_err = reg.column_err()
        if saved is not None:
            self._leave_group(saved)
        return W.cpu().numpy(), H.cpu().numpy(), err

    @comm_timing()
    def pynmfk_per_k(self):
        """Ensemble, clustering, silhouettes and the regression fit for ``self.k`` (pyDNMFk.py:214-258)."""
        from .data_io import data_write
        from .dist_clustering import custom_clustering
        self.params.results_paths = self.params.results_path + str(self.k) + '/'
        if self.rank == 0:
            os.makedirs(self.params.results_paths, exist_ok=True)
            if self.verbose:
                print('*************Computing for k=', self.k, '************')
        self.fit_ensemble(self.k)
        perturbation = self.perturbations - 1
        self.params.flag = 1
        self.cp._save_checkpoint(self.params.flag, perturbation, self.k)
        spread = self._spread()
        saved = self._enter_group() if spread else None              # replica mode: every group clusters its own copy
        clusters = custom_clustering(self._Wall_dev, self._Hall_dev, self.params)
        [processAvg, processSTD, Hall_dev, self.clusterSilhouetteCoefficients, self.avgSilhouetteCoefficients,
         idx] = clusters.fit()
        if saved is not None:
            self._leave_group(saved)
        self._Hall_dev = Hall_dev
        self.Hall = Hall_dev.cpu().numpy()
        self.params.flag = 2
        self.cp._save_checkpoint(self.params.flag, perturbation, self.k)
        AvgH_dev = D.default_ops().median_last(Hall_dev)              # np.median(self.Hall, axis=-1)
        self.AvgW, self.AvgH, self.L_errDist = self.fit_regression(processAvg, AvgH_dev)
        self.avgErr = np.mean(self.recon_err)
        self.AIC = 2 * self.k + self.params.m * self.params.n * numpy.log(self.avgErr / (self.params.m * self.params.n))
        cluster_stats = {'clusterSilhouetteCoefficients': self.clusterSilhouetteCoefficients,
                         'avgSilhouetteCoefficients': self.avgSilhouetteCoefficients, 'L_errDist': self.L_errDist,
                         'L_err': self.col_err, 'avgErr': self.avgErr, 'recon_err': self.recon_err, 'AIC': self.AIC}
        if not spread:
            data_writer = data_write(self.params)
            data_writer.save_factors([self.AvgW, self.AvgH], reg=True)
            data_writer.save_cluster_results(cluster_stats)
        else:
            # every replica group holds the same (deterministic) regression factors: group 0 writes them, with ITS
            # communicator on params -- save_factors ends in a barrier over params.comm1, which must only span the
            # ranks that call it
            saved = self._enter_group()
            if self._group_index == 0:
                data_writer = data_write(self.params)
                data_writer.save_factors([self.AvgW, self.AvgH], reg=True)
                data_writer.save_cluster_results(cluster_stats)
            self._leave_group(saved)
        self.params.flag = 3
        self.cp._save_checkpoint(self.params.flag, perturbation, self.k)

    @comm_timing()
    def pvalueAnalysis(self):
        """Rank selection from the per-k regression errors and silhouettes (pyDNMFk.py:261-299): walk k upwards and
        accept k while the previous k clustered stably (min silhouette > sill_thr) and the per-column regression errors
        dropped significantly (Wilcoxon signed-rank p < 0.05)."""
        from scipy.stats import wilcoxon
        from .data_io import read_results
        k_swap_range = range(self.params.start_k, self.params.end_k + 1, self.step_k)
        pvalue = np.ones(len(k_swap_range))
        sill_min, err_regres = [], []
        for k in k_swap_range:
            data = read_results(self.params.results_path + str(k) + '/')
            err_regres.append(np.array(data['L_err']))
            sill_min.append(round(np.min(np.array(data['clusterSilhouetteCoefficients'])), 2))
        one_distr_err = err_regres[0]
        nopt = 1
        for i in range(1, len(k_swap_range)):
            if sill_min[i - 1] > self.sill_thr:
                pvalue[i] = wilcoxon(one_distr_err, err_regres[i])[1]
                if pvalue[i] < 0.05:
                    nopt = i
                    one_distr_err = np.copy(err_regres[i])
        return k_swap_range[nopt - 1], pvalue

    @comm_timing()
    def fit(self):
        """NMFk over ``start_k .. end_k``: returns the estimated number of latent features (pyDNMFk.py:169-212)."""
        self.params.results_path = self.params.results_path + self.params.fname + '/'
        if self.rank == 0:
            os.makedirs(self.params.results_path, exist_ok=True)
        if self.params.checkpoint:
            try:
                self.cp.load_from_checkpoint()
                self.start_k = self.cp.k + self.step_k if self.cp.flag > 3 else self.cp.k
            except Exception:
                pass
        self.comm1.barrier()
        for self.k in range(self.start_k, self.end_k + 1, self.step_k):
            self.params.k = self.k
            self.pynmfk_per_k()
        self.comm1.barrier()
        if self.rank == 0:
            nopt1, pvalue1 = self.pvalueAnalysis()
            print('Rank estimated by NMFk = ', nopt1)
        else:
            nopt1 = None
        nopt1 = self.comm1.bcast(nopt1, root=0)
        self.comm1.barrier()
        return nopt1
