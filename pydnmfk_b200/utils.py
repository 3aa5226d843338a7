"""Shard geometry, pruning masks and the small helpers of the reference's ``utils.py``.

Only the hot-path part of ``pyDNMFk/utils.py`` is mirrored (SURVEY.md section 2 row 4):
``determine_block_params`` (:15-46), ``data_operations`` (:49-217), ``norm`` (:367-391),
``str2bool`` (:462-471), ``var_init`` (:473-477), ``parse`` (:480-483), ``Checkpoint``
(:486-536) and ``comm_timing`` (:539-567).  Index maps are plain integer arithmetic on the
host; the per-element work (non-zero counts, compaction, un-prune scatter) runs on the device.
"""
import copy
import os
import pickle

import numpy
import numpy as np
import torch

from . import config
from .dist_comm import MPI
from . import device as D
from .sparse import SparseShard, is_sparse_input

config.init(0)


class determine_block_params():
    """Index range / shape of the block of a ``shape`` array owned by one rank of a ``pgrid``.

    Same contract as utils.py:15-46: ``comm`` may be an int (rank) or a communicator; ranks map
    row-major onto the grid; the remainder is spread over the leading blocks; ``end`` is inclusive;
    a 1-element grid always behaves as rank 0.
    """

    def __init__(self, comm, pgrid, shape):
        self.rank = comm if type(comm) == int else comm.rank
        self.pgrid = tuple(int(g) for g in pgrid)
        if int(np.prod(self.pgrid)) <= 1:
            self.rank = 0
        self.shape = shape

    def _bounds(self):
        where = np.unravel_index(self.rank, self.pgrid)
        lo, hi = [], []
        for extent, parts, i in zip(self.shape, self.pgrid, where):
            base, extra = divmod(int(extent), parts)
            i = int(i)
            lo.append(i * base + min(i, extra))
            hi.append((i + 1) * base + min(i + 1, extra) - 1)
        return lo, hi

    def determine_block_index_range_asymm(self):
        return self._bounds()

    def determine_block_shape_asymm(self):
        lo, hi = self._bounds()
        return [b - a + 1 for a, b in zip(lo, hi)]


class data_operations():
    """Global / local dimensions, zero row/column pruning and un-pruning of one shard.

    ``data`` may be a numpy array or a CUDA tensor; it is moved to the device once and stays
    there.  Side effects on ``params`` match the reference: ``m, n, m_loc, n_loc, W_start,
    W_end, H_start, H_end`` (utils.py:73-115) and the four boolean masks (utils.py:169).
    """

    def __init__(self, data, params):
        self.params = params
        self.comm1 = self.params.comm1
        self.cart_1d_row = self.params.row_comm
        self.cart_1d_column = self.params.col_comm
        self.rank = self.comm1.rank
        self.p_r = self.params.p_r
        self.p_c = self.params.p_c
        self.topo = self.params.topo
        self.k = self.params.k
        self.ten = data
        self.compute_global_dim()
        self.compute_local_dim()
        (self.A_ij_m, self.A_ij_n) = self.ten.shape
        self.m = self.params.m
        self.n = self.params.n

    # -- dimensions (integer, host) ----------------------------------------------------------
    def compute_global_dim(self):
        """utils.py:73-93."""
        self.loc_m, self.loc_n = int(self.ten.shape[0]), int(self.ten.shape[1])
        if self.p_r != 1 and self.p_c == 1:
            self.params.n = self.loc_n
            self.params.m = self.comm1.allreduce(self.loc_m)
        elif self.p_c != 1 and self.p_r == 1:
            self.params.n = self.comm1.allreduce(self.loc_n)
            self.params.m = self.loc_m
        else:
            first_col = (self.rank % self.p_c == 0)
            first_row = (self.rank // self.p_c == 0)
            self.params.m = self.comm1.allreduce(self.loc_m if first_col else 0)
            self.params.n = self.comm1.allreduce(self.loc_n if first_row else 0)

    def compute_local_dim(self):
        """utils.py:97-115: factor-shard sizes and their position inside the local A block."""
        if self.topo == '2d':
            blk_m = determine_block_params(self.cart_1d_column, (self.p_c, 1), (self.ten.shape[0], self.k))
            blk_n = determine_block_params(self.cart_1d_row, (1, self.p_r), (self.k, self.ten.shape[1]))
        else:
            blk_m = determine_block_params(self.comm1, (self.p_r, 1), (self.params.m, self.k))
            blk_n = determine_block_params(self.comm1, (1, self.p_c), (self.k, self.params.n))
        (w_lo, _), (w_hi, _) = blk_m.determine_block_index_range_asymm()
        (_, h_lo), (_, h_hi) = blk_n.determine_block_index_range_asymm()
        self.params.m_loc, self.params.n_loc = w_hi - w_lo + 1, h_hi - h_lo + 1
        self.params.W_start, self.params.W_end = w_lo, w_hi + 1
        self.params.H_start, self.params.H_end = h_lo, h_hi + 1

    # -- pruning -------------------------------------------------------------------------------
    def _device_data(self):
        if is_sparse_input(self.ten):
            self.ten = SparseShard.from_any(self.ten)
        elif not (isinstance(self.ten, torch.Tensor) and self.ten.is_cuda):
            self.ten = D.to_device(self.ten)
        return self.ten

    def zero_idx_prune(self):
        """Boolean keep-masks (utils.py:117-135): counts on the device, integer all-reduce over the
        communicator that spans the other grid dimension, thresholds on the host."""
        ops = D.default_ops()
        A = self._device_data()
        row_cnt, col_cnt = ops.nnz_counts(A)
        if self.topo == '2d':
            row_cnt = self.cart_1d_column.allreduce_(row_cnt)
            col_cnt = self.cart_1d_row.allreduce_(col_cnt)
        else:
            if self.p_c > 1:
                row_cnt = self.comm1.allreduce_(row_cnt)
            if self.p_r > 1:
                col_cnt = self.comm1.allreduce_(col_cnt)
        row_cnt = row_cnt.cpu().numpy()
        col_cnt = col_cnt.cpu().numpy()
        row_zero_idx_x = row_cnt > 0
        col_zero_idx_x = col_cnt > 0
        if self.topo == '2d':
            col_zero_idx_h = col_cnt[self.params.H_start:self.params.H_end] > 0
            row_zero_idx_w = row_cnt[self.params.W_start:self.params.W_end] > 0
        else:
            row_zero_idx_w = row_cnt > 0
            col_zero_idx_h = col_cnt > 0
        return row_zero_idx_x, col_zero_idx_x, row_zero_idx_w, col_zero_idx_h

    @staticmethod
    def _idx(mask, length):
        mask = np.asarray(mask, dtype=bool)
        assert mask.shape[0] == length
        return torch.from_numpy(np.flatnonzero(mask).astype(np.int64))

    def prune(self, data, row_zero_idx, col_zero_idx):
        """data[np.ix_(rows, cols)] as a device gather (utils.py:137-156).  A sparse shard is compacted instead: kept rows
        and columns are renumbered, values and their order stay (the dropped rows and columns are empty)."""
        ops = D.default_ops()
        if is_sparse_input(data):
            X = SparseShard.from_any(data)
            return X.compact(self._idx(row_zero_idx, X.shape[0]).to(X.device),
                             self._idx(col_zero_idx, X.shape[1]).to(X.device))
        X = D.to_device(data)
        ri = self._idx(row_zero_idx, X.shape[0]).to(X.device)
        ci = self._idx(col_zero_idx, X.shape[1]).to(X.device)
        return ops.compact(X, ri, ci)

    def prune_all(self, W, H):
        """utils.py:158-176."""
        (self.params.row_zero_idx_x, self.params.col_zero_idx_x,
         self.params.row_zero_idx_w, self.params.col_zero_idx_h) = self.zero_idx_prune()
        self.ten = self.prune(self.ten, self.params.row_zero_idx_x, self.params.col_zero_idx_x)
        W = self.prune(W, self.params.row_zero_idx_w, [True] * W.shape[1])
        H = self.prune(H, [True] * H.shape[0], self.params.col_zero_idx_h)
        return self.ten, W, H

    def unprune(self, data, row_zero_idx, col_zero_idx):
        """Scatter back into float64 zeros (utils.py:178-199); guarded by len(mask) > 1 as there."""
        ops = D.default_ops()
        X = D.to_device(data)
        if len(row_zero_idx) > 1:
            ri = self._idx(row_zero_idx, len(row_zero_idx)).to(X.device)
            return ops.scatter_rows(X, ri, len(row_zero_idx))
        elif len(col_zero_idx) > 1:
            ci = self._idx(col_zero_idx, len(col_zero_idx)).to(X.device)
            return ops.scatter_cols(X, ci, len(col_zero_idx))
        raise UnboundLocalError("unprune: mask of length <= 1 (the reference fails the same way)")

    def unprune_factors(self, W, H):
        """utils.py:201-217."""
        W = self.unprune(W, self.params.row_zero_idx_w, [])
        H = self.unprune(H, [], self.params.col_zero_idx_h)
        return W, H


class transform_H_index():
    """Order in which the per-rank H shards of a p_r x p_c grid tile the columns of H (utils.py:345-364).

    The shard of rank ``i * p_c + j`` covers sub-block ``i`` of block column ``j`` (SURVEY A2), so the column order is
    "for j: for i".  The reference computes ``i * p_r + j``, which is the same only for square grids; the rank index
    used here is the one that reassembles H correctly on every grid (tests/test_host_logic.py, tests -m gpu).
    """

    def __init__(self, grid):
        self.p_r = grid[0]
        self.p_c = grid[1]

    def rankidx2blkidx(self):
        return [i * self.p_c + j for j in range(self.p_c) for i in range(self.p_r)]

    def transform_H_idx(self, rank):
        return self.rankidx2blkidx()[rank]


def norm(X, comm, norm=2, axis=None, p=-1):
    """Distributed vector 2-norm (utils.py:367-391): local sum of squares on the device, optional
    all-reduce, square root.  Returns a python float."""
    if norm != 2 or axis is not None:
        raise NotImplementedError('only the global 2-norm is used by the update loop')
    ops = D.default_ops()
    t = D.to_device(X)
    if t.dim() == 1:
        t = t.reshape(1, -1)
    sq = ops.sqnorm(t.contiguous())
    if p != 1:
        sq = comm.allreduce_(sq)
    return float(np.sqrt(sq.item()))


def str2bool(v):
    """utils.py:462-471."""
    if isinstance(v, bool):
        return v
    if v.lower() in ('yes', 'true', 't', 'y', '1'):
        return True
    elif v.lower() in ('no', 'false', 'f', 'n', '0'):
        return False
    else:
        raise NameError('Boolean value expected.')


def var_init(clas, var, default):
    """Lazy default of an attribute bag (utils.py:473-477)."""
    if not hasattr(clas, var):
        setattr(clas, var, default)
    return clas.__getattribute__(var)


class parse():
    """Free-form attribute bag used as ``params`` (utils.py:480-483)."""

    def __init__(self):
        pass


class Checkpoint():
    """NMFk-level checkpoint of (flag, perturbation, k) on rank 0 (utils.py:486-536)."""

    def __init__(self, checkpoint_save, params):
        self.checkpoint_save = checkpoint_save if checkpoint_save else False
        self.params = params
        self.perturbation = 0
        self.k = 0
        self.flag = 0

    def load_from_checkpoint(self):
        if self.checkpoint_save:
            with open(self.params.results_path + "/checkpoint.p", "rb") as f:
                saved = pickle.load(f)
            self._set_params(vars(saved))
            if self.params.rank == 0:
                print("Continuing from checkpoint for k=", self.k, 'perturbation=', self.perturbation)

    def _save_checkpoint(self, flag, perturbation, k):
        state = parse()
        state.flag, state.perturbation, state.k = flag, perturbation, k
        if self.checkpoint_save and self.params.rank == 0:
            os.makedirs(self.params.results_path, exist_ok=True)
            with open(self.params.results_path + "checkpoint.p", "wb") as f:
                pickle.dump(state, f)

    def _set_params(self, class_parameters):
        for parameter, value in class_parameters.items():
            setattr(self, parameter, value)


class comm_timing(object):
    """Per-function wall-clock accumulation into ``config.time`` (utils.py:539-567).  As in the
    reference the switch is sampled when the decorated class body is executed; device-side
    profiling uses CUDA events / ncu instead (see bench.py, profiles/)."""

    def __init__(self):
        self.flag = config.flag
        self.time = copy.copy(config.time)

    def __call__(self, original_function):
        if not self.flag:
            return original_function

        def wrapper_timer(*args, **kwargs):
            start = MPI.Wtime()
            value = original_function(*args, **kwargs)
            self.time[original_function.__name__] = self.time.get(original_function.__name__, 0) + MPI.Wtime() - start
            config.time.update(self.time)
            return value

        return wrapper_timer
