"""Rank functions for the sparse-shard tests (spawned by tests/mp_util.run, so they live at module level)."""
import numpy as np


def _to_host(x):
    return x.cpu().numpy() if hasattr(x, 'cpu') else np.asarray(x)


def sparse_fit_worker(rank, world, case, kind='scipy'):
    """PyNMF.fit of a parity case with this rank's shard passed as a scipy.sparse.csr_matrix (kind='scipy') or as a CUDA
    torch sparse CSR tensor (kind='torch')."""
    import scipy.sparse as sp
    import torch
    from oracle import cases as C
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.utils import parse, determine_block_params, data_operations
    from pydnmfk_b200.pyDNMF import PyNMF
    torch.cuda.set_device(0)
    p_r, p_c = case['grid']
    comm = MPI.COMM_WORLD
    comms = MPI_comm(comm, p_r, p_c)
    np.random.seed(case['seed'])
    A = C.draw_global(case, np.random)
    args = parse()
    args.size, args.rank, args.comm1, args.comm, args.p_r, args.p_c = world, rank, comms.comm, comms, p_r, p_c
    args.m, args.n, args.k = case['m'], case['n'], case['k']
    args.itr, args.init, args.verbose = case['itr'], 'rand', False
    args.row_comm, args.col_comm = comms.cart_1d_row(), comms.cart_1d_column()
    args.norm, args.method, args.prune = case['norm'], case['method'], case['prune']
    args.W_update = case['W_update']
    blk = determine_block_params(rank, (p_r, p_c), A.shape).determine_block_index_range_asymm()
    A_ij = np.ascontiguousarray(A[blk[0][0]:blk[1][0] + 1, blk[0][1]:blk[1][1] + 1])
    factors = None
    if case['given_factors']:
        args.topo = '2d' if (p_r != 1 and p_c != 1) else '1d'
        dop = data_operations(A_ij, args)
        ml, nl = (dop.params.m_loc, dop.params.n_loc) if args.topo == '2d' else A_ij.shape
        factors = list(C.draw_given_factors(case, np.random, ml, nl))
    if kind == 'scipy':
        shard = sp.csr_matrix(A_ij)
    else:
        shard = torch.from_numpy(A_ij).cuda().to_sparse_csr()
    nmf = PyNMF(shard, factors=factors, params=args)
    W, H, err = nmf.fit()
    out = dict(W=_to_host(W), H=_to_host(H), err=float(err), out_type=type(W).__name__,
               geom=[int(v) for v in (args.m, args.n, args.m_loc, args.n_loc, args.W_start, args.W_end,
                                      args.H_start, args.H_end)])
    if case['prune']:
        out.update(row_zero_idx_x=np.asarray(args.row_zero_idx_x), col_zero_idx_x=np.asarray(args.col_zero_idx_x),
                   row_zero_idx_w=np.asarray(args.row_zero_idx_w), col_zero_idx_h=np.asarray(args.col_zero_idx_h))
    return out


def sparse_fit_many_worker(rank, world, cases):
    """Several cases of one world size in one process group; per-case failures are captured, not raised."""
    import traceback
    from pydnmfk_b200.dist_comm import MPI
    out = {}
    for case in cases:
        try:
            out[case['name']] = ('ok', sparse_fit_worker(rank, world, case))
            ok = 1
        except BaseException:
            out[case['name']] = ('err', traceback.format_exc())
            ok = 0
        if MPI.COMM_WORLD.allreduce(ok) != world:
            break
    return out
