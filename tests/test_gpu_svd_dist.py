"""The truncated SVD embeddings on a row partition (parallel.dist_compute_svd_embeddings, gdr_dense_gram_dist) in an
NCCL group of one rank: byte-equal to the one-GPU compute_svd_embeddings / gdr_dense_gram."""
import os
import socket

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def comm():
    import torch.distributed as dist
    from gdr import parallel as par
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    c = par.Comm(dist)
    yield c
    c.close()
    dist.destroy_process_group()


def _bits(x):
    x = x.cpu().numpy() if isinstance(x, torch.Tensor) else x
    return np.ascontiguousarray(x, dtype=np.float32).view(np.int32)


def _check(comm, nu, ni, u, i, dim, seed):
    """dist_compute_svd_embeddings from the lines (u, i) against compute_svd_embeddings of the same matrix."""
    import gdr
    from gdr import parallel as par
    R = sp.csr_matrix((np.ones(len(u), np.float32), (u, i)), shape=(nu, ni))
    ue, ie = gdr.compute_svd_embeddings(R, dim, seed=seed)
    dev = torch.device("cuda", torch.cuda.current_device())
    pu, pi = par.RowPartition(nu, 1, 0), par.RowPartition(ni, 1, 0)
    R_l, RT_l = par.dist_build_interaction(comm, pu, pi, torch.from_numpy(np.asarray(u)).to(dev),
                                           torch.from_numpy(np.asarray(i)).to(dev))
    ud, idd = par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, dim, seed=seed)
    assert ud.is_cuda and idd.is_cuda and ud.dtype == torch.float32
    assert tuple(ud.shape) == ue.shape and tuple(idd.shape) == ie.shape
    np.testing.assert_array_equal(_bits(ud), _bits(ue))
    np.testing.assert_array_equal(_bits(idd), _bits(ie))


def test_ali_display_subset(comm):
    sub = golden("recsys_ali_subset.npz")
    _check(comm, int(sub["nu"]), int(sub["ni"]), sub["u"].astype(np.int64), sub["i"].astype(np.int64),
           int(golden("svd_ali.npz")["dim"]), 42)


@pytest.mark.parametrize("shape,k", [((300, 100), 16), ((2000, 400), 64), ((120, 900), 24), ((40, 30), 8), ((50, 9), 8)])
def test_small_matrices(comm, shape, k):
    """test_gpu_svd's shapes: the exact path on either side and the clamped Krylov space."""
    rs = np.random.RandomState(shape[0] + k)
    M = sp.random(shape[0], shape[1], density=0.15, format="coo", random_state=rs, dtype=np.float32)
    _check(comm, shape[0], shape[1], M.row.astype(np.int64), M.col.astype(np.int64), k, 3)


def test_synthetic_3000_by_2000(comm):
    rs = np.random.RandomState(3)
    P = rs.rand(3000, 24) < 0.08
    Qm = rs.rand(24, 2000) < 0.08
    M = sp.coo_matrix(((P.astype(np.float32) @ Qm.astype(np.float32)) > 0).astype(np.float32))
    _check(comm, 3000, 2000, M.row.astype(np.int64), M.col.astype(np.int64), 16, 1)


def test_yelp2018_shape(comm):
    from gdr import synth
    cfg = synth.BIPARTITE["C"]
    u, i = synth.bipartite_interactions(cfg["users"], cfg["items"], cfg["inter"], seed=1236)
    _check(comm, cfg["users"], cfg["items"], u, i, cfg["d"], 42)


def test_rejects_a_bad_dim(comm):
    from gdr import parallel as par
    dev = torch.device("cuda", torch.cuda.current_device())
    pu, pi = par.RowPartition(1, 1, 0), par.RowPartition(5, 1, 0)
    u, i = torch.zeros(3, dtype=torch.int64, device=dev), torch.arange(3, dtype=torch.int64, device=dev)
    R_l, RT_l = par.dist_build_interaction(comm, pu, pi, u, i)
    with pytest.raises(ValueError):
        par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, 4)


@pytest.mark.parametrize("N", [2047, 2048, 2049, 32769])
def test_gram_dist_against_gram(comm, N):
    from gdr import parallel as par
    from gdr import svd as gsvd
    dev = torch.device("cuda", torch.cuda.current_device())
    rs = np.random.RandomState(N)
    W = torch.from_numpy(rs.standard_normal((N, 107)) * np.exp(rs.uniform(-6, 6, (N, 1)))).to(dev)
    ops = par.CudaOps()
    for A, B in ((W[:, :37], W[:, 37:]), (W[:, :64], W[:, :64]), (W[:, 5:6], W[:, 100:107])):
        got = ops.gram_dist(comm, N, 0, A, B)
        assert torch.equal(got.view(torch.int64), gsvd._gram(A, B).view(torch.int64))


def test_gram_dist_argument_checks(comm):
    from gdr import _lib
    from gdr import parallel as par
    dev = torch.device("cuda", torch.cuda.current_device())
    ops = par.CudaOps()
    A = torch.ones((10, 3), dtype=torch.float64, device=dev)
    with pytest.raises(_lib.GdrError):          # the blocks cover 10 rows, not 11
        ops.gram_dist(comm, 11, 0, A, A)
    with pytest.raises(_lib.GdrError):          # one rank must start at row 0
        ops.gram_dist(comm, 11, 1, A, A)
    C = ops.gram_dist(comm, 0, 0, A[:0], A[:0])   # no rows at all: C = 0
    assert torch.equal(C, torch.zeros((3, 3), dtype=torch.float64, device=dev))
