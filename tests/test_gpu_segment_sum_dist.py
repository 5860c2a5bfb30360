"""Cluster means and mean pooling on a row partition (parallel.dist_segment_sum / dist_cluster_means /
dist_segment_mean_pool, gdr_segment_sum_dist) in an NCCL group of one rank: byte-equal to the one-GPU segment_sum /
cluster_means / segment_mean_pool, and every rejection raises ValueError with the communicator usable afterwards."""
import os
import socket

import numpy as np
import pytest
import torch

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


def _bits(t):
    return t.contiguous().view(torch.int32)


def _data(N, F, K, seed, padded=True, labels=None):
    from gdr._dev import new_padded
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev).manual_seed(seed)
    X = torch.randn((N, F), generator=g, device=dev) * torch.exp(torch.empty((N, 1), device=dev).uniform_(-6, 6, generator=g))
    if padded:                                # the layout dist_propagate returns: a [N, F] view of [N, pad4(F)]
        Xp = new_padded(N, F, dev)
        Xp.copy_(X)
        X = Xp
    lab = torch.randint(0, K, (N,), generator=g, device=dev, dtype=torch.int32) if labels is None else labels
    return X, lab


def _check(comm, X, lab, K):
    import gdr
    from gdr import parallel as par
    from gdr._dev import padded_rows
    N, F = X.shape
    part = par.RowPartition(N, 1, 0)
    s1, c1 = gdr.segment_sum(padded_rows(X.to(torch.float32)), lab.to(torch.int32).contiguous(), K)
    s2, c2 = par.dist_segment_sum(comm, part, X, lab, K)
    assert s2.shape == (K, F) and c2.dtype == torch.int32
    assert torch.equal(_bits(s2), _bits(s1)) and torch.equal(c2, c1)
    m1, m2 = gdr.cluster_means(X, lab, K), par.dist_cluster_means(comm, part, X, lab, K)
    assert m2.shape == m1.shape and torch.equal(_bits(m2), _bits(m1))
    p1, p2 = gdr.segment_mean_pool(X, lab, K), par.dist_segment_mean_pool(comm, part, X, lab, K)
    assert p2.shape == p1.shape and torch.equal(_bits(p2), _bits(p1))
    return c1, m2


@pytest.mark.parametrize("N,F,K", [(2449029, 100, 10000),     # config E
                                   (169343, 128, 1000),       # config B
                                   (2708, 1433, 140),         # Dp4 > 1024: two column passes
                                   (50000, 7, 300), (50000, 47, 2000)])
def test_bytes_equal_to_one_gpu(comm, N, F, K):
    X, lab = _data(N, F, K, seed=N + F)
    counts, _ = _check(comm, X, lab, K)
    assert int(counts.sum()) == N


def test_unpadded_input_and_int64_labels(comm):
    X, lab = _data(3001, 7, 50, seed=5, padded=False)
    assert X.stride(0) == 7
    _check(comm, X, lab.to(torch.int64), 50)


def test_empty_clusters_nan_rows(comm):
    dev = torch.device("cuda", torch.cuda.current_device())
    lab = 2 * torch.randint(0, 40, (9000,), device=dev, dtype=torch.int32)     # every odd cluster empty
    X, lab = _data(9000, 47, 80, seed=7, labels=lab)
    counts, means = _check(comm, X, lab, 80)
    empty = counts == 0
    assert int(empty.sum()) == 40 and bool(torch.isnan(means[empty]).all()) and not bool(torch.isnan(means[~empty]).any())


def test_single_cluster_and_more_clusters_than_rows(comm):
    X, lab = _data(10007, 100, 1, seed=9)
    _check(comm, X, lab, 1)
    X, lab = _data(5, 47, 64, seed=10)
    _check(comm, X, lab, 64)


def test_rejections_then_a_valid_call(comm):
    from gdr import parallel as par
    X, lab = _data(4000, 47, 30, seed=11)
    part = par.RowPartition(4000, 1, 0)
    for bad in (30, -1, 1 << 20):
        lb = lab.clone()
        lb[1234] = bad
        with pytest.raises(ValueError):
            par.dist_cluster_means(comm, part, X, lb, 30)
    lb = lab.to(torch.int64)
    lb[7] = (1 << 32) + 3                      # would wrap to a valid label in a plain int32 cast
    with pytest.raises(ValueError):
        par.dist_segment_mean_pool(comm, part, X, lb, 30)
    for K in (0, -5):
        with pytest.raises(ValueError):
            par.dist_cluster_means(comm, part, X, lab, K)
    with pytest.raises(ValueError):
        par.dist_segment_sum(comm, part, X, lab[:-1], 30)      # labels for fewer rows than X has
    _check(comm, X, lab, 30)
