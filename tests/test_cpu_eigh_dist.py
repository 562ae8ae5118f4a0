"""`not gpu`: world-size-2 gloo tests of finalize_head_spectra(with_components=True): the owner of a head computes its principal
axes and every rank ends with every head's, equal to what one process computes from the same samples, on the covariance route
and on the Gram route (rank-sharded parked rows)."""
import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from audio_residual_b200.parallel import shard_range
from test_cpu_dist import _free_port


class Acc:                # a MomentAccumulator's state without the CUDA update path
    def __init__(self, X):
        self.D, self.n = X.shape[1], X.shape[0]
        self.s1 = torch.from_numpy(X.sum(0))
        self.s2 = torch.from_numpy(X.T @ X)


class Parked:             # what finalize_head_spectra reads of a MomentAccumulator that still holds every row
    def __init__(self, rows):
        self.D, self.n, self._buf, self._fill = rows.shape[1], rows.shape[0], rows, rows.shape[0]
        self._s1 = torch.zeros(self.D, dtype=torch.float64)

    def parked_rows(self):
        return self._buf[:self._fill]

    @property
    def s1(self):
        return self._buf.double().sum(0)

    @property
    def s2(self):
        return self._buf.double().t() @ self._buf.double()


def cov_data(h):
    rng = np.random.default_rng(10 + h)
    return rng.standard_normal((400, 12)) * np.linspace(2, 0.2, 12) + h


def gram_data(h):
    rng = np.random.default_rng(20 + h)
    return torch.from_numpy((rng.random((30, 64)) ** 2 + h).astype(np.float32))


def cov_accs(lo, hi):
    return [Acc(cov_data(h)[lo:hi]) for h in range(5)]


def gram_accs(lo, hi, rank=0):
    # heads 0-2 parked on every rank (Gram route); head 3 has been folded on rank 1 (moment route for the whole head)
    return [Acc(gram_data(h)[lo:hi].double().numpy()) if (h == 3 and rank == 1) else Parked(gram_data(h)[lo:hi]) for h in range(4)]


def _worker(rank, world, port, out):
    import os
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from audio_residual_b200.analyze_attention import finalize_head_spectra
    lo, hi = shard_range(400, rank, world)
    cov = finalize_head_spectra(cov_accs(lo, hi), with_components=True)
    lo, hi = (0, 11) if rank == 0 else (11, 30)                   # uneven shards
    gram = finalize_head_spectra(gram_accs(lo, hi, rank), with_components=True)
    out.put((rank, cov, gram))
    dist.barrier()
    dist.destroy_process_group()


def _check(got, ref, rows):
    (spec, comps), (rspec, rcomps) = got, ref
    for h, (w, c, rw, rc) in enumerate(zip(spec, comps, rspec, rcomps)):
        assert c.shape == rc.shape == (len(rw), len(rw)) and c.dtype == np.float64
        assert np.allclose(w, rw, rtol=1e-9, atol=1e-12 * rw[0]), h
        assert np.abs(c[:rows] - rc[:rows]).max() <= 1e-8, h
        assert np.abs(c @ c.T - np.eye(len(rw))).max() <= 1e-10, h                 # an orthonormal basis, completion included


def test_head_sharded_components_match_single_process():
    from audio_residual_b200.analyze_attention import finalize_head_spectra
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    ref_cov = finalize_head_spectra(cov_accs(0, 400), with_components=True)
    ref_gram = finalize_head_spectra(gram_accs(0, 30), with_components=True)
    for h in range(5):                # the single-process axes themselves: numpy eigh of the float64 covariance
        w, v = np.linalg.eigh(np.cov(cov_data(h).T, ddof=1))
        v = v[:, ::-1].T
        v = v * np.sign(v[np.arange(12), np.abs(v).argmax(1)])[:, None]
        assert np.abs(ref_cov[1][h] - v).max() <= 1e-9, h
    for rank, cov, gram in results:
        _check(cov, ref_cov, 12)
        _check(gram, ref_gram, 29)    # 30 centred samples: 29 axes with variance, the rest an orthonormal completion
