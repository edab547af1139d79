"""CPU: bench.py --dump-outputs writes the scores exactly (16-bit words in float32), keeps the same seeded sample of
coefficient positions from run to run, and stays under 64 MB at the benchmark's own shape."""
import os

import numpy as np

import bench


def _scores(rng, shape, n):
    s = np.zeros(shape + (n + 1,), dtype=np.uint64)
    s[..., :n] = rng.integers(0, 1 << 55, size=shape + (n,), dtype=np.uint64)
    return s


def _read(d):
    words = np.load(os.path.join(d, "scores.npy"))
    index = np.load(os.path.join(d, "scores_coeff_index.npy"))
    assert words.dtype == np.float32 and index.dtype == np.float32
    u = words.astype(np.uint64)
    return sum(u[..., i] << np.uint64(16 * i) for i in range(4)), index.astype(np.int64)


def test_dump_is_exact_and_sampled_the_same_way_every_time(tmp_path):
    rng = np.random.default_rng(5)
    s = _scores(rng, (2, 3, 2, 4), 64)
    bench.dump_outputs(str(tmp_path / "all"), s)
    got, index = _read(str(tmp_path / "all"))
    assert np.array_equal(index, np.arange(64)) and np.array_equal(got, s[..., :64])
    budget = s[..., 0].size * 16 * 20                     # room for 20 of the 64 coefficients
    bench.dump_outputs(str(tmp_path / "a"), s, budget=budget)
    bench.dump_outputs(str(tmp_path / "b"), s, budget=budget)
    got, index = _read(str(tmp_path / "a"))
    assert len(index) == 20 and np.all(np.diff(index) > 0) and index.max() < 64
    assert np.array_equal(got, s[..., index])
    for name in ("scores.npy", "scores_coeff_index.npy"):
        assert open(str(tmp_path / "a" / name), "rb").read() == open(str(tmp_path / "b" / name), "rb").read()


def test_dump_of_the_benchmark_shape_stays_under_64_mb(tmp_path):
    rng = np.random.default_rng(6)
    s = _scores(rng, (8, 10, 2, len(bench.PRIMES)), bench.N_POLY)   # default batch, 10 scores per image
    bench.dump_outputs(str(tmp_path), s)
    total = sum(os.path.getsize(str(tmp_path / f)) for f in os.listdir(str(tmp_path)))
    assert total <= 64 * 10**6
    got, index = _read(str(tmp_path))
    assert np.array_equal(got, s[..., index])
