"""bench.py --dump-outputs: the dumped arrays are what the timed steps computed (GPU: against the oracle stepped from the
same seeded state, and identical from run to run), whole interiors when they fit the size budget and the same seeded
sample otherwise (CPU)."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fake_model(shape, FT):
    rng = np.random.default_rng(7)
    fields = {}
    for n in "uvwb":
        a = np.asfortranarray(rng.uniform(-1, 1, shape).astype(FT))
        fields[n] = types.SimpleNamespace(interior=lambda a=a: a)
    return types.SimpleNamespace(names=tuple(fields), fields=fields)


def test_dump_writes_whole_interiors_within_budget(tmp_path):
    m = fake_model((8, 6, 5), np.float32)
    bench.dump_outputs(m, str(tmp_path))
    for n in m.names:
        got = np.load(tmp_path / f"{n}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, m.fields[n].interior())


def test_dump_samples_large_outputs_the_same_way_every_time(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 64 * 10 ** 3)
    m = fake_model((40, 30, 20), np.float64)
    bench.dump_outputs(m, str(tmp_path / "a"))
    bench.dump_outputs(m, str(tmp_path / "b"))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == [f"{n}.npy" for n in sorted(m.names)]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 3
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and a.ndim == 1 and a.size > 1000 and np.array_equal(a, b)
        assert np.all(np.isin(a, m.fields[f[:-4]].interior()))


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr


def run_bench(out_dir, N, steps, warmup):
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", str(N), "--steps", str(steps),
                    "--warmup", str(warmup), "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)],
                   capture_output=True, text=True, timeout=600, check=True)


@pytest.mark.gpu
def test_dumped_outputs_are_the_timed_steps(tmp_path):
    import oracle as O
    N, steps, warmup = 32, 2, 1
    run_bench(tmp_path / "a", N, steps, warmup)
    run_bench(tmp_path / "b", N, steps, warmup)
    go = O.RectilinearGrid(np.float64, size=(N,) * 3, extent=(1, 1, 1), topology=("Periodic",) * 3)
    mo = O.NonhydrostaticModel(go, advection=O.WENO5(), tracers=("b",), buoyancy=O.BuoyancyTracer(),
                               timestepper="RungeKutta3")
    mo.set(**bench.synthetic_state((N,) * 3))
    for _ in range(warmup + steps):
        mo.time_step(0.1 / N)
    for n in mo.names:
        ref = mo.fields[n].interior
        got = np.load(tmp_path / "a" / f"{n}.npy")
        assert got.dtype == np.float64 and got.shape == ref.shape
        assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < 1e-12, n
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{n}.npy")), n
