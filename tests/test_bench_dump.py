"""bench.py --steps and --dump-outputs: the timed loops run exactly --steps steps, and the dump holds what the timed path returned in
its last step (the CPU tests need no GPU; the native headline run is marked gpu)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

import bench  # noqa: E402  (conftest puts the repository root on sys.path)

HB = ("H_pp", "H_lp", "H_ll", "b_p", "b_l")


def _load(d, names):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in names}


def test_dump_sample_is_fixed_and_shared_by_every_array(tmp_path, monkeypatch):
    """The seeded-sample branch (the default 4096-window benchmark takes it): every array holds the same windows, the choice does not
    change between runs, the files stay within the budget, and a smaller sample of the same W is a subset of a larger one."""
    W = 300
    outs = {"H_pp": np.zeros((W, 6, 6)), "H_lp": np.zeros((W, 5, 6)), "b_p": np.zeros((W, 6))}
    for v in outs.values():
        v += np.arange(W).reshape((W,) + (1,) * (v.ndim - 1))          # every entry of window w is w
    per_window = sum(v[0].nbytes for v in outs.values())
    monkeypatch.setattr(bench, "DUMP_BYTES", 40 * per_window)
    info = bench.dump_outputs(str(tmp_path / "a"), outs)
    again = bench.dump_outputs(str(tmp_path / "b"), outs)
    assert info["windows"] == 40 and info["of_windows"] == W and info == {**again, "dir": info["dir"]}
    want = np.sort(np.random.default_rng(bench.DUMP_SEED).permutation(W)[:40])
    assert len(np.unique(want)) == 40
    a, b = _load(tmp_path / "a", outs), _load(tmp_path / "b", outs)
    for k in outs:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k]), k
        assert np.array_equal(a[k].reshape(40, -1), np.broadcast_to(want[:, None].astype(np.float64), (40, a[k][0].size))), k
    assert sum(a[k].nbytes for k in outs) <= bench.DUMP_BYTES
    assert np.isin(bench.dump_windows(W, 25), want).all()
    assert np.array_equal(bench.dump_windows(W, W), np.arange(W))


def test_reference_arm_runs_steps_and_dumps_its_outputs(pkg, orc, cfg, tmp_path, monkeypatch, capsys):
    """--impl reference: exactly warmup + steps calls of the CPU path (no cap on the step count), and --dump-outputs writes what the
    last call returned (H/b and S/g of every window: 8 windows fit the budget)."""
    calls = []

    class Counting:
        def __getattr__(self, name):
            return getattr(orc, name)

        def linearize_batch(self, *a, **kw):
            calls.append(1)
            return orc.linearize_batch(*a, **kw)

    monkeypatch.setattr(bench.ge, "load_oracle", lambda: Counting())
    W, steps, warm = 8, 5, 3
    bench.run_reference(argparse.Namespace(gpus=1, steps=steps, warmup=warm, windows=W, dump_outputs=str(tmp_path)))
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert len(calls) == warm + steps and line["steps"] == steps
    names = HB + ("S", "g")
    assert line["dump_outputs"]["windows"] == W and sorted(os.listdir(tmp_path)) == sorted(n + ".npy" for n in names)
    abi, synth = pkg._abi, pkg.synth
    batch, _ = synth.with_line_map(synth.make_windows(W, seed=0x5EED + 2, f32_obs=True), cfg)
    ref = orc.linearize_batch(cfg, batch, abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY)
    got = _load(tmp_path, names)
    for n in names:
        assert got[n].dtype == np.float64 and np.array_equal(got[n], ref[n]), n


def _native(tmp, W, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                        "--windows", str(W), "--skip-extras", "--skip-cpu", "--skip-assoc", "--dump-outputs", str(tmp)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_native_headline_runs_steps_and_dumps_its_outputs(pkg, orc, cfg, tmp_path):
    """Two small headline runs (2 and 5 steps): every kernel's launch count inside the timed window is proportional to --steps, both
    dumps equal what the oracle computes for the same seeded windows (64 windows fit the budget, so all are written), and the
    two runs' dumps agree (same inputs from run to run)."""
    W = 64
    lines = {s: _native(tmp_path / str(s), W, s) for s in (2, 5)}
    n2, n5 = (lines[s]["roofline"]["kernel_launches_timed"] for s in (2, 5))
    assert n2 and set(n2) == set(n5) and all(5 * n2[k] == 2 * n5[k] for k in n2), (n2, n5)
    abi, synth = pkg._abi, pkg.synth
    batch, _ = synth.with_line_map(synth.make_windows(W, seed=0x5EED + 2, f32_obs=True), cfg)   # bench.py's rank-0 batch
    ref = orc.linearize_batch(cfg, batch, abi.OUT_HB | abi.LOSS_CAUCHY, nthreads=8)
    dumps = {}
    for s in (2, 5):
        assert lines[s]["steps"] == s and lines[s]["dump_outputs"]["windows"] == W
        assert sorted(os.listdir(tmp_path / str(s))) == sorted(n + ".npy" for n in HB)
        dumps[s] = _load(tmp_path / str(s), HB)
        assert sum(os.path.getsize(tmp_path / str(s) / (n + ".npy")) for n in HB) <= 64 << 20
        for n in HB:
            assert dumps[s][n].dtype == np.float64 and dumps[s][n].shape[0] == W
            assert pkg.parity.unit_err(n, dumps[s][n], ref[n]) < 1e-9, (s, n)
    for n in HB:   # the pose blocks are summed through shared-memory atomics: equal to rounding only
        assert pkg.parity.unit_err(n, dumps[5][n], dumps[2][n]) < 1e-12, n
