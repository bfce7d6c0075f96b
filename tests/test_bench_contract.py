"""bench.py's reference arm: one JSON line with the contract's keys; what --dump-outputs writes after the timed steps
(dump_outputs itself on the host, the whole bench on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oraclebind
import refbind
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _with_nonfinite(a, recs):
    """undoes bench.split_nonfinite: the (row, column, code) records back into the table"""
    a = a.copy()
    r, c, code = recs.T
    a[r.astype(int), c.astype(int)] = np.where(code == 2, np.nan, code * np.inf)
    return a


@pytest.mark.skipif(not refbind.available("glibc"), reason="oracle/_ref/libref_glibc.so not built")
def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "512", "--steps", "1",
                          "--warmup", "0", "--ref-threads", "2"], capture_output=True, text=True, timeout=300, check=True).stdout
    d = json.loads(out.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "lsd_source_mpixel_per_s" and d["unit"] == "Mpixel/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == 2
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_steps_tables(tmp_path):
    """--dump-outputs DIR: finite float64 .npy files holding the segment tables of the last timed step (non-finite entries
    recorded beside them), equal to the CPU oracle's on the same seeded maps."""
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", "512", "--maps-per-gpu", "4", "--inflight", "2",
                    "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                   capture_output=True, text=True, timeout=600, check=True)
    names = ("counts", "maps", "lines", "lines_nonfinite", "rects", "rects_nonfinite")
    assert sorted(os.listdir(tmp_path)) == sorted(f"{k}.npy" for k in names)
    d = {k: np.load(tmp_path / f"{k}.npy") for k in names}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in d.values())
    for k in ("lines", "rects"):
        d[k] = _with_nonfinite(d[k], d[k + "_nonfinite"])
    assert np.isinf(d["lines"]).any()                    # the maps have vertical segments: k = -inf, b = NaN
    assert np.array_equal(d["maps"], np.arange(4))
    off = 0
    for i in range(4):
        o = oraclebind.lsd(synth.occupancy_grid(512, 512, seed=1000 + i), want_maps=False, want_line_im=False)
        assert d["counts"][i] == o["n"]
        assert np.array_equal(d["lines"][off:off + o["n"]], o["lines"], equal_nan=True)
        assert np.array_equal(d["rects"][off:off + o["n"]], o["rects"], equal_nan=True)
        off += o["n"]
    assert off == len(d["lines"]) == len(d["rects"]) > 0


def test_dump_outputs_round_trip_and_sample(lsdb, tmp_path, monkeypatch):
    """bench.dump_outputs on the oracle's tables of seeded maps (vertical segments: k = -inf, b = NaN): finite float64 files
    from which the tables come back bit for bit; past DUMP_LIMIT a fixed seeded sample of whole maps, within the limit."""
    import bench
    maps = [synth.occupancy_grid(512, 512, seed=1000 + i) for i in range(4)]
    o = [oraclebind.lsd(m, want_maps=False, want_line_im=False) for m in maps]
    got = dict(counts=np.array([x["n"] for x in o], np.int32), lines=[lsdb.array_to_lines(x["lines"]) for x in o],
               rects=[x["rects"] for x in o])
    assert any(np.isinf(x["lines"]).any() for x in o)
    for limit, name in ((bench.DUMP_LIMIT, "all"), (16000, "sample")):
        monkeypatch.setattr(bench, "DUMP_LIMIT", limit)
        out = tmp_path / name
        bench.dump_outputs(str(out), got, lsdb.lines_to_array)
        d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
        assert sorted(d) == ["counts", "lines", "lines_nonfinite", "maps", "rects", "rects_nonfinite"]
        assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in d.values())
        assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= limit
        assert np.array_equal(d["counts"], got["counts"])
        kept = d["maps"].astype(int)
        assert (len(kept) == 4) == (name == "all") and len(kept) > 0
        assert np.array_equal(_with_nonfinite(d["lines"], d["lines_nonfinite"]), np.concatenate([o[i]["lines"] for i in kept]), equal_nan=True)
        assert np.array_equal(_with_nonfinite(d["rects"], d["rects_nonfinite"]), np.concatenate([o[i]["rects"] for i in kept]), equal_nan=True)
