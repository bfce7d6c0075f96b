"""The region stage's two kernel builds — ban plane in shared memory (run when every map of the batch fits) and ban plane
read from global memory (any batch) — give the same segment tables, labels and used-maps, and the oracle's."""
import numpy as np
import pytest

import oraclebind
import synth
from test_gpu_lsd import lsdb_env

pytestmark = pytest.mark.gpu

# ban planes of 34 .. 30 400 bytes: each fits the 48 KB the library allows the shared copy by default
SMALL = [(500, 300), (34, 40), (128, 128), (1000, 90), (90, 1000), (600, 400)]
# 777x555 (55 KB) and 1200x900 (134 KB) do not: a batch holding them runs the global build unless the limit is raised
LARGE = [(777, 555), (1200, 900)]


def _run(lsdb, ctx, maps, env):
    with lsdb_env(env):
        b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
        b.upload(maps); b.run()
    got = b.download(want_rects=True)
    out = [(int(got["counts"][i]), got["rects"][i], b.planes(i)["labels"], b.planes(i)["used"]) for i in range(len(maps))]
    b.close()
    return out


def _same(x, y):
    assert x[0] == y[0]
    assert np.array_equal(x[1], y[1], equal_nan=True)
    assert np.array_equal(x[2], y[2]) and np.array_equal(x[3], y[3])


def test_shared_and_global_ban_plane_builds_agree(lsdb, ctx):
    small = [synth.occupancy_grid(c, r, seed=300 + i) for i, (c, r) in enumerate(SMALL)]
    large = [synth.occupancy_grid(c, r, seed=400 + i, border_walls=i == 1) for i, (c, r) in enumerate(LARGE)]
    ragged = small[:3] + large[:1] + small[3:] + large[1:]
    where = [0, 1, 2, 4, 5, 6]   # the small maps' places in the ragged batch
    shared = _run(lsdb, ctx, small, {})                                  # every plane fits: shared build
    glob = _run(lsdb, ctx, small, dict(LSDB_NO_SMEM_BAN="1"))            # global build forced
    mixed = _run(lsdb, ctx, ragged, {})                                  # two planes do not fit: global build
    mixed_shared = _run(lsdb, ctx, ragged, dict(LSDB_SMEM_BAN_KB="160"))  # limit raised: every plane fits, shared build
    for i in range(len(small)):
        _same(shared[i], glob[i])
        _same(shared[i], mixed[where[i]])
    for i in range(len(ragged)):
        _same(mixed[i], mixed_shared[i])
    for i, m in enumerate(ragged):
        o = oraclebind.lsd(m)
        assert mixed[i][0] == o["n"]
        assert np.array_equal(mixed[i][1], o["rects"], equal_nan=True)
        assert np.array_equal(mixed[i][2], o["labels"]) and np.array_equal(mixed[i][3], o["used"])
