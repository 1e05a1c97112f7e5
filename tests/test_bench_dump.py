"""bench.py --dump-outputs: the arrays carry a tick's results exactly, a long array becomes the same seeded sample on
every run, and the files stay float64 and within 64 MB."""
import importlib
import os
import types

import numpy as np
import pytest

bench = importlib.import_module("bench")


def fake_tick(pkg, n_lobbies, L=10, G=32):
    lob = np.zeros(n_lobbies, pkg.engine.LOBBY_DTYPE)
    lob["first_member"] = np.arange(n_lobbies) * L
    lob["n_members"] = L
    lob["group"] = np.arange(n_lobbies) % G
    mem = pkg.synth.mix64(np.arange(n_lobbies * L, dtype=np.uint64))  # full 64-bit ids
    st = types.SimpleNamespace(pool_before=n_lobbies * L + 3, n_lobbies=n_lobbies, n_matched=n_lobbies * L,
                               n_residual=3, n_dead=0)
    return st, lob, mem


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


@pytest.mark.parametrize("n_lobbies", [0, 7, bench.DUMP_ROWS + 5])
def test_dump_outputs_exact_sampled_and_bounded(pkg, tmp_path, n_lobbies):
    st, lob, mem = fake_tick(pkg, n_lobbies)
    bench.dump_outputs(str(tmp_path / "a"), st, lob, mem)
    bench.dump_outputs(str(tmp_path / "b"), st, lob, mem)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert set(a) == {"tick_counts", "lobbies", "lobbies_rows", "member_ids", "member_ids_rows"}
    assert all(np.array_equal(a[k], b[k]) for k in a)  # same results -> same files
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= 64 << 20
    assert a["tick_counts"].tolist() == [st.pool_before, st.n_lobbies, st.n_matched, st.n_residual, st.n_dead]
    for name, full in (("lobbies", lob), ("member_ids", mem)):
        rows = a[name + "_rows"].astype(np.int64)
        assert len(rows) == min(len(full), bench.DUMP_ROWS)
        assert (np.diff(rows) > 0).all() and (len(rows) == 0 or rows[-1] < len(full))
    r = a["lobbies_rows"].astype(np.int64)
    want = np.stack([lob["first_member"], lob["n_members"], lob["mode"], lob["group"]], axis=1)[r]
    assert np.array_equal(a["lobbies"], want)
    hi, lo = a["member_ids"].astype(np.uint64).T
    assert np.array_equal(hi << np.uint64(32) | lo, mem[a["member_ids_rows"].astype(np.int64)])
