"""Linear ('l') and free ('u') blocks next to PSD blocks, host side (no GPU): TXT ingest, host-only typed plans and
shards, and the typed oracle's own checks against scipy's LP solver and against known optima."""
import numpy as np
import pytest
import resource

import cuadmm_b200 as cu
import cones_util as cz

MIX = [("s", 3), ("l", 7), ("u", 4), ("s", 5), ("l", 1), ("l", 2), ("u", 3), ("s", 1)]


def _mix_problem(seed=0, m=20):
    return cz.typed_synthetic(MIX, m, seed=seed)


def test_txt_ingest_of_typed_blocks(tmp_path):
    P = _mix_problem()
    d = str(tmp_path / "mix") + "/"
    cz.write_txt(P, d)
    Q = cu.Problem(d)
    assert Q.vec_len == P["vec_len"] == 6 + 7 + 4 + 15 + 1 + 2 + 3 + 1
    assert Q.mat_num == len(MIX) and Q.blk_types == "slusllus"
    assert np.array_equal(Q.array(7), P["blk"])
    R = cz.read_problem_txt(d)
    assert R["types"] == Q.blk_types and R["vec_len"] == Q.vec_len
    Q.close()
    # an At row index past the typed vec_len (it would fit an all-'s' reading of the same sizes)
    lines = open(d + "At.txt").read().splitlines()
    open(d + "At.txt", "w").write("\n".join(lines + [f"{P['vec_len']} 0 1.0"]) + "\n")
    with pytest.raises(cu.CuadmmError) as e:
        cu.Problem(d)
    assert e.value.code == -5 and "row index" in str(e.value)
    open(d + "At.txt", "w").write("\n".join(lines) + "\n")
    # warm start: X.txt must have the typed length
    rng = np.random.default_rng(1)
    for name, n in (("X", P["vec_len"]), ("y", P["con_num"]), ("S", P["vec_len"])):
        open(d + name + ".txt", "w").write("".join(f"{t:.17g}\n" for t in rng.standard_normal(n)))
    Q = cu.Problem(d, warm_start=True)
    assert Q.has_warm and Q.array(8).shape == (P["vec_len"],)
    Q.close()
    open(d + "X.txt", "w").write("".join(f"{t:.17g}\n" for t in rng.standard_normal(P["vec_len"] + 1)))
    with pytest.raises(cu.CuadmmError) as e:
        cu.Problem(d, warm_start=True)
    assert e.value.code == -5 and "warmstarted X" in str(e.value)
    # bare sizes stay PSD; any other letter is still rejected
    open(d + "blk.txt", "w").write("3\nl 7\nu 4\ns 5\nl 1\nl 2\nu 3\n1\n")
    Q = cu.Problem(d)
    assert Q.blk_types == "slusllus" and Q.vec_len == P["vec_len"]
    Q.close()
    open(d + "blk.txt", "w").write("s 3\nq 2\n")
    with pytest.raises(cu.CuadmmError) as e:
        cu.Problem(d)
    assert e.value.code == -5


def test_host_plan_of_typed_blocks():
    blk = [n for _, n in MIX]
    types = "".join(t for t, _ in MIX)
    p = cu.Plan(blk, device=-1, types=types)
    assert p.vec_len == int(cz.svec_offsets(blk, types)[-1]) and p.nblk == len(MIX)
    # the reference-layout helpers have no place for 'l' / 'u' blocks
    for call in (p.sizes, p.totals, lambda: p.start_indices(0), p.maps):
        with pytest.raises(cu.CuadmmError) as e:
            call()
        assert e.value.code == -1 and "'l'/'u'" in str(e.value)
    # the same plan without types keeps them
    q = cu.Plan(blk, device=-1)
    assert q.vec_len == int(cz.svec_offsets(blk)[-1]) and len(q.maps()[0]) == q.vec_len
    # types=None and an all-'s' string are the same plan
    r = cu.Plan(blk, device=-1, types="s" * len(blk))
    assert all(np.array_equal(a, b) for a, b in zip(q.sizes(), r.sizes()))
    assert np.array_equal(q.totals(), r.totals()) and np.array_equal(q.partition(3)[0], r.partition(3)[0])
    with pytest.raises(cu.CuadmmError):
        cu.Plan(blk, device=-1, types="q" + types[1:])
    with pytest.raises(ValueError):
        cu.Plan(blk, device=-1, types=types[:-1])


def test_huge_linear_block_builds_without_quadratic_memory():
    # n = 1e7: an n^2 (8e14 B) or n(n+1)/2 allocation would fail outright, and n^2 arithmetic would take hours
    n = 10_000_000
    before = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    p = cu.Plan([40, n, 7], device=-1, types="sls")
    assert p.vec_len == 820 + n + 28 and p.nblk == 3
    owner, cost = p.partition(2)
    assert owner[1] != owner[0] or owner[1] != owner[2]
    sh = cu.Shard([40, n, 7], 2, int(owner[1]), types="sls")
    assert sh.vec_len == p.vec_len and n <= sh.vec_len_local <= n + 848
    grown_kb = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss - before
    assert grown_kb < 2_000_000            # linear bookkeeping only (the shard's maps: 16 B per entry)


@pytest.mark.parametrize("world", [1, 2, 3])
def test_typed_shard_covers_every_entry_once(world):
    rng = np.random.default_rng(world)
    types = "".join(rng.choice(list("slu"), 40, p=[0.5, 0.3, 0.2]))
    blk = rng.integers(1, 60, 40).astype(np.int32)
    off = cz.svec_offsets(blk, types)
    vec_len = int(off[-1])
    seen = np.zeros(vec_len, np.int64)
    owners = None
    for r in range(world):
        sh = cu.Shard(blk, world, r, types=types)
        assert sh.vec_len == vec_len
        seen[sh.loc2glob] += 1
        # the local blocks in ascending global order, whole, with their own types
        assert np.all(np.diff(sh.local_block_ids) > 0)
        assert sh.local_types == "".join(types[k] for k in sh.local_block_ids)
        assert np.array_equal(sh.local_blk, blk[sh.local_block_ids])
        exp = np.concatenate([np.arange(off[k], off[k + 1]) for k in sh.local_block_ids]) if len(sh.local_block_ids) \
            else np.zeros(0, np.int64)
        assert np.array_equal(sh.loc2glob, exp)
        assert sh.vec_len_local == len(exp)
        if owners is None:
            owners = sh.owner.copy()
        assert np.array_equal(sh.owner, owners)          # every rank computes the same partition
        sh.close()
    assert np.all(seen == 1)
    # deterministic
    again = cu.Shard(blk, world, 0, types=types)
    assert np.array_equal(again.owner, owners)
    p = cu.Plan(blk, device=-1, types=types)
    assert np.array_equal(p.partition(world)[0], owners)


def test_all_psd_partition_unchanged_by_the_typed_entry_point():
    blk = np.random.default_rng(5).integers(1, 400, 300).astype(np.int32)
    for world in (2, 3, 8):
        a = cu.Shard(blk, world, 0)
        b = cu.Shard(blk, world, 0, types="s" * len(blk))
        assert np.array_equal(a.owner, b.owner) and np.array_equal(a.loc2glob, b.loc2glob)


# ------------------------------------------------------------------ the typed oracle's own checks
@pytest.mark.parametrize("n_free", [0, 8])
def test_oracle_lp_matches_linprog(n_free):
    P = cz.random_lp(40, n_free, 15, seed=1)
    f = cz.linprog_objective(P)
    o = cz.oracle_for(P)
    X, y, S, it = o.solve(20000, 1e-6, 500, 50, 100, 11000, 1.05)
    assert it < 20000
    assert abs(o.hist["pobj"][-1] - f) <= 1e-4 * abs(f)
    assert np.all(S[P["blk"][0]:] == 0.0)                  # the free part of S is exactly zero
    assert abs(P["pstar"] - f) <= 1e-9 * (1 + abs(f))     # the generator's optimum is the LP's


def test_oracle_typed_synthetic_reaches_known_optimum():
    P = cz.typed_synthetic([("s", 5), ("l", 30), ("s", 8), ("u", 6), ("s", 3), ("l", 12)], 40, seed=4)
    o = cz.oracle_for(P)
    X, y, S, it = o.solve(20000, 1e-6, 500, 50, 100, 11000, 1.05)
    assert it < 20000
    assert abs(o.hist["pobj"][-1] - P["pstar"]) <= 1e-4 * (1 + abs(P["pstar"]))


def test_oracle_projection_of_typed_blocks():
    blk = [n for _, n in MIX]
    types = "".join(t for t, _ in MIX)
    off = cz.svec_offsets(blk, types)
    x = np.random.default_rng(3).standard_normal(int(off[-1]))
    out = cz.project_typed(blk, types, x)
    for k, (t, n) in enumerate(MIX):
        seg, ref = out[off[k]:off[k + 1]], x[off[k]:off[k + 1]]
        if t == "l":
            assert np.array_equal(seg, np.maximum(ref, 0.0))
        elif t == "u":
            assert np.array_equal(seg, ref)
        else:
            assert np.allclose(seg, cz.onp.project_svec([n], ref), rtol=0, atol=1e-14)
