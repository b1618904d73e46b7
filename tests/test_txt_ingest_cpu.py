"""TXT ingest (cuadmm_problem_from_txt <-> Problem::from_txt, src/problem.cu:11-83, src/utils/io.cu) — host code, no GPU.
The SDPT3-style files are written from a committed fixture, read back through the C ABI and compared with the source
arrays.  The triplets hold unique (row, col) pairs, so the sorted CSC they are compared with is also the one result the
reference's COO_to_CSC can give on them."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

import cuadmm_b200 as cu
from util_problems import load_fixture, synthetic_sdp, write_txt


def _csc(P):
    M = sp.csc_matrix((P["vals"], P["row_ids"], P["col_ptrs"]), shape=(P["vec_len"], P["con_num"]))
    M.sort_indices()
    return M


@pytest.mark.parametrize("slash", ["/", ""])
def test_round_trip_fixture(tmp_path, slash):
    P = load_fixture("hinf12")
    d = str(tmp_path / "hinf12")
    write_txt(P, d)
    Q = cu.Problem(d + slash)          # the reference needs the trailing '/', both are accepted here
    assert (Q.vec_len, Q.con_num, Q.mat_num) == (P["vec_len"], P["con_num"], len(P["blk"]))
    assert not Q.has_warm and Q.array(8) is None
    M = _csc(P)
    assert np.array_equal(Q.array(0), M.indptr) and np.array_equal(Q.array(1), M.indices)
    assert np.array_equal(Q.array(2), M.data)                      # "%.17g" round-trips doubles exactly
    assert np.array_equal(Q.array(7), np.asarray(P["blk"], np.int32))
    ob = np.argsort(P["b_idx"]); oc = np.argsort(P["C_idx"])
    assert np.array_equal(Q.array(3), np.asarray(P["b_idx"])[ob]) and np.array_equal(Q.array(4), np.asarray(P["b_val"])[ob])
    assert np.array_equal(Q.array(5), np.asarray(P["C_idx"])[oc]) and np.array_equal(Q.array(6), np.asarray(P["C_val"])[oc])
    Q.close()


def test_shuffled_triplets_plain_blk_lines_and_warm_start(tmp_path):
    P = synthetic_sdp([3, 5, 2, 4], 12, seed=7)
    d = str(tmp_path / "p") + "/"
    write_txt(P, d)
    # blk.txt without the type letter ("<n>" lines, src/utils/io.cu:311-326), At.txt triplets in random order
    open(d + "blk.txt", "w").write("".join(f"{int(n)}\n" for n in P["blk"]))
    lines = open(d + "At.txt").read().splitlines()
    rng = np.random.default_rng(0)
    rng.shuffle(lines)
    open(d + "At.txt", "w").write("\n".join(lines) + "\n")
    x0 = rng.standard_normal(P["vec_len"]); y0 = rng.standard_normal(P["con_num"]); s0 = rng.standard_normal(P["vec_len"])
    for name, v in (("X", x0), ("y", y0), ("S", s0)):
        open(d + name + ".txt", "w").write("".join(f"{t:.17g}\n" for t in v))
    Q = cu.Problem(d, warm_start=True)
    M = _csc(P)
    assert np.array_equal(Q.array(0), M.indptr) and np.array_equal(Q.array(1), M.indices) and np.array_equal(Q.array(2), M.data)
    assert Q.has_warm
    assert np.array_equal(Q.array(8), x0) and np.array_equal(Q.array(9), y0) and np.array_equal(Q.array(10), s0)
    Q.close()


def test_errors_are_returned_not_fatal(tmp_path):
    with pytest.raises(cu.CuadmmError):
        cu.Problem(str(tmp_path / "does_not_exist") + "/")
    P = synthetic_sdp([3, 2], 4, seed=1)
    d = str(tmp_path / "bad") + "/"
    write_txt(P, d)
    open(d + "blk.txt", "w").write("s 3\nq 2\n")      # only 's' blocks are accepted (src/problem.cu:28-36)
    with pytest.raises(cu.CuadmmError):
        cu.Problem(d)
