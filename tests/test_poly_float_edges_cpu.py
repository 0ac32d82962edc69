"""The polygon float-edge cases of tests/_poly_float_edges.py, checked on the CPU: the oracle agrees with the independent
Python restatement on them, they tell every mutant of the float rules apart from the reference in every size class,
and they contain what the families promise (signed-zero ties, subnormal products, overflowing differences,
non-finite values in y only)."""
import numpy as np

import _poly_float_edges as E


def _all_kills(oracle):
    """Kill arrays of every mutant over the kill set followed by the non-finite set, and the class of each case."""
    cs, kills = E.kill_cases(oracle)
    nf, _, _ = E.nonfinite_cases(oracle)
    with np.errstate(all="ignore"):
        nk, _ = E.kill_matrix(oracle, *nf.packed())
    return {m: np.concatenate([kills[m], nk[m]]) for m in kills}, cs.classes + nf.classes


def test_kill_table(oracle):
    kills, classes = _all_kills(oracle)
    names = [c[0] for c in E.CLASSES]
    cls = np.array(classes)
    table = {m: [int((k & (cls == c)).sum()) for c in names] for m, k in kills.items()}
    print("\nkills per mutant and size class (kill set + non-finite set)")
    print("%-13s" % "mutant" + "".join("%7s" % c for c in names) + "  total")
    for m, row in table.items():
        print("%-13s" % m + "".join("%7d" % v for v in row) + "%7d" % sum(row))
    for m, (_, rule) in oracle.MUTANTS.items():
        missing = [c for c, v in zip(names, table[m]) if v == 0]
        assert not missing, f"mutant {m} ({rule}) survives in classes {missing}"


def test_kill_set_covers_every_class(oracle):
    cs, _ = E.kill_cases(oracle)
    nf, flagged, _ = E.nonfinite_cases(oracle)
    names = {c[0] for c in E.CLASSES}
    assert set(cs.classes) == names and set(nf.classes) == names
    assert flagged.any() and (~flagged).any()


def test_oracle_agrees_with_pyref_on_small_cases(oracle):
    """The unmutated C oracle against oracle/pyref.py (with the oracle's atan2f) on every selected case of up to 16
    points: the two restatements agree at signed zeros, subnormals and overflow, not only on ordinary inputs."""
    from oracle import pyref

    cs, _ = E.kill_cases(oracle)
    atan2 = lambda y, x: np.float32(oracle.atan2f(float(y), float(x)))
    checked = 0
    with np.errstate(all="ignore"):
        for p, (off, prime) in zip(cs.polys, cs.op):
            n = len(p)
            if n > E.PYREF_MAX_N:
                continue
            r = oracle.polygon_batch(p, np.array([0, n]), offset_prime=[off, prime])
            st_c = int(r["status"][0])
            if st_c & ~(4 | 8 | 128):  # arena caps and statuses outside pyref's vocabulary
                continue
            order = oracle.unirand_sequence(n, int(off), int(prime))
            ids, st = pyref.triangulate_ids(p, order, atan2=atan2)
            cap = 3 * (n - 2)
            if st == "null_unwrap":
                assert st_c & 4, (p.tolist(), off, prime)
            else:
                exp = np.full(cap, 0xFFFFFFFF, dtype=np.uint32)
                m = min(cap, len(ids))
                exp[:m] = ids[:m]
                assert np.array_equal(exp, r["ids"]), (p.tolist(), off, prime)
                assert (len(ids) > cap) == bool(st_c & 8) and (len(ids) < cap) == bool(st_c & 128)
            checked += 1
    assert checked >= 20, checked


def test_generator_delivers_what_it_claims(oracle):
    cs, _ = E.kill_cases(oracle)
    nf, flagged, desc = E.nonfinite_cases(oracle)
    with np.errstate(all="ignore"):
        _, r = E.per_polygon_outputs(oracle, *cs.packed())
        _, rn = E.per_polygon_outputs(oracle, *nf.packed())
    assert {c for c, p in zip(cs.classes, cs.polys) if E.has_pm0_y_tie(p)} == {c[0] for c in E.CLASSES}
    assert sum(E.has_subnormal_product(p) for p in cs.polys) >= 10
    assert sum(E.has_overflowing_difference(p) for p in cs.polys) >= 5
    # non-finite: flagged exactly where expected, including values in y only, in every class
    assert np.array_equal(rn["status"] == 2, flagged), [d for d, s, f in zip(desc, rn["status"], flagged) if (s == 2) != f]
    y_only = [d[0] for d, f, p in zip(desc, flagged, nf.polys) if f and d[2] == "y" and np.isfinite(p[:, 0]).all()]
    assert set(y_only) == {c[0] for c in E.CLASSES}
    assert any(np.abs(p).max() == E.FLT_MAX for p, f in zip(nf.polys, flagged) if not f)
    # a zero bbox component is always +0 (the accumulators start at +0 and a tie keeps them)
    for b in (r["bbox"], rn["bbox"]):
        z = b == 0
        assert not np.signbit(b[z]).any()
