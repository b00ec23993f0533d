"""GPU parity: SumcheckProof::prove / ZeroCheckProof::prove / eq table against the oracle, bit-exact, on the
reference's own test shapes (sumcheck.rs:159-230, zerocheck.rs:85-211), the golden file, seeded random shapes up to
BASELINE.json's 2^24, and edge cases (0 and 1 variables, constants, unused tables, false claims, cancelling terms)."""
import json
import os
import random

import numpy as np
import pytest

import quill_zkvm_b200 as q
from oracle import coracle as co
from oracle import pyref as py
from tests import util

pytestmark = pytest.mark.gpu
FR = py.FR
G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))
hx = lambda s: int(s, 16)  # noqa: E731
NCPU = os.cpu_count() or 1


def gpu_prove(ctx, n, tables, nodes, consts, claimed, domain, zerocheck=False, device_tables=False):
    store = q.VirtualPolynomialStore(n)
    bufs = []
    for t in tables:
        if device_tables:
            b = ctx.upload(t)
            bufs.append(b)
            store.allocate_polynomial(b)
        else:
            store.allocate_polynomial(t)
    h = store.new_virtual_from_expr(util.to_qexpr(nodes, consts))
    tr = q.Transcript(domain, ctx)
    if zerocheck:
        proof, claim = q.ZeroCheckProof.prove(ctx, store, h, tr)
        sc = proof.sumcheck_proof
        z = proof.z
    else:
        sc, claim = q.SumcheckProof.prove(ctx, n, store, h, claimed, tr)
        z = None
    for b in bufs:
        b.free()
    return sc, claim, tr.state.copy(), z


def oracle_prove(n, tables, nodes, consts, claimed, domain, zerocheck=False, threads=1):
    """the oracle's proof; o["state"] is its final transcript state"""
    st = co.transcript_new(domain)
    o = co.sumcheck_prove(n, tables, nodes, consts, claimed, st, max_coeffs=q._lib.QZ_MAX_ROUND_COEFFS,
                          zerocheck=zerocheck, threads=threads)
    o["state"] = st
    return o


def assert_matches_oracle(n, got, o, zerocheck=False):
    """got = gpu_prove(...): every round polynomial and its length, the point, the evaluation, the state and z"""
    sc, claim, state, z = got
    assert [p.shape[0] for p in sc.r_polys] == o["lens"].tolist()
    for j in range(n):
        assert np.array_equal(sc.r_polys[j], o["coeffs"][j][: o["lens"][j]]), f"round {j}"
    assert np.array_equal(claim.point, o["point"])
    assert np.array_equal(claim.evaluation, o["evaluation"])
    assert state.tobytes() == o["state"].tobytes()
    if zerocheck:
        assert np.array_equal(z, o["z"])


def assert_same(ctx, n, tables, nodes, consts, claimed, domain, zerocheck=False, device_tables=False, threads=1):
    got = gpu_prove(ctx, n, tables, nodes, consts, claimed, domain, zerocheck, device_tables)
    o = oracle_prove(n, tables, nodes, consts, claimed, domain, zerocheck, threads)
    assert_matches_oracle(n, got, o, zerocheck)
    return got[0], got[1], o


def test_reference_sumcheck_test(ctx):
    g = G["sumcheck_test"]
    g1 = [((i >> 0) & 1) + 2 * ((i >> 1) & 1) + 3 * ((i >> 2) & 1) for i in range(8)]
    g2 = [((i >> 0) & 1) * 2 * ((i >> 1) & 1) + 3 * ((i >> 0) & 1) * ((i >> 2) & 1) for i in range(8)]
    nodes, consts = util.expr_product(2)
    sc, claim, st, _ = gpu_prove(ctx, 3, [co.to_mont(g1), co.to_mont(g2)], nodes, consts, co.fr1(48), b"sumcheck_test")
    assert [co.from_mont(p) for p in sc.r_polys] == [[hx(c) for c in p] for p in g["r_polys"]]
    assert co.from_mont(claim.point) == [hx(x) for x in g["point"]]
    assert co.from_mont(claim.evaluation)[0] == hx(g["evaluation"])
    assert st.tobytes().hex() == g["state_end"]
    # the reference's own assertions: verifier agrees, closed form at the point
    mc = q._lib.QZ_MAX_ROUND_COEFFS
    coeffs = np.zeros((3, mc, 32), dtype=np.uint8)
    for j, p in enumerate(sc.r_polys):
        coeffs[j, : p.shape[0]] = p
    ok, vp, ve = co.sumcheck_verify(3, co.fr1(48), coeffs, np.array([p.shape[0] for p in sc.r_polys], np.uint32),
                                    co.transcript_new(b"sumcheck_test"))
    assert ok and np.array_equal(vp, claim.point) and np.array_equal(ve, claim.evaluation)
    pt = co.from_mont(claim.point)
    assert (pt[0] + 2 * pt[1] + 3 * pt[2]) * (pt[0] * 2 * pt[1] + 3 * pt[0] * pt[2]) % FR == hx(g["evaluation"])


@pytest.mark.parametrize("name", ["zerocheck_test", "zerocheck_test_not_zero"])
def test_reference_zerocheck_tests(ctx, name):
    g = G[name]
    hz = py.e_sub(py.e_mul(py.e_in(0), py.e_in(0)), py.e_in(1))
    nodes, consts = util.expr_from_py(hz)
    tabs = [co.to_mont(list(range(8))), co.to_mont(g["g2"])]
    sc, claim, st, z = gpu_prove(ctx, 3, tabs, nodes, consts, None, b"zerocheck_test", zerocheck=True)
    assert [co.from_mont(p) for p in sc.r_polys] == [[hx(c) for c in p] for p in g["r_polys"]]
    assert co.from_mont(claim.point) == [hx(x) for x in g["point"]]
    assert co.from_mont(claim.evaluation)[0] == hx(g["evaluation"])
    assert co.from_mont(z) == [hx(x) for x in g["z"]]
    assert st.tobytes().hex() == g["state_end"]


def test_golden_product_and_mixed(ctx):
    g = G["product3_n6"]
    tabs = [co.to_mont([hx(x) for x in tb]) for tb in g["tables"]]
    nodes, consts = util.expr_product(3)
    sc, claim, st, _ = gpu_prove(ctx, 6, tabs, nodes, consts, co.fr1(hx(g["claimed_sum"])), b"sumcheck_bench")
    assert [co.from_mont(p) for p in sc.r_polys] == [[hx(c) for c in p] for p in g["r_polys"]]
    assert st.tobytes().hex() == g["state_end"]
    gm = G["mixed_n6"]
    hm = py.e_add(py.e_sub(py.e_mul(py.e_in(0), py.e_in(1)), py.e_in(3)),
                  py.e_mul(py.e_const(7), py.e_mul(py.e_in(2), py.e_in(2))))
    nodes, consts = util.expr_from_py(hm)
    sc, claim, st, _ = gpu_prove(ctx, 6, tabs, nodes, consts, co.fr1(123), b"mixed")
    assert [co.from_mont(p) for p in sc.r_polys] == [[hx(c) for c in p] for p in gm["r_polys"]]
    assert co.from_mont(claim.evaluation)[0] == hx(gm["evaluation"]) and st.tobytes().hex() == gm["state_end"]


@pytest.mark.parametrize("n", [0, 1, 2, 5, 10, 11, 12, 13, 16])
@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_product_fast_path_sizes(ctx, n, k):
    """crosses the single-block tail (<= 2^11) / streaming-round boundary for every fast-path arity"""
    tabs = [util.rand_fr(1 << n, 100 * n + t) for t in range(k)]
    nodes, consts = util.expr_product(k)
    assert_same(ctx, n, tabs, nodes, consts, co.fr1(12345), b"prod")


@pytest.mark.parametrize("n", [1, 4, 12, 14])
def test_generic_expressions(ctx, n):
    rnd = random.Random(n)
    k = 5
    tabs = [util.rand_fr(1 << n, 7 * n + t) for t in range(k)]
    exprs = [
        py.e_sub(py.e_mul(py.e_in(0), py.e_in(0)), py.e_in(1)),                       # g0^2 - g1 (repeated input)
        py.e_add(py.e_mul(py.e_in(0), py.e_in(1)), py.e_mul(py.e_in(2), py.e_in(3))),  # sum of products
        py.e_const(rnd.randrange(FR)),                                                # constant only: summed per point
        py.e_add(py.e_in(4), py.e_const(5)),                                          # degree 1
        py.e_sub(py.e_mul(py.e_in(0), py.e_in(1)), py.e_mul(py.e_in(1), py.e_in(0))),  # cancels to zero: empty polys
        py.e_mul(py.e_mul(py.e_mul(py.e_in(0), py.e_in(1)), py.e_mul(py.e_in(2), py.e_in(3))),
                 py.e_add(py.e_in(4), py.e_in(0))),                                   # degree 5
    ]
    for i, e in enumerate(exprs):
        nodes, consts = util.expr_from_py(e)
        sc, claim, o = assert_same(ctx, n, tabs, nodes, consts, co.fr1(i), b"generic%d" % i)
        if i == 4:
            assert all(p.shape[0] == 0 for p in sc.r_polys)


def _power(e, m):
    """e^m as a balanced tree of products"""
    if m == 1:
        return e
    return py.e_mul(_power(e, m // 2), _power(e, m - m // 2))


@pytest.mark.parametrize("deg", [29, 30, 31, 32])
@pytest.mark.parametrize("n", [3, 13])
def test_high_degree_round_polynomials(ctx, deg, n):
    """round polynomials of 30..33 coefficients: from 31 on `state ‖ len ‖ coeffs` no longer fits one blake3 chunk
    (32 + 8 + 32 * 31 > 1024), which the device transcript must hash as a two-chunk tree like the reference's blake3"""
    tabs = [util.rand_fr(1 << n, 31 * n + t) for t in range(2)]
    e = py.e_add(_power(py.e_in(0), deg), py.e_mul(py.e_in(1), py.e_const(3)))
    nodes, consts = util.expr_from_py(e)
    sc, claim, o = assert_same(ctx, n, tabs, nodes, consts, co.fr1(deg), b"deg%d" % deg, threads=NCPU)
    assert sc.r_polys[0].shape[0] == deg + 1
    if deg < 32:  # the zero-check multiplies by eq: one more degree
        assert_same(ctx, n, tabs, nodes, consts, None, b"zdeg%d" % deg, zerocheck=True, threads=NCPU)


@pytest.mark.parametrize("n,k", [(17, 3), (18, 3), (19, 3), (20, 3), (19, 1), (19, 2), (20, 4)])
def test_product_sizes_across_the_persistent_rounds(ctx, n, k):
    """2^17 .. 2^20: the proof starts inside sc_mid (<= 2^18 entries), or streams one or two rounds and hands over to it"""
    tabs = [util.rand_fr(1 << n, 300 * n + t) for t in range(k)]
    nodes, consts = util.expr_product(k)
    assert_same(ctx, n, tabs, nodes, consts, co.fr1(7), b"mid", threads=NCPU, device_tables=True)
    if k <= 3:
        assert_same(ctx, n, tabs, nodes, consts, None, b"midzc", zerocheck=True, threads=NCPU, device_tables=True)


@pytest.mark.parametrize("n", [18, 19])
def test_generic_expression_across_the_persistent_rounds(ctx, n):
    tabs = [util.rand_fr(1 << n, 17 * n + t) for t in range(4)]
    e = py.e_add(py.e_sub(py.e_mul(py.e_in(0), py.e_in(1)), py.e_in(3)), py.e_mul(py.e_const(7), py.e_mul(py.e_in(2), py.e_in(2))))
    nodes, consts = util.expr_from_py(e)
    assert_same(ctx, n, tabs, nodes, consts, co.fr1(1), b"midgen", threads=NCPU)
    assert_same(ctx, n, tabs, nodes, consts, None, b"midgenzc", zerocheck=True, threads=NCPU)


@pytest.mark.parametrize("k,deg", [(6, 2), (8, 3), (3, 7), (2, 6), (9, 2), (4, 8)])
@pytest.mark.parametrize("n", [6, 13, 15])
def test_shapes_around_the_split_pass(ctx, k, deg, n):
    """The short rounds run the split pass (one work item per folded element, then per (pair, evaluation point)) when at
    most 8 tables and 8 evaluation points are involved, and whole pairs per thread otherwise: both sides of each limit,
    with row widths of 1, 2 and 4 warps per evaluation point."""
    tabs = [util.rand_fr(1 << n, 41 * n + 7 * k + t) for t in range(k)]
    # sum over the tables of g_t * g_{t+1} ... (deg factors, wrapping around) + a constant: degree `deg`, all k tables used
    e = py.e_const(11)
    for t in range(k):
        term = py.e_in(t)
        for j in range(1, deg if t == 0 else min(deg, 2)):
            term = py.e_mul(term, py.e_in((t + j) % k))
        e = py.e_add(e, term)
    nodes, consts = util.expr_from_py(e)
    assert_same(ctx, n, tabs, nodes, consts, co.fr1(k * deg), b"split%d" % k, threads=NCPU)
    if deg < 8:
        assert_same(ctx, n, tabs, nodes, consts, None, b"splitzc%d" % k, zerocheck=True, threads=NCPU, device_tables=True)


def test_logup_shaped_expression(ctx):
    """the batched expression of multiset_check.rs:132-157: (d_l (gamma + f) - 1) + alpha (d_r (gamma + g) - 1) ... times eq via zerocheck"""
    n = 13
    tabs = [util.rand_fr(1 << n, 900 + t) for t in range(4)]
    gamma, alpha = 0x1234567, 0x7654321
    one = py.e_const(1)
    left = py.e_sub(py.e_mul(py.e_in(2), py.e_add(py.e_in(0), py.e_const(gamma))), one)
    right = py.e_sub(py.e_mul(py.e_in(3), py.e_add(py.e_in(1), py.e_const(gamma))), one)
    e = py.e_add(left, py.e_mul(py.e_const(alpha), right))
    nodes, consts = util.expr_from_py(e)
    assert_same(ctx, n, tabs, nodes, consts, None, b"logup", zerocheck=True)


@pytest.mark.parametrize("n", [0, 1, 3, 12, 15])
def test_zerocheck_sizes(ctx, n):
    tabs = [util.rand_fr(1 << n, 50 + t) for t in range(3)]
    e = py.e_sub(py.e_mul(py.e_in(0), py.e_in(1)), py.e_in(2))
    nodes, consts = util.expr_from_py(e)
    assert_same(ctx, n, tabs, nodes, consts, None, b"zc", zerocheck=True)


@pytest.mark.parametrize("k", [1, 2, 3])
@pytest.mark.parametrize("n", [12, 13, 16, 18])
def test_zerocheck_product_fast_path(ctx, n, k, monkeypatch):
    """h = a product of k tables: the eq-factored rounds (weights instead of a streamed eq table, round polynomial =
    linear factor x degree-k sum) must give the bytes of the reference's formulation -- against the oracle, with host and
    device tables, and against the library's own streamed-eq path (QZ_ZC_STREAM_EQ=1)."""
    tabs = [util.rand_fr(1 << n, 900 + 10 * n + t) for t in range(k)]
    if n == 13:  # a table that vanishes on half the cube and a constant one: trailing-zero trimming of s_j
        tabs[0][::2] = 0
        if k > 1:
            tabs[1][:] = co.fr1(5)
    nodes, consts = util.expr_product(k)
    sc, claim, o = assert_same(ctx, n, tabs, nodes, consts, None, b"zc_fast", zerocheck=True, threads=NCPU)
    assert_same(ctx, n, tabs, nodes, consts, None, b"zc_fast", zerocheck=True, device_tables=True, threads=NCPU)
    monkeypatch.setenv("QZ_ZC_STREAM_EQ", "1")
    sc2, claim2, state2, z2 = gpu_prove(ctx, n, tabs, nodes, consts, None, b"zc_fast", zerocheck=True)
    assert all(np.array_equal(a, b) for a, b in zip(sc.r_polys, sc2.r_polys)) and len(sc.r_polys) == len(sc2.r_polys)
    assert np.array_equal(claim.evaluation, claim2.evaluation) and np.array_equal(claim.point, claim2.point)


def test_unused_store_tables_and_device_tables(ctx):
    n = 12
    tabs = [util.rand_fr(1 << n, 300 + t) for t in range(5)]
    nodes = [(0, 3, 0), (0, 1, 0), (3, 0, 1)]  # h = g3 * g1; g0, g2, g4 are in the store but unused
    consts = np.zeros((0, 32), dtype=np.uint8)
    assert_same(ctx, n, tabs, nodes, consts, co.fr1(1), b"unused")
    assert_same(ctx, n, tabs, nodes, consts, co.fr1(1), b"unused", device_tables=True)


def test_eq_table_matches_oracle(ctx):
    for n in (0, 1, 2, 5, 9, 14):
        pt = util.rand_fr(n, 77 + n)
        got = q.fast_eq_eval_hypercube(ctx, n, pt)
        assert np.array_equal(got, co.eq_table(pt)), n
    g = G["eq_n5"]
    got = q.fast_eq_eval_hypercube(ctx, 5, co.to_mont([hx(x) for x in g["point"]]))
    assert co.from_mont(got) == [hx(x) for x in g["table"]]


def test_errors(ctx):
    n = 4
    tabs = [util.rand_fr(1 << n, 1)]
    store = q.VirtualPolynomialStore(n)
    store.allocate_polynomial(tabs[0])
    with pytest.raises(AssertionError):  # virtual_polynomial.rs:162-166
        store.allocate_polynomial(util.rand_fr(3, 1))
    h = store.new_virtual_from_expr(q.VirtualPolyExpr.Input(7))  # index outside the store
    with pytest.raises(q.QuillError) as e:
        q.SumcheckProof.prove(ctx, n, store, h, co.fr1(0), q.Transcript(b"x", ctx))
    assert e.value.status == q._lib.QZ_ERR_EXPR


@pytest.mark.parametrize("n", [20, 24])
def test_baseline_sizes_product3(ctx, n):
    """BASELINE.json config 3: degree-3 product of 2^n-entry tables, inputs generated on the device (the 2^24 case is
    1.5 GiB), oracle on all host cores.  Also checks size-independent properties: the verifier accepts with the true
    sum, and the final claim equals the product of the tables' MLE evaluations at the point."""
    bufs = [ctx.random_fr(1 << n, 1000 + t) for t in range(3)]
    tabs = [b.download().reshape(-1, 32) for b in bufs]
    store = q.VirtualPolynomialStore(n)
    for b in bufs:
        store.allocate_polynomial(b)
    h = store.new_virtual_from_expr(util.to_qexpr(*util.expr_product(3)))
    claimed = co.fr1(777)
    tr = q.Transcript(b"sumcheck_bench", ctx)
    sc, claim = q.SumcheckProof.prove(ctx, n, store, h, claimed, tr)
    for b in bufs:
        b.free()
    st = co.transcript_new(b"sumcheck_bench")
    nodes, consts = util.expr_product(3)
    o = co.sumcheck_prove(n, tabs, nodes, consts, claimed, st, max_coeffs=8, threads=NCPU)
    for j in range(n):
        assert np.array_equal(sc.r_polys[j], o["coeffs"][j][: o["lens"][j]]), f"round {j}"
    assert np.array_equal(claim.point, o["point"]) and np.array_equal(claim.evaluation, o["evaluation"])
    assert tr.state.tobytes() == st.tobytes()
    evs = [co.mle_evaluate(t, claim.point) for t in tabs]
    prod = co.field_op(0, 2, co.field_op(0, 2, evs[0], evs[1]), evs[2])
    assert np.array_equal(prod.reshape(32), claim.evaluation)
    # s_0(0) + s_0(1) is the true sum: prove again with it and the verifier accepts
    c0 = co.from_mont(sc.r_polys[0])
    true_sum = (2 * c0[0] + sum(c0[1:])) % FR
    coeffs = np.zeros((n, 8, 32), dtype=np.uint8)
    store = q.VirtualPolynomialStore(n)
    for t in tabs:
        store.allocate_polynomial(t)
    h = store.new_virtual_from_expr(util.to_qexpr(*util.expr_product(3)))
    sc2, claim2 = q.SumcheckProof.prove(ctx, n, store, h, co.fr1(true_sum), q.Transcript(b"v", ctx))
    for j, p in enumerate(sc2.r_polys):
        coeffs[j, : p.shape[0]] = p
    ok, vp, ve = co.sumcheck_verify(n, co.fr1(true_sum), coeffs, np.array([p.shape[0] for p in sc2.r_polys], np.uint32),
                                    co.transcript_new(b"v"))
    assert ok and np.array_equal(ve, claim2.evaluation)


@pytest.mark.parametrize("n", [20, 24])
def test_baseline_sizes_zerocheck_product3(ctx, n):
    """BASELINE.json config 3, zero-check form: h = f * g * e with the eq table as a fourth factor (degree 4), z drawn on
    the device, tables resident on the device; every round polynomial, z, the point, the claim (already divided by
    eq(z, r), zerocheck.rs:34-40) and the transcript state against the oracle on all host cores."""
    bufs = [ctx.random_fr(1 << n, 2000 + t) for t in range(3)]
    tabs = [b.download().reshape(-1, 32) for b in bufs]
    nodes, consts = util.expr_product(3)
    store = q.VirtualPolynomialStore(n)
    for b in bufs:
        store.allocate_polynomial(b)
    h = store.new_virtual_from_expr(util.to_qexpr(nodes, consts))
    tr = q.Transcript(b"zerocheck_bench", ctx)
    proof, claim = q.ZeroCheckProof.prove(ctx, store, h, tr)
    for b in bufs:
        b.free()
    st = co.transcript_new(b"zerocheck_bench")
    o = co.sumcheck_prove(n, tabs, nodes, consts, None, st, max_coeffs=q._lib.QZ_MAX_ROUND_COEFFS, zerocheck=True,
                          threads=NCPU)
    sc = proof.sumcheck_proof
    assert [p.shape[0] for p in sc.r_polys] == o["lens"].tolist()
    for j in range(n):
        assert np.array_equal(sc.r_polys[j], o["coeffs"][j][: o["lens"][j]]), f"round {j}"
    assert np.array_equal(proof.z, o["z"]) and np.array_equal(claim.point, o["point"])
    assert np.array_equal(claim.evaluation, o["evaluation"]) and tr.state.tobytes() == st.tobytes()
    # the claim is h at the point: the product of the three tables' MLE evaluations (zerocheck.rs:142-158)
    evs = [co.mle_evaluate(t, claim.point) for t in tabs]
    prod = co.field_op(0, 2, co.field_op(0, 2, evs[0], evs[1]), evs[2])
    assert np.array_equal(prod.reshape(32), claim.evaluation)


def test_2_26_product3_verifier_and_mle(ctx):
    """the upper end of north_star's range (2^16..2^26; 3 x 2 GiB of tables): every round polynomial, the point, the
    evaluation and the transcript state against the oracle on all host cores (the device buffers are freed first), and
    the size-independent properties: the reference's verifier (sumcheck.rs:116-150) accepts the transcript with the
    true sum and reproduces the prover's point and claim, and the claim equals the product of the tables' MLE
    evaluations at that point (the reference's own acceptance test, sumcheck.rs:216-229)."""
    n = 26
    bufs = [ctx.random_fr(1 << n, 2600 + t) for t in range(3)]
    store = q.VirtualPolynomialStore(n)
    for b in bufs:
        store.allocate_polynomial(b)
    h = store.new_virtual_from_expr(util.to_qexpr(*util.expr_product(3)))
    sc, _ = q.SumcheckProof.prove(ctx, n, store, h, co.fr1(1), q.Transcript(b"probe", ctx))
    c0 = co.from_mont(sc.r_polys[0])
    true_sum = (2 * c0[0] + sum(c0[1:])) % FR  # s_0(0) + s_0(1)
    tr = q.Transcript(b"sumcheck_bench", ctx)
    sc, claim = q.SumcheckProof.prove(ctx, n, store, h, co.fr1(true_sum), tr)
    tabs = []
    for b in bufs:
        tabs.append(b.download().reshape(-1, 32))
        b.free()
    ctx.trim()
    nodes, consts = util.expr_product(3)
    o = oracle_prove(n, tabs, nodes, consts, co.fr1(true_sum), b"sumcheck_bench", threads=NCPU)
    assert_matches_oracle(n, (sc, claim, tr.state, None), o)
    coeffs = np.zeros((n, 8, 32), dtype=np.uint8)
    for j, p in enumerate(sc.r_polys):
        coeffs[j, : p.shape[0]] = p
    st = co.transcript_new(b"sumcheck_bench")
    ok, vp, ve = co.sumcheck_verify(n, co.fr1(true_sum), coeffs, np.array([p.shape[0] for p in sc.r_polys], np.uint32), st)
    assert ok and np.array_equal(vp, claim.point) and np.array_equal(ve, claim.evaluation)
    assert st.tobytes() == tr.state.tobytes()
    prod = None
    for t in tabs:
        ev = co.mle_evaluate(t, claim.point)
        prod = ev if prod is None else co.field_op(0, 2, prod, ev)
    assert np.array_equal(prod.reshape(32), claim.evaluation)
