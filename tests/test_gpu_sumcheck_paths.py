"""GPU parity of the streaming-round variants that sumcheck_run selects only above 2^20 entries: the deferred-reduction
("wide") product and zero-check kernels, the four-table fold through the c_fold constant table, the skip-X=1 zero-check
rounds, round 0 on host tables copied in slices behind the kernel, and the generic expression folded through c_fold.

Every case records its launches under torch.profiler and asserts the kernel instances it exists for, then compares the
proof byte for byte with the oracle: every round polynomial and its length, the point, the evaluation, z and the final
transcript state.  Which instance runs depends on the occupancy the runtime reports (a round is wide from
8 * 128 * SMs * blocks-per-SM pairs on), so the sizes are the ones that select each instance on a B200 (148 SMs; blocks
per SM as the kernels' register counts allow, 128 and 168 registers a thread):

  k = 3 product, wide        4 blocks / SM  ->  606,208 pairs: the first folding round is wide from 2^22 on
  k = 4 product, wide        3 blocks / SM  ->  454,656 pairs: wide from 2^21 on; round-0 slices of host tables at 2^23
  K = 3 zero-check, wide     3 blocks / SM  ->  454,656 pairs: the first folding round is wide from 2^21 on
  skip-X=1 zero-check rounds                    num_vars >= 21
  sliced round 0                                host tables, sumcheck, 2^21 entries or more
  generic fold by c_fold                        a folding round of 2^16 pairs or more
"""
import os
import re
import threading
from collections import Counter

import numpy as np
import pytest

import quill_zkvm_b200 as q
from oracle import coracle as co
from oracle import pyref as py
from tests import util
from tests.test_gpu_sumcheck import assert_matches_oracle, assert_same, gpu_prove, oracle_prove

pytestmark = pytest.mark.gpu
FR = py.FR
NCPU = os.cpu_count() or 1
FALSE_CLAIM = 0xF00D  # not the sum of any table set below


# ---- launch list -----------------------------------------------------------------------------------------------------
def kernel_name(raw: str):
    """'void qz::sc_round_prod<3, true, false>(qz::ScTables, ...)' -> 'qz::sc_round_prod<3, 1, 0>'; None if not ours"""
    s = raw.replace("(anonymous namespace)::", "")
    s = s[5:] if s.startswith("void ") else s
    s = s.split("(", 1)[0].strip()
    s = re.sub(r"\btrue\b", "1", re.sub(r"\bfalse\b", "0", s))
    s = re.sub(r"\s*,\s*", ", ", s)
    return s if s.startswith("qz::") else None


def launches(fn):
    """(fn(), Counter of the qz:: kernel instances fn launched), recorded by torch.profiler with CUDA activities"""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
    names = Counter()
    for e in prof.key_averages():
        nm = kernel_name(e.key)
        if nm:
            names[nm] += e.count
    assert names, "the profiler recorded no qz:: kernel"
    return out, names


def expect(names, present=(), absent=(), counts=None):
    """every instance in `present` ran, none matching a pattern in `absent` did, each in `counts` ran that often"""
    shown = dict(sorted(names.items()))
    for inst in present:
        assert names[inst] >= 1, f"{inst} did not run; launched: {shown}"
    for pat in absent:
        hit = [nm for nm in names if re.fullmatch(pat, nm)]
        assert not hit, f"{hit} ran; launched: {shown}"
    for inst, c in (counts or {}).items():
        assert names[inst] == c, f"{inst} ran {names[inst]} times, expected {c}; launched: {shown}"


def prod_inst(k, wide, fold):
    return f"qz::sc_round_prod<{k}, {wide}, {fold}>"


def zc_inst(k, wide, fold, skip1):
    return f"qz::sc_round_zc<{k}, {wide}, {fold}, {skip1}>"


GEN0, GEN1 = "qz::sc_round_generic<0>", "qz::sc_round_generic<1>"
WIDE = r"qz::sc_round_(prod|zc)<\d, 1(, \d)+>"
ANY_ZC = r"qz::sc_round_zc<.*>"


# ---- inputs and comparisons ----------------------------------------------------------------------------------------------
def device_tables(ctx, n, k, seed):
    """k tables of 2^n entries uniform below r (ctx.random_fr, like the bench's), downloaded"""
    out = []
    for t in range(k):
        b = ctx.random_fr(1 << n, seed + t)
        out.append(b.download().reshape(-1, 32))
        b.free()
    return out


def true_sum(sc):
    """s_0(0) + s_0(1) of a proof: the sum of h over the cube"""
    c = co.from_mont(sc.r_polys[0]) if sc.r_polys[0].shape[0] else [0]
    return co.fr1((2 * c[0] + sum(c[1:])) % FR)


def assert_same_proof(a, b):
    """two gpu_prove results carry the same bytes"""
    assert [p.shape[0] for p in a[0].r_polys] == [p.shape[0] for p in b[0].r_polys]
    for j, (x, y) in enumerate(zip(a[0].r_polys, b[0].r_polys)):
        assert np.array_equal(x, y), f"round {j}"
    assert np.array_equal(a[1].point, b[1].point) and np.array_equal(a[1].evaluation, b[1].evaluation)
    assert a[2].tobytes() == b[2].tobytes()
    if a[3] is not None or b[3] is not None:
        assert np.array_equal(a[3], b[3])


_REF = {}


def product_reference(ctx, zerocheck, n, k):
    """seeded product tables and the oracle's proof over them, shared by the switch and two-context tests"""
    key = (zerocheck, n, k)
    if key not in _REF:
        tabs = device_tables(ctx, n, k, 8000 + 10 * n + k)
        nodes, consts = util.expr_product(k)
        claimed = None if zerocheck else co.fr1(FALSE_CLAIM)
        _REF[key] = tabs, oracle_prove(n, tabs, nodes, consts, claimed, b"paths_ref", zerocheck, NCPU)
    return _REF[key]


def sumcheck_case(ctx, n, tabs, nodes, consts, domain, dev_expect, host_expect):
    """The proof with a false claim, then with the true sum.  Device tables (dev_expect not None) are pinned to the
    oracle; host tables (host_expect not None) to the device proof of the same inputs, or to the oracle when there is
    none.  *_expect: keyword arguments of `expect`.  Returns the last proof."""
    claimed = co.fr1(FALSE_CLAIM)
    for _ in range(2):
        dev = None
        if dev_expect is not None:
            (sc, claim, o), names = launches(lambda: assert_same(ctx, n, tabs, nodes, consts, claimed, domain,
                                                                 device_tables=True, threads=NCPU))
            expect(names, **dev_expect)
            dev = (sc, claim, o["state"], None)
        if host_expect is not None:
            if dev is None:
                (sc, claim, o), names = launches(lambda: assert_same(ctx, n, tabs, nodes, consts, claimed, domain,
                                                                     threads=NCPU))
            else:
                got, names = launches(lambda: gpu_prove(ctx, n, tabs, nodes, consts, claimed, domain))
                assert_same_proof(got, dev)
            expect(names, **host_expect)
        claimed = true_sum(sc)
    return sc


# ---- products --------------------------------------------------------------------------------------------------------------
# (n, k): (round 0 on device tables, folding rounds, round 0 of each of the 8 host-table slices); None: not run
PRODUCT_CASES = {
    (21, 1): (prod_inst(1, 0, 0), [prod_inst(1, 0, 1)], prod_inst(1, 0, 0)),
    (21, 2): (prod_inst(2, 0, 0), [prod_inst(2, 0, 1)], prod_inst(2, 0, 0)),
    (22, 3): (prod_inst(3, 1, 0), [prod_inst(3, 1, 1), prod_inst(3, 0, 1)], prod_inst(3, 0, 0)),
    (21, 4): (prod_inst(4, 1, 0), [prod_inst(4, 1, 1), prod_inst(4, 0, 1)], None),
    (23, 4): (None, [prod_inst(4, 1, 1), prod_inst(4, 0, 1)], prod_inst(4, 1, 0)),  # the slices themselves go wide
}


@pytest.mark.parametrize("n,k", list(PRODUCT_CASES))
def test_product_sumcheck_paths(ctx, n, k):
    round0, folds, slice0 = PRODUCT_CASES[(n, k)]
    mid = f"qz::sc_mid<{k}>"
    tabs = device_tables(ctx, n, k, 5000 + 10 * n + k)
    nodes, consts = util.expr_product(k)
    dev = None if round0 is None else dict(present=[round0, *folds, mid], counts={round0: 1})
    host = None if slice0 is None else dict(present=[slice0, *folds, mid], counts={slice0: 8})
    sumcheck_case(ctx, n, tabs, nodes, consts, b"paths_prod%d" % k, dev, host)


# ---- generic expressions -----------------------------------------------------------------------------------------------
GAMMA, LAMBDA, ALPHA = 0x1234567, 0x7654321, 0x2468ACE


def logup_terms():
    """the multiset check's zero-check expression over f, g, dl, dr = tables 0..3 (multiplicities 1):
    (dl (gamma + f) - 1) + lambda (dr (gamma + g) - 1)"""
    one = py.e_const(1)
    left = py.e_sub(py.e_mul(py.e_in(2), py.e_add(py.e_const(GAMMA), py.e_in(0))), one)
    right = py.e_sub(py.e_mul(py.e_in(3), py.e_add(py.e_const(GAMMA), py.e_in(1))), one)
    return py.e_add(left, py.e_mul(py.e_const(LAMBDA), right))


GENERIC_EXPRS = {
    # hyperplonk.py's multiset-check sumcheck: logup terms * eq (table 4) * alpha + dl - dr
    "logup_eq": py.e_sub(py.e_add(py.e_mul(py.e_mul(logup_terms(), py.e_in(4)), py.e_const(ALPHA)), py.e_in(2)),
                         py.e_in(3)),
    "constant": py.e_const(0x5EED),  # references no table: round 0 is sliced with nothing to copy
    "cancels": py.e_sub(py.e_mul(py.e_in(0), py.e_in(1)), py.e_mul(py.e_in(1), py.e_in(0))),  # every polynomial empty
    "unused_tables": py.e_add(py.e_mul(py.e_in(3), py.e_in(1)), py.e_in(1)),  # tables 0, 2 and 4 are not referenced
}


def logup_tables(ctx, n, seed):
    """f, g, dl, dr uniform below r and the eq table of a random point"""
    return device_tables(ctx, n, 4, seed) + [q.fast_eq_eval_hypercube(ctx, n, util.rand_fr(n, seed + 99))]


@pytest.mark.parametrize("n,name", [(21, "logup_eq"), (21, "constant"), (21, "cancels"), (21, "unused_tables"),
                                    (23, "logup_eq")])
def test_generic_sumcheck_paths(ctx, n, name):
    """the interpreted rounds fold through c_fold from 2^16 pairs on; host tables (2^21) run round 0 in 8 slices"""
    tabs = logup_tables(ctx, n, 6000 + n)
    nodes, consts = util.expr_from_py(GENERIC_EXPRS[name])
    dev = dict(present=[GEN0, GEN1, "qz::sc_mid<0>"], counts={GEN0: 1})
    host = dict(present=[GEN0, GEN1, "qz::sc_mid<0>"], counts={GEN0: 8}) if n == 21 else None
    sc = sumcheck_case(ctx, n, tabs, nodes, consts, b"paths_" + name.encode(), dev, host)
    if name == "cancels":
        assert all(p.shape[0] == 0 for p in sc.r_polys)


# ---- zero-checks -------------------------------------------------------------------------------------------------------
# (n, K): instances of the eq-factored rounds.  From num_vars = 21 on every folding round derives t_j(1) (skip-X=1)
ZC_CASES = {
    (21, 1): [zc_inst(1, 0, 0, 0), zc_inst(1, 0, 1, 1)],
    (21, 2): [zc_inst(2, 0, 0, 0), zc_inst(2, 0, 1, 1)],
    (21, 3): [zc_inst(3, 1, 0, 0), zc_inst(3, 1, 1, 1), zc_inst(3, 0, 1, 1)],
    (22, 3): [zc_inst(3, 1, 0, 0), zc_inst(3, 1, 1, 1), zc_inst(3, 0, 1, 1)],
}


@pytest.mark.parametrize("n,k,structured", [(21, 1, False), (21, 1, True), (21, 2, False), (21, 2, True),
                                            (21, 3, False), (22, 3, False)])
def test_zerocheck_product_paths(ctx, n, k, structured):
    """h = a product of K tables: device tables against the oracle, host tables against the device proof.
    structured: table 0 vanishes on the even entries and table 1 is constant, so s_j has trailing zeros to trim while
    t_j(1) is derived from the running claim"""
    tabs = device_tables(ctx, n, k, 7000 + 10 * n + k)
    if structured:
        tabs[0][::2] = 0
        if k > 1:
            tabs[1][:] = co.fr1(5)
    nodes, consts = util.expr_product(k)
    present = ZC_CASES[(n, k)] + ["qz::zc_materialize_eq", f"qz::sc_mid<{k + 1}>"]
    absent = [re.escape(zc_inst(k, w, 1, 0)) for w in (0, 1)]  # no folding round without the skip-X=1 derivation
    (sc, claim, o), names = launches(lambda: assert_same(ctx, n, tabs, nodes, consts, None, b"paths_zc%d" % k,
                                                         zerocheck=True, device_tables=True, threads=NCPU))
    expect(names, present, absent)
    got, names = launches(lambda: gpu_prove(ctx, n, tabs, nodes, consts, None, b"paths_zc%d" % k, zerocheck=True))
    assert_same_proof(got, (sc, claim, o["state"], o["z"]))
    expect(names, present, absent)


def test_generic_zerocheck_streams_eq(ctx):
    """a zero-check of an expression that is not a product: the eq table is built and streamed as one more table"""
    n = 21
    tabs = device_tables(ctx, n, 4, 7500)
    nodes, consts = util.expr_from_py(logup_terms())
    _, names = launches(lambda: assert_same(ctx, n, tabs, nodes, consts, None, b"paths_zcgen", zerocheck=True,
                                            device_tables=True, threads=NCPU))
    expect(names, [GEN0, GEN1, "qz::eq_expand", "qz::sc_mid<0>"], [ANY_ZC], {GEN0: 1})


# ---- measurement switches: same bytes, other kernels ---------------------------------------------------------------
def test_no_skip1_switch(ctx, monkeypatch):
    """QZ_ZC_NO_SKIP1=1 runs the folding rounds without the 1 / z_j derivation: the kernel the redo after a degenerate
    z launches"""
    n, k = 22, 3
    tabs, o = product_reference(ctx, True, n, k)
    nodes, consts = util.expr_product(k)
    monkeypatch.setenv("QZ_ZC_NO_SKIP1", "1")
    got, names = launches(lambda: gpu_prove(ctx, n, tabs, nodes, consts, None, b"paths_ref", zerocheck=True,
                                            device_tables=True))
    assert_matches_oracle(n, got, o, zerocheck=True)
    expect(names, [zc_inst(3, 1, 1, 0)], [r"qz::sc_round_zc<\d, \d, 1, 1>"])


@pytest.mark.parametrize("zerocheck,k", [(False, 3), (False, 4), (True, 3)], ids=["sumcheck3", "sumcheck4", "zerocheck3"])
def test_narrow_switch(ctx, monkeypatch, zerocheck, k):
    """QZ_SC_NARROW=1 forces the fully reduced sums where the deferred-reduction kernels would run"""
    n = 22
    tabs, o = product_reference(ctx, zerocheck, n, k)
    nodes, consts = util.expr_product(k)
    monkeypatch.setenv("QZ_SC_NARROW", "1")
    claimed = None if zerocheck else co.fr1(FALSE_CLAIM)
    got, names = launches(lambda: gpu_prove(ctx, n, tabs, nodes, consts, claimed, b"paths_ref", zerocheck=zerocheck,
                                            device_tables=True))
    assert_matches_oracle(n, got, o, zerocheck=zerocheck)
    expect(names, [zc_inst(k, 0, 1, 1) if zerocheck else prod_inst(k, 0, 1)], [WIDE])


# ---- contexts sharing a device ---------------------------------------------------------------------------------------
def test_two_contexts_on_one_device(ctx):
    """quill_b200.h promises independent contexts, but c_fold is one table per device.  Three contexts on one device,
    one thread each, a fixed three calls each: a k = 3 sumcheck at 2^22 (wide passes fold through c_fold), a generic
    sumcheck at 2^21 (sc_round_generic<1> folds through it), and the fold test hook with its own challenge.  Every
    result equals the oracle's bytes, computed beforehand."""
    calls = 3
    tabs_a, o_a = product_reference(ctx, False, 22, 3)
    nodes_a, consts_a = util.expr_product(3)
    tabs_b = logup_tables(ctx, 21, 7700)
    nodes_b, consts_b = util.expr_from_py(GENERIC_EXPRS["logup_eq"])
    o_b = oracle_prove(21, tabs_b, nodes_b, consts_b, co.fr1(FALSE_CLAIM), b"paths_ctx_b", threads=NCPU)
    a0, a1 = device_tables(ctx, 20, 2, 7800)
    r = util.rand_fr(1, 7900)[0]
    want_c = co.field_op(0, 0, a0, co.field_op(0, 2, co.field_op(0, 1, a1, a0), np.tile(r, (a0.shape[0], 1))))

    ctxs = [q.Context(0) for _ in range(3)]
    jobs = [
        lambda: gpu_prove(ctxs[0], 22, tabs_a, nodes_a, consts_a, co.fr1(FALSE_CLAIM), b"paths_ref", device_tables=True),
        lambda: gpu_prove(ctxs[1], 21, tabs_b, nodes_b, consts_b, co.fr1(FALSE_CLAIM), b"paths_ctx_b", device_tables=True),
        lambda: ctxs[2].fold(r, a0, a1),
    ]
    results = [[] for _ in jobs]
    errors = []
    start = threading.Barrier(len(jobs), timeout=120)

    def run(i):
        try:
            start.wait()
            for _ in range(calls):
                results[i].append(jobs[i]())
        except BaseException as e:  # reported by the main thread
            errors.append(e)

    threads = [threading.Thread(target=run, args=(i,)) for i in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for c in ctxs:
        c.close()
    assert not errors, errors
    assert [len(r) for r in results] == [calls] * len(jobs)
    for got in results[0]:
        assert_matches_oracle(22, got, o_a)
    for got in results[1]:
        assert_matches_oracle(21, got, o_b)
    for got in results[2]:
        assert np.array_equal(got, want_c)
