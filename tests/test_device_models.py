"""CPU models of the device-side reformulations, checked against the oracle (no GPU needed).

The CUDA path may compute a value by a different route than the reference as long as every byte is the same.  Each route
that is not a transcription of the reference is restated here in a few lines of Python -- the same recurrences the
kernels run -- and compared with `oracle/pyref.py` (the reference's formulation), so the identity each kernel relies on
is pinned independently of the GPU tests:
  * eq-factored zero-check rounds (csrc/sumcheck.cu sc_round_zc, sumcheck.cuh sc_round_close with zc_z)
  * blake3 compression with the state columns spread over four lanes (csrc/sumcheck.cuh b3_compress_quad)
  * the inverse by the binary extended Euclidean algorithm (csrc/ff.cuh fp_inv_serial)
  * the merge of partial bucket runs by a segmented scan with early exit (csrc/msm.cu msm_partials_finish)
  * the streamed MSM's point ranges (csrc/msm.cu msm_plan)
  * NTT passes as plain local transforms + one correction product per element (csrc/mlpcs.cu ntt_pass)
  * the K = 3 round polynomial from samples at X = 0, 1, -1, infinity with lazily added operands, X = 1 restored from the
    running claim (csrc/sumcheck.cu prod_core_toom3, csrc/sumcheck.cuh sc_expand_evals / sc_toom3_to_coeffs)
  * the MSM's optional pair levels: equal-key neighbours of the sorted list added in affine coordinates with the
    denominators inverted through a product tree, outputs placed by an exclusive scan (csrc/msm.cu msm_pair_*)
"""
import os
import random
import re

import pytest

from oracle import pyref as py

FR = py.FR
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "quill_zkvm_b200", "csrc")


# ---------------------------------------------------------------------------------------------------------------------
def zerocheck_eq_factored(num_vars, tables, tr):
    """ZeroCheckProof::prove for h = prod(tables) the way sc_round_zc + sc_round_close do it:
    s_j(X) = P_j * eq(X, z_j) * t_j(X),  t_j(X) = sum_p E_{j+1}[p] * prod_t g_t(X, p), weights folded by addition."""
    k = len(tables)
    z = [tr.draw_field_element() for _ in range(num_vars)]
    tr.append_usize(num_vars)
    tr.append_fr(0)
    gs = [list(t) for t in tables]
    weights = py.fast_eq_eval_hypercube(num_vars - 1, z[1:]) if num_vars else []  # E_1
    prefix = 1
    r_polys, point = [], []
    for j in range(num_vars):
        pairs = len(gs[0]) // 2
        assert len(weights) == pairs
        # evaluations of t_j at X = 0..k (the weight scales one factor), then Lagrange interpolation on nodes 0..k
        evals = []
        for x in range(k + 1):
            acc = 0
            for p in range(pairs):
                term = weights[p]
                for g in gs:
                    term = term * (g[2 * p] + x * (g[2 * p + 1] - g[2 * p])) % FR
                acc = (acc + term) % FR
            evals.append(acc)
        coeffs = [0] * (k + 1)
        for i, yi in enumerate(evals):  # Lagrange basis polynomials
            num, den = [1], 1
            for m in range(k + 1):
                if m != i:
                    num = py.poly_mul(num, [(-m) % FR, 1])
                    den = den * (i - m) % FR
            scale = yi * pow(den, FR - 2, FR) % FR
            num = num + [0] * (k + 1 - len(num))
            coeffs = [(c + scale * nc) % FR for c, nc in zip(coeffs, num)]
        a, b = prefix * (1 - z[j]) % FR, prefix * (2 * z[j] - 1) % FR  # P_j * eq(X, z_j) = a + b X
        s = [(a * (coeffs[t] if t <= k else 0) + b * (coeffs[t - 1] if t >= 1 else 0)) % FR for t in range(k + 2)]
        s = py.trim(s)
        tr.append_fr_vec(s)
        r_polys.append(s)
        r = tr.draw_field_element()
        point.append(r)
        prefix = prefix * ((r * z[j] + (1 - r) * (1 - z[j])) % FR) % FR
        gs = [[(g[2 * p] + r * (g[2 * p + 1] - g[2 * p])) % FR for p in range(pairs)] for g in gs]
        weights = [(weights[2 * p] + weights[2 * p + 1]) % FR for p in range(pairs // 2)]  # eq(0,z) + eq(1,z) = 1
    ev = 1
    for g in gs:
        ev = ev * g[0] % FR
    # the reference returns h_hat(point) / eq(z, point) = h(point); prefix == eq(z, point) ties the two together
    assert prefix == py.eq_eval(z, point)
    return r_polys, point, ev, z


@pytest.mark.parametrize("n,k", [(1, 1), (2, 2), (3, 3), (5, 1), (5, 2), (6, 3)])
def test_eq_factored_zerocheck_equals_reference_formulation(n, k):
    rnd = random.Random(100 * n + k)
    tables = [[rnd.randrange(FR) for _ in range(1 << n)] for _ in range(k)]
    if n == 5:
        tables[0][::2] = [0] * (1 << (n - 1))  # round polynomials with vanishing leading coefficients get trimmed
    h = py.e_in(0)
    for t in range(1, k):
        h = py.e_mul(h, py.e_in(t))
    t1, t2 = py.Transcript(b"zc_model"), py.Transcript(b"zc_model")
    want = py.zerocheck_prove(n, tables, h, t1)
    got = zerocheck_eq_factored(n, tables, t2)
    assert got[0] == [py.trim([c % FR for c in p]) for p in want[0]]
    assert got[1] == want[1] and got[2] == want[2] % FR and got[3] == want[3]
    assert t1.state == t2.state


# ---------------------------------------------------------------------------------------------------------------------
IV = [0x6A09E667, 0xBB67AE85, 0x3C6EF372, 0xA54FF53A, 0x510E527F, 0x9B05688C, 0x1F83D9AB, 0x5BE0CD19]
PERM = [2, 6, 3, 10, 7, 0, 4, 13, 1, 11, 12, 5, 9, 14, 15, 8]
M32 = 0xFFFFFFFF


def _ror(x, n):
    return ((x >> n) | (x << (32 - n))) & M32


def _g(a, b, c, d, mx, my):
    a = (a + b + mx) & M32
    d = _ror(d ^ a, 16)
    c = (c + d) & M32
    b = _ror(b ^ c, 12)
    a = (a + b + my) & M32
    d = _ror(d ^ a, 8)
    c = (c + d) & M32
    b = _ror(b ^ c, 7)
    return a, b, c, d


def _device_schedule():
    """the nibble-packed message schedule constants of b3_compress_quad, read from the header"""
    src = open(os.path.join(CSRC, "sumcheck.cuh")).read()
    body = re.search(r"B3_SCHED\[7\]\s*=\s*\{([^}]*)\}", src).group(1)
    words = [int(w.rstrip("ul"), 16) for w in re.findall(r"0x[0-9a-fA-F]+ull", body)]
    assert len(words) == 7
    return [[(w >> (4 * j)) & 15 for j in range(16)] for w in words]


def compress_quad(cv, m, block_len, flags, sched):
    """b3_compress_quad: lane i holds column i; shuffles rotate b, c, d into the diagonals and back"""
    a, b, c = list(cv[:4]), list(cv[4:]), IV[:4]
    d = [0, 0, block_len, flags]
    for r in range(7):
        for i in range(4):  # column step
            a[i], b[i], c[i], d[i] = _g(a[i], b[i], c[i], d[i], m[sched[r][2 * i]], m[sched[r][2 * i + 1]])
        b, c, d = [b[(i + 1) & 3] for i in range(4)], [c[(i + 2) & 3] for i in range(4)], [d[(i + 3) & 3] for i in range(4)]
        for i in range(4):  # diagonal step
            a[i], b[i], c[i], d[i] = _g(a[i], b[i], c[i], d[i], m[sched[r][8 + 2 * i]], m[sched[r][9 + 2 * i]])
        b, c, d = [b[(i + 3) & 3] for i in range(4)], [c[(i + 2) & 3] for i in range(4)], [d[(i + 1) & 3] for i in range(4)]
    out_lo = [a[i] ^ c[i] for i in range(4)] + [b[i] ^ d[i] for i in range(4)]
    out_hi = [c[i] ^ cv[i] for i in range(4)] + [d[i] ^ cv[4 + i] for i in range(4)]
    return out_lo, out_hi


def blake3_single_chunk_quad(data: bytes, out_len: int, sched) -> bytes:
    assert len(data) <= 1024 and out_len <= 64
    nblocks = max(1, (len(data) + 63) // 64)
    cv = list(IV)
    for blk in range(nblocks):
        chunk = data[64 * blk: 64 * blk + 64]
        m = [int.from_bytes(chunk[4 * i: 4 * i + 4].ljust(4, b"\0"), "little") for i in range(16)]
        last = blk + 1 == nblocks
        flags = (1 if blk == 0 else 0) | ((2 | 8) if last else 0)
        lo, hi = compress_quad(cv, m, len(chunk) if last else 64, flags, sched)
        cv = lo
    return b"".join(w.to_bytes(4, "little") for w in lo + hi)[:out_len]


def test_quad_lane_blake3_matches_blake3():
    blake3 = pytest.importorskip("blake3")
    sched = _device_schedule()
    ref = [list(range(16))]
    for _ in range(6):
        ref.append([ref[-1][PERM[j]] for j in range(16)])
    assert sched == ref  # the packed constants are the iterated message permutation
    rnd = random.Random(7)
    for n in (0, 1, 41, 63, 64, 65, 80, 168, 200, 1024):
        data = bytes(rnd.randrange(256) for _ in range(n))
        assert blake3_single_chunk_quad(data, 48, sched) == blake3.blake3(data).digest(length=48), n


# ---------------------------------------------------------------------------------------------------------------------
def inv_binary_euclid(a, p):
    """fp_inv_serial: invariants x1 * a = u and x2 * a = v (mod p)"""
    if a == 0:
        return 0
    u, v, x1, x2 = a, p, 1, 0
    while u != 1 and v != 1:
        while u & 1 == 0:
            u >>= 1
            x1 = (x1 + p) >> 1 if x1 & 1 else x1 >> 1
        while v & 1 == 0:
            v >>= 1
            x2 = (x2 + p) >> 1 if x2 & 1 else x2 >> 1
        if u >= v:
            u, x1 = u - v, (x1 - x2) % p
        else:
            v, x2 = v - u, (x2 - x1) % p
    return x1 if u == 1 else x2


@pytest.mark.parametrize("p", [FR, py.FQ])
def test_binary_euclid_inverse(p):
    rnd = random.Random(3)
    R = 1 << 256
    for a in [1, 2, 3, p - 1, p - 2, (p + 1) // 2, 1 << 128, (1 << 253) % p] + [rnd.randrange(1, p) for _ in range(200)]:
        assert inv_binary_euclid(a, p) == pow(a, p - 2, p)
        # Montgomery bookkeeping of the device routine: input aR, raw inverse (aR)^-1, one Montgomery product with R^3
        raw = inv_binary_euclid(a * R % p, p)
        assert raw * pow(R, 3, p) % p * pow(R, p - 2, p) % p == pow(a, p - 2, p) * R % p
    assert inv_binary_euclid(0, p) == 0


# ---------------------------------------------------------------------------------------------------------------------
def segmented_scan_finish(keys, vals):
    """msm_partials_finish with integers standing in for group elements: compact the non-empty slots, Hillis-Steele scan
    restricted to equal (ascending) keys, stop when a step adds nothing, the last slot of every run is the bucket"""
    ck = [k for k in keys if k is not None]
    cur = [v for k, v in zip(keys, vals) if k is not None]
    m, d, steps = len(ck), 1, 0
    while d < m or d == 1:
        nxt, added = list(cur), False
        for i in range(m):
            if i >= d and ck[i - d] == ck[i]:
                nxt[i] = cur[i] + cur[i - d]
                added = True
        cur, steps = nxt, steps + 1
        if not added:
            break
        d <<= 1
    return {ck[i]: cur[i] for i in range(m) if i + 1 == m or ck[i + 1] != ck[i]}, steps


def test_segmented_scan_merges_partial_runs():
    rnd = random.Random(11)
    for trial in range(200):
        n = rnd.randrange(0, 80)
        runs = sorted(rnd.randrange(1, 12) for _ in range(rnd.randrange(1, 10)))
        keys, vals = [], []
        while len(keys) < n:
            if rnd.random() < 0.3:
                keys.append(None), vals.append(0)
            else:
                keys.append(rnd.choice(runs)), vals.append(rnd.randrange(1000))
        it = iter(sorted(k for k in keys if k is not None))  # non-empty keys ascend; empty slots stay interleaved
        keys = [None if k is None else next(it) for k in keys]
        want = {}
        for k, v in zip(keys, vals):
            if k is not None:
                want[k] = want.get(k, 0) + v
        got, steps = segmented_scan_finish(keys, vals)
        assert got == want
        longest = max([sum(1 for k in keys if k == key) for key in want] + [1])
        assert steps <= max(1, (longest - 1).bit_length()) + 1  # early exit: log2(longest run) + 1 steps


# ---------------------------------------------------------------------------------------------------------------------
def segment_bounds(n, weights):
    """msm_plan: cumulative weights -> range ends rounded up to 256 points, empty ranges dropped, last end = n"""
    total, run, lo = sum(weights), 0.0, [0]
    for s, w in enumerate(weights):
        run += w
        hi = n if s == len(weights) - 1 else min(n, (int(n * run / total) + 255) & ~255)
        if hi > lo[-1]:
            lo.append(hi)
    return lo


def test_streamed_msm_ranges_partition_the_points():
    for n in (1, 2, 255, 256, 257, 1000, 70001, 1 << 19, (1 << 24) + 5):
        for weights in ([1], [1, 1], [1, 3, 9], [1] * 8, [1, 1000], [5, 0.001]):
            lo = segment_bounds(n, weights)
            assert lo[0] == 0 and lo[-1] == n and all(a < b for a, b in zip(lo, lo[1:])) and len(lo) - 1 <= len(weights)
            assert all(x % 256 == 0 for x in lo[1:-1])


# ---------------------------------------------------------------------------------------------------------------------
NTT_P = 12289  # 3 * 2^12 + 1: a small NTT-friendly prime stands in for Fr (the identity is about exponents of w)


def _ntt_root(order):
    w = pow(11, (NTT_P - 1) // order, NTT_P)
    assert pow(w, order, NTT_P) == 1 and pow(w, order // 2, NTT_P) != 1
    return w


def _brev(x, bits):
    return int(format(x, f"0{bits}b")[::-1], 2) if bits else 0


def ntt_dif_reference(a, log_m):
    """radix-2 decimation in frequency, natural -> bit-reversed, full twiddle w^((i mod half) << s) at stage s"""
    m, w, a = 1 << log_m, _ntt_root(1 << log_m), list(a)
    for s in range(log_m):
        half = m >> (s + 1)
        for i in range(m):
            if (i // half) % 2 == 0:
                u, v = a[i], a[i + half]
                a[i], a[i + half] = (u + v) % NTT_P, (u - v) * pow(w, (i % half) << s, NTT_P) % NTT_P
    return a


def ntt_pass_model(a, log_m, s0, T, inverse):
    """ntt_pass: stages [s0, s0 + T) on the sub-tiles (hi, lo); butterflies use only the twiddle part shared by all
    sub-tiles, and element t is corrected by w^(+-(lo * brev_T(t) << s0)) on the way out (forward) / in (inverse)"""
    m, w, a = 1 << log_m, _ntt_root(1 << log_m), list(a)
    lo_bits = log_m - s0 - T
    for hi in range(1 << s0):
        for lo in range(1 << lo_bits):
            idx = [(hi << (log_m - s0)) + lo + (t << lo_bits) for t in range(1 << T)]
            tile = [a[i] for i in idx]
            if inverse and lo:
                tile = [v * pow(w, (m - ((lo * _brev(t, T)) << s0)) % m, NTT_P) % NTT_P for t, v in enumerate(tile)]
            for ls in (range(T - 1, -1, -1) if inverse else range(T)):
                lhalf, s = 1 << (T - 1 - ls), s0 + ls
                for b in range(1 << (T - 1)):
                    j_l = b & (lhalf - 1)
                    i0 = ((b - j_l) << 1) + j_l
                    i1, e = i0 + lhalf, (j_l << lo_bits) << s
                    u, v = tile[i0], tile[i1]
                    if not inverse:
                        tile[i0], tile[i1] = (u + v) % NTT_P, (u - v) * pow(w, e, NTT_P) % NTT_P
                    else:
                        vw = v * pow(w, (m - e) % m, NTT_P) % NTT_P
                        tile[i0], tile[i1] = (u + vw) % NTT_P, (u - vw) % NTT_P
            if not inverse and lo:
                tile = [v * pow(w, (lo * _brev(t, T)) << s0, NTT_P) % NTT_P for t, v in enumerate(tile)]
            for t, i in enumerate(idx):
                a[i] = tile[t]
    return a


@pytest.mark.parametrize("log_m,groups", [(5, (5,)), (6, (3, 3)), (6, (2, 2, 2)), (7, (3, 2, 2)), (8, (3, 3, 2)), (10, (4, 3, 3))])
def test_ntt_passes_with_per_pass_correction(log_m, groups):
    rnd = random.Random(log_m)
    a = [rnd.randrange(NTT_P) for _ in range(1 << log_m)]
    got, s0 = list(a), 0
    for T in groups:
        got = ntt_pass_model(got, log_m, s0, T, False)
        s0 += T
    assert got == ntt_dif_reference(a, log_m)
    for T in reversed(groups):  # the inverse passes, last group first, undo it up to the factor m
        s0 -= T
        got = ntt_pass_model(got, log_m, s0, T, True)
    assert got == [x * (1 << log_m) % NTT_P for x in a]


def test_fixed_multiplier_bounds_and_value():
    """ff.cuh fp_mul_fixed: r * d = sum_i d_i * C_i with C_i = r * 2^(32 i + 32 q_i) mod p, rows 0..3, one Montgomery
    reduction row, rows 4..7, two more reduction rows.  The running value must stay below 2^288 (nine 32-bit columns)
    and end below 2p, for ANY 256-bit d (the kernels pass a1 - a0 + p unreduced) -- checked on the extremes."""
    import random
    p = FR
    inv = (-pow(p, -1, 1 << 32)) % (1 << 32)
    exps = [32 * i + (96 if i < 4 else 64) for i in range(8)]

    def mont_row(v):
        m = (v & 0xFFFFFFFF) * inv & 0xFFFFFFFF
        v += m * p
        assert v < 1 << 288 and v & 0xFFFFFFFF == 0
        return v >> 32

    def model(d, r):
        C = [r * pow(2, e, p) % p for e in exps]
        w = [(d >> (32 * i)) & 0xFFFFFFFF for i in range(8)]
        v = sum(w[i] * C[i] for i in range(4))
        v = mont_row(v)
        v += sum(w[i] * C[i] for i in range(4, 8))
        assert v < 1 << 288
        v = mont_row(mont_row(v))
        assert v < 2 * p
        return v - p if v >= p else v

    rnd = random.Random(5)
    ds = [0, 1, p - 1, 2 * p - 1, (1 << 256) - 1, (1 << 256) - (1 << 32), 0xFFFFFFFF] + [rnd.randrange(1 << 256) for _ in range(200)]
    rs = [0, 1, p - 1, p - 2, (1 << 253) % p] + [rnd.randrange(p) for _ in range(20)]
    for r in rs:
        for d in ds:
            assert model(d, r) == r * d % p


# ---------------------------------------------------------------------------------------------------------------------
def sumcheck_toom3_skip1(num_vars, tables, claimed, tr):
    """SumcheckProof::prove for h = g0 g1 g2 the way sc_round_prod<3, WIDE> + sc_finalize do it (csrc/sumcheck.cu
    prod_core_toom3, sumcheck.cuh sc_expand_evals / sc_toom3_to_coeffs): the cubic is sampled at X = 0, 1, -1 and
    infinity, with q(-1) = 2 q(0) + 2 q(inf) - q(1) of the quadratic g0 g1 and g2(-1) = 2 lo - hi formed as plain
    (unreduced) integers below 2^256; from round 1 on s(1) is not summed but restored from the running claim."""
    gs = [list(t) for t in tables]
    tr.append_usize(num_vars)
    tr.append_fr(claimed)
    r_polys, point, claim = [], [], None
    inv2 = pow(2, -1, FR)
    for j in range(num_vars):
        pairs = len(gs[0]) // 2
        s0 = s1 = sm = sinf = 0
        for p in range(pairs):
            lo = [g[2 * p] for g in gs]
            hi = [g[2 * p + 1] for g in gs]
            q0, q1 = lo[0] * lo[1] % FR, hi[0] * hi[1] % FR
            d0 = (hi[0] - lo[0]) % FR               # reduced: first operand of a reducing product
            d1 = hi[1] - lo[1] + FR                 # lazy, in (0, 2p)
            q2 = d0 * d1 % FR
            d2 = hi[2] - lo[2] + FR                 # lazy
            qm = 2 * (q0 + q2) + (FR - q1)          # plain integers: must stay below 2^256
            gm = lo[2] + (lo[2] - hi[2] + FR)
            assert 0 < d1 < 2 * FR and 0 < d2 < 2 * FR and 0 < qm < 5 * FR < (1 << 256) and 0 < gm < 3 * FR
            s0 += q0 * lo[2]                        # deferred reduction: the products are summed as integers
            s1 += q1 * hi[2]
            sinf += q2 * d2
            sm += qm * gm
        s0, s1, sm, sinf = s0 % FR, s1 % FR, sm % FR, sinf % FR
        if j > 0:                                    # SKIP1: s_j(1) = s_{j-1}(r_{j-1}) - s_j(0)
            assert s1 == (claim - s0) % FR
            s1 = (claim - s0) % FR
        c0, c3 = s0, sinf
        c2 = ((s1 + sm) * inv2 - c0) % FR
        c1 = ((s1 - sm) * inv2 - c3) % FR
        poly = py.trim([c0, c1, c2, c3])
        tr.append_fr_vec(poly)
        r = tr.draw_field_element()
        claim = sum(c * pow(r, i, FR) for i, c in enumerate([c0, c1, c2, c3])) % FR
        gs = [[(g[2 * p] + r * (g[2 * p + 1] - g[2 * p])) % FR for p in range(pairs)] for g in gs]
        r_polys.append(poly)
        point.append(r)
    return r_polys, point, gs[0][0] * gs[1][0] * gs[2][0] % FR


@pytest.mark.parametrize("n", [1, 4, 7])
def test_toom3_sampling_with_derived_s1_equals_reference_formulation(n):
    rnd = random.Random(300 + n)
    tables = [[rnd.randrange(FR) for _ in range(1 << n)] for _ in range(3)]
    tables[0][0] = tables[1][1] = 0
    tables[2][2 % (1 << n)] = FR - 1
    h = py.e_mul(py.e_mul(py.e_in(0), py.e_in(1)), py.e_in(2))
    for claimed in (sum(a * b * c for a, b, c in zip(*tables)) % FR, 12345):  # the true sum and a false claim
        tr_ref = py.Transcript(b"toom")
        want = py.sumcheck_prove(n, [list(t) for t in tables], h, claimed, tr_ref)
        tr = py.Transcript(b"toom")
        got = sumcheck_toom3_skip1(n, tables, claimed, tr)
        assert got == want and tr.state == tr_ref.state


# ---------------------------------------------------------------------------------------------------------------------
PAIR_B, PAIR_THREADS, PAIR_G, VAL_PAIR = 16, 128, 16, 1 << 30
PAIR_TILE = PAIR_B * PAIR_THREADS


def _batch_inverse_tree(v, p):
    """msm_pair_tree_up / _root / _down: invert every element through a product tree of fan-in PAIR_G climbed to ONE
    root (one modular inversion); `pre` holds the running product before each element"""
    levels, pres = [list(v)], []
    while len(levels[-1]) > 1:
        cur, pre, up = levels[-1], [0] * len(levels[-1]), []
        for u in range(0, len(cur), PAIR_G):
            run = 1
            for i in range(u, min(u + PAIR_G, len(cur))):
                pre[i] = run
                run = run * cur[i] % p
            up.append(run)
        pres.append(pre)
        levels.append(up)
    levels[-1] = [pow(levels[-1][0], p - 2, p)]
    for depth in reversed(range(len(pres))):
        cur, pre, up = levels[depth], pres[depth], levels[depth + 1]
        for u in range(len(up)):
            inv = up[u]
            for i in reversed(range(u * PAIR_G, min(u * PAIR_G + PAIR_G, len(cur)))):
                x = cur[i]
                cur[i] = inv * pre[i] % p
                inv = inv * x % p
    return levels[0]


def pair_level(keys, vals, dmask, bases, sums):
    """One pair level of csrc/msm.cu (msm_pair_scan, the inversion tree, msm_pair_apply) over Python ints: returns the
    output list; appends this level's pair sums to `sums`.  Points are (x, y) with (0, 0) = infinity, values carry the
    sign in bit 31 and VAL_PAIR when they address `sums`.  A block owns a tile of PAIR_TILE pairs, thread i the pairs
    i, i + 128, .. of it."""
    q = py.FQ
    m = len(keys)

    def point(val):
        x, y = (sums if val & VAL_PAIR else bases)[val & (VAL_PAIR - 1)]
        return (x, (-y) % q if val >> 31 else y)

    def entries(pair):  # keys and values of entries 2p, 2p + 1; 0 past the end of the list
        a = 2 * pair
        ka, va = (keys[a], vals[a]) if a < m else (0, 0)
        kb, vb = (keys[a + 1], vals[a + 1]) if a + 1 < m else (0, 0)
        return ka, kb, va, vb

    n_tiles = (m + 2 * PAIR_TILE - 1) // (2 * PAIR_TILE)
    pair_of = lambda tile, j, i: tile * PAIR_TILE + j * PAIR_THREADS + i  # noqa: E731
    codes, prefix, totals, counts = {}, {}, [], []
    for tile in range(n_tiles):  # scan
        n_out = n_sum = 0
        for i in range(PAIR_THREADS):
            run = 1
            for j in range(PAIR_B):
                pr = pair_of(tile, j, i)
                ka, kb, va, vb = entries(pr)
                code = (ka & dmask != 0) + (kb & dmask != 0)
                if ka == kb and ka & dmask:
                    xa, xb = point(va)[0], point(vb)[0]
                    d = (xb - xa) % q
                    if xa and xb and d:  # the chord rule applies; anything else passes through to the XYZZ law
                        code = 4 | 1
                        prefix[pr] = run
                        run = run * d % q
                codes[pr] = code
                n_out, n_sum = n_out + (code & 3), n_sum + (code >> 2)
            totals.append(run)
        counts.append((n_out, n_sum))
    offs = [(0, 0)]
    for c in counts:  # exclusive scan over the tiles, with the extra item that receives the totals
        offs.append((offs[-1][0] + c[0], offs[-1][1] + c[1]))
    inv_totals = _batch_inverse_tree(totals, q) if totals else []
    sum_base = len(sums)
    m_out, n_sums = offs[n_tiles]
    keys_out, vals_out = [None] * m_out, [None] * m_out
    sums.extend([None] * n_sums)
    for tile in range(n_tiles):  # apply
        off, run_out, run_sum = {}, 0, 0
        for j in range(PAIR_B):  # offsets inside the tile, in list order = (row, thread) order
            for i in range(PAIR_THREADS):
                off[(j, i)] = (run_out, run_sum)
                c = codes[pair_of(tile, j, i)]
                run_out, run_sum = run_out + (c & 3), run_sum + (c >> 2)
        for i in range(PAIR_THREADS):
            inv = inv_totals[tile * PAIR_THREADS + i]
            for j in reversed(range(PAIR_B)):
                pr = pair_of(tile, j, i)
                code = codes[pr]
                if not code & 3:
                    continue
                ka, kb, va, vb = entries(pr)
                pos = offs[tile][0] + off[(j, i)][0]
                if code & 4:
                    (xa, ya), (xb, yb) = point(va), point(vb)
                    dinv = inv * prefix[pr] % q
                    inv = inv * ((xb - xa) % q) % q
                    lam = (yb - ya) * dinv % q
                    x3 = (lam * lam - xa - xb) % q
                    sidx = sum_base + offs[tile][1] + off[(j, i)][1]
                    sums[sidx] = (x3, (lam * (xa - x3) - ya) % q)
                    keys_out[pos], vals_out[pos] = ka, VAL_PAIR | sidx
                else:
                    if ka & dmask:
                        keys_out[pos], vals_out[pos] = ka, va
                        pos += 1
                    if kb & dmask:
                        keys_out[pos], vals_out[pos] = kb, vb
            assert inv == 1
    assert None not in keys_out and None not in sums
    return keys_out, vals_out


def test_pair_levels_keep_every_bucket_sum():
    rnd = random.Random(5)
    c = 6
    dmask = (1 << c) - 1
    base_pts = [py.g1_mul(py.G1_GEN, k) for k in range(1, 40)]
    bases = [(0, 0)] + base_pts  # index 0: infinity in the SRS

    def as_opt(pt):
        return None if pt == (0, 0) else pt

    for trial in range(12):
        m = rnd.choice([1, 2, 31, 32, 33, 64, 65, 200, 333, 4095, 4097, 5000])
        n_keys = rnd.choice([1, 3, 20])
        entries = []
        for _ in range(m):
            key = (rnd.randrange(2) << c) | rnd.choice([0] + list(range(1, n_keys + 1)))
            if trial % 3 == 0:  # few distinct points: equal x (P + P and P - P) and infinite operands inside buckets
                idx = rnd.randrange(0, 3)
            else:
                idx = rnd.randrange(0, len(bases))
            entries.append((key, idx | (rnd.randrange(2) << 31)))
        entries.sort(key=lambda e: e[0])
        keys, vals = [e[0] for e in entries], [e[1] for e in entries]
        want = {}
        for k, v in zip(keys, vals):
            if k & dmask:
                pt = as_opt(bases[v & (VAL_PAIR - 1)])
                want[k] = py.g1_add(want.get(k), py.g1_neg(pt) if v >> 31 else pt)
        sums = []
        for level in range(4):
            before = len(keys)
            keys, vals = pair_level(keys, vals, dmask, bases, sums)
            assert keys == sorted(keys) and all(k & dmask for k in keys)
            assert len(sums) <= max(0, m - 1) and len(keys) <= before
            got = {}
            for k, v in zip(keys, vals):
                x, y = (sums if v & VAL_PAIR else bases)[v & (VAL_PAIR - 1)]
                pt = as_opt((x, (-y) % py.FQ if v >> 31 else y))
                got[k] = py.g1_add(got.get(k), pt)
            assert {k: v for k, v in got.items() if v is not None} == {k: v for k, v in want.items() if v is not None}
        assert all(py.g1_is_on_curve(s) for s in sums)
