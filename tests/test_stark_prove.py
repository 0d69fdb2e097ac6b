"""starky prove() with logUp lookups (starky/src/{prover.rs:40-484, lookup.rs, vanishing_poly.rs, verifier.rs}).

CPU (-m "not gpu"): the column-wise restatement of lookup_helper_columns (tests/emu/logup_oracle.cpp) satisfies the logUp
identities; the device's row evaluation (gl_logup.cuh, compiled for the host from tests/emu/logup_emu.cpp) equals it bit
for bit; a CPU twin of prove() built from oracle pieces is accepted by the restated verify_stark_proof below, which
rejects it after tampering; and prove()'s host logic, with the oracle standing in for the device calls, equals the twin.
GPU (-m gpu): the helper-column kernel, the quotient with auxiliary polynomials and prove() itself against the twin."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

P = 0xFFFFFFFF00000001
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ----------------------------------------------------------------------------- test STARKs
def _stark_mod():
    from plonky2_b200 import stark as S

    return S


class RangeCheckStark:
    """A range check through logUp. Column 0 is the table t (t(0) = 0, t' = t + 1, t(n-1) = public input 0), columns 1
    and 2 the two lookups' frequencies, columns 3 and 4 selector bits s, u (constrained to 0/1), then `num_looking`
    looking columns of lookup 1 and, with `second_lookup`, two of lookup 2, which shares the table. Looking column 1 of
    lookup 1 reads the NEXT row and is filtered by s; column 2 is 2 * a (a < n/2); column 3 is filtered by the product
    s * u; lookup 2's second column is filtered by u."""

    def __new__(cls, num_rows, degree, num_looking=5, second_lookup=True):
        S = _stark_mod()

        class _RangeCheck(S.Stark):
            PUBLIC_INPUTS = 1

            def __init__(self):
                self.num_rows, self.degree, self.num_looking, self.second_lookup = num_rows, degree, num_looking, second_lookup
                self.first = 5
                self.second = 5 + num_looking
                self.COLUMNS = self.second + (2 if second_lookup else 0)

            def constraint_degree(self):
                return self.degree

            def eval(self, vars, yc):
                t, tn, s, u = vars.local(0), vars.next(0), vars.local(3), vars.local(4)
                yc.constraint_first_row(t)
                yc.constraint_transition(tn - t - 1)
                yc.constraint_last_row(t - vars.public_input(0))
                yc.constraint(s * (s - 1))
                yc.constraint(u * (u - 1))

            def _looking(self):
                cols, filts = [], []
                for k in range(self.num_looking):
                    c = self.first + k
                    if k == 1:
                        cols.append(S.Column.single_next_row(c))
                        filts.append(S.Filter.new_simple(S.Column.single(3)))
                    elif k == 2:
                        cols.append(S.Column.linear_combination_with_constant([(c, 2)], 0))
                        filts.append(S.Filter())
                    elif k == 3:
                        cols.append(S.Column.single(c))
                        filts.append(S.Filter([(S.Column.single(3), S.Column.single(4))], []))
                    else:
                        cols.append(S.Column.single(c))
                        filts.append(S.Filter())
                return cols, filts

            def lookups(self):
                cols, filts = self._looking()
                lks = [S.Lookup(cols, S.Column.single(0), S.Column.single(1), filts)]
                if self.second_lookup:
                    lks.append(S.Lookup([S.Column.single(self.second), S.Column.single(self.second + 1)], S.Column.single(0),
                                        S.Column.single(2), [S.Filter(), S.Filter.new_simple(S.Column.single(4))]))
                return lks

            def generate_trace(self, seed=1):
                n = self.num_rows
                rng = np.random.default_rng(seed)
                tr = np.zeros((self.COLUMNS, n), dtype=np.uint64)
                tr[0] = np.arange(n, dtype=np.uint64)
                tr[3], tr[4] = rng.integers(0, 2, n), rng.integers(0, 2, n)
                for k in range(self.num_looking):
                    tr[self.first + k] = rng.integers(0, n // 2 if k == 2 else n, n)
                if self.second_lookup:
                    tr[self.second:self.second + 2] = rng.integers(0, n, (2, n))
                for lk, fcol in zip(self.lookups(), (1, 2)):
                    m = np.zeros(n, dtype=np.float64)
                    for col, f in zip(lk.columns, lk.filter_columns):
                        vals = np.array([col.eval_table(tr, r) for r in range(n)]) if n <= 4096 else _eval_fast(col, tr)
                        w = np.array([_filter_table(f, tr, r) for r in range(n)]) if n <= 4096 else _filter_fast(f, tr)
                        m += np.bincount(vals.astype(np.int64), weights=w.astype(np.float64), minlength=n)[:n]
                    tr[fcol] = m.astype(np.uint64)
                return tr

        return _RangeCheck()


def _filter_table(f, tr, r):
    """Filter::eval_table (lookup.rs:114-125) on a host trace."""
    return (sum(a.eval_table(tr, r) * b.eval_table(tr, r) for a, b in f.products)
            + sum(c.eval_table(tr, r) for c in f.constants)) % P


def _eval_fast(col, tr):  # small-valued columns only (the range-check traces): exact in int64
    v = np.full(tr.shape[1], col.constant, dtype=np.int64)
    for c, f in col.linear_combination:
        v += tr[c].astype(np.int64) * f
    for c, f in col.next_row_linear_combination:
        v += np.roll(tr[c], -1).astype(np.int64) * f
    return v


def _filter_fast(f, tr):
    v = np.zeros(tr.shape[1], dtype=np.int64)
    for a, b in f.products:
        v += _eval_fast(a, tr) * _eval_fast(b, tr)
    for c in f.constants:
        v += _eval_fast(c, tr)
    return v


def fast_config(rate_bits=1):
    """standard_fast_config, with rate_bits 2 where the test asks for it."""
    S = _stark_mod()
    cfg = S.StarkConfig.standard_fast_config()
    if rate_bits != cfg.fri_config.rate_bits:
        from plonky2_b200.fri import FriConfig

        f = cfg.fri_config
        cfg = S.StarkConfig(cfg.security_bits, cfg.num_challenges,
                            FriConfig(rate_bits, f.cap_height, f.proof_of_work_bits, f.reduction_strategy, f.num_query_rounds))
    return cfg


def case(name, num_rows=None):
    """(stark, config, trace, public inputs) of the test STARKs (a) permutation, (b) range check of degree 3,
    (c) range check of degree 2 at rate_bits 2, (d) Fibonacci."""
    S = _stark_mod()
    if name == "permutation":
        st = S.PermutationStark(num_rows or 1 << 5)
        return st, fast_config(), st.generate_trace(0), [0]
    if name == "range3":
        st = RangeCheckStark(num_rows or 1 << 7, 3)
        return st, fast_config(), st.generate_trace(3), [st.num_rows - 1]
    if name == "range2":
        st = RangeCheckStark(num_rows or 1 << 7, 2)
        return st, fast_config(2), st.generate_trace(4), [st.num_rows - 1]
    if name == "fibonacci":
        st = S.FibonacciStark(num_rows or 1 << 6)
        tr = st.generate_trace(0, 1)
        return st, fast_config(), tr, [0, 1, int(tr[1, -1])]
    raise KeyError(name)


LOOKUP_CASES = ["permutation", "range3", "range2"]
ALL_CASES = LOOKUP_CASES + ["fibonacci"]


# ----------------------------------------------------------------------------- host builds of the helper-column sources
@pytest.fixture(scope="module")
def logup_libs(tmp_path_factory):
    d = tmp_path_factory.mktemp("logup")
    libs = {}
    for name, flags in (("logup_emu", ["-DGL_FORCE_32BIT_PATH"]), ("logup_oracle", [])):
        out = str(d / ("lib%s.so" % name))
        subprocess.check_call(["g++", "-O2", "-std=c++17"] + flags + ["-shared", "-fPIC", "-o", out,
                                                                      os.path.join(ROOT, "tests", "emu", name + ".cpp")])
        libs[name] = C.CDLL(out)
    return libs


_ORACLE_LIB = {}


def _oracle_lib():
    """The column-wise restatement, built once per process (also used by the timing tool)."""
    if "lib" not in _ORACLE_LIB:
        import tempfile

        d = tempfile.mkdtemp(prefix="logup_oracle_")
        out = os.path.join(d, "liblogup_oracle.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out,
                               os.path.join(ROOT, "tests", "emu", "logup_oracle.cpp")])
        _ORACLE_LIB["lib"] = C.CDLL(out)
    return _ORACLE_LIB["lib"]


def _run_helper(fn, stark, trace, challenges):
    S = _stark_mod()
    trace = np.ascontiguousarray(trace, dtype=np.uint64)
    ncols, n = trace.shape
    out = np.zeros((max(1, stark.num_lookup_helper_columns(None, len(challenges))), n), dtype=np.uint64)
    desc, keep = S.logup_descriptor(stark.lookups())
    ch = np.array([int(c) % P for c in challenges] + [0], dtype=np.uint64)
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    rc = fn(trace.ctypes.data, n, n.bit_length() - 1, C.addressof(desc), ch.ctypes.data, len(challenges),
            stark.constraint_degree(), out.ctypes.data)
    if rc == 1:
        raise ZeroDivisionError("Tried to invert zero")
    assert rc == 0
    return out[:stark.num_lookup_helper_columns(None, len(challenges))]


def oracle_helper_columns(stark, trace, challenges):
    return _run_helper(_oracle_lib().oracle_logup_helper_columns, stark, trace, challenges)


# ----------------------------------------------------------------------------- the CPU twin of prove()
def observe_config(ch, config):
    """StarkConfig::observe (config.rs:102-108) with FriConfig::observe (fri/mod.rs:73-79)."""
    f = config.fri_config
    ch.observe_elements([config.security_bits, config.num_challenges, f.rate_bits, f.cap_height, f.proof_of_work_bits])
    assert f.reduction_strategy[0] == "ConstantArityBits"
    ch.observe_elements([1, f.reduction_strategy[1], f.reduction_strategy[2], f.num_query_rounds])


def dummy_openings(ch, num_columns, num_aux, constraint_degree):
    """get_dummy_polys (get_challenges.rs:205-255) on the oracle's challenger."""
    from plonky2_b200 import field as F
    from plonky2_b200.proof import StarkOpeningSet

    total = 2 * num_columns + 2 * num_aux
    pow_degree = max(2, constraint_degree + 1)
    log_pow = int(np.ceil(np.log2(pow_degree)))
    nep = max(1, 50 // log_pow - 1)
    evals = []
    for _ in range(-(-total // nep)):
        z = ch.get_extension_challenge()
        for _ in range(min(nep + 1, total)):
            evals.append(z)
            z = F.ext_pow(z, pow_degree)
    a = np.array(evals, dtype=np.uint64).reshape(-1, 2)
    c0, c1 = 2 * num_columns, 2 * num_columns + num_aux
    return StarkOpeningSet(a[:num_columns], a[num_columns:c0], a[c0:c1] if num_aux else None, a[c1:] if num_aux else None)


def host_quotient(stark, trace_c, aux_c, public_inputs, alphas, lookup_challenges):
    """compute_quotient_polys (prover.rs:488-668) on the host: the constraint program at every point of the quotient coset,
    read from the oracle commitments' LDE rows, divided by Z_H, then oracle.coset_ifft. -> (num_alphas, size) coeffs."""
    import oracle_lib as oracle
    from plonky2_b200 import field as F

    S = _stark_mod()
    qdf = stark.quotient_degree_factor()
    qd_bits = (qdf - 1).bit_length()
    db, rb = trace_c.log_n, trace_c.rate_bits
    n, size = 1 << db, (1 << db) << qd_bits
    step, log_N = 1 << (rb - qd_bits), db + rb
    lc = list(lookup_challenges) if lookup_challenges is not None else []
    b = stark.constraint_program(len(lc))
    consts = b.bind(public_inputs, lc)
    rows = np.array([F.reverse_bits(i * step, log_N) for i in range(size)])
    nxt = np.array([F.reverse_bits(((i + (1 << qd_bits)) % size) * step, log_N) for i in range(size)])
    tl = trace_c.leaves[:, :trace_c.B]
    al = aux_c.leaves[:, :aux_c.B] if aux_c is not None else None
    w = F.primitive_root_of_unity(db + qd_bits)
    g = F.coset_shift()
    out = np.zeros((len(alphas), size), dtype=np.uint64)
    for i in range(size):
        x = g * pow(w, i, P) % P
        L = tl[rows[i]], tl[nxt[i]]
        A = (al[rows[i]], al[nxt[i]]) if al is not None else (None, None)
        ext = [(int(v), 0) for v in L[0]], [(int(v), 0) for v in L[1]]
        aux = ([(int(v), 0) for v in A[0]], [(int(v), 0) for v in A[1]]) if al is not None else (None, None)
        acc = S.eval_program_ext(b, consts, ext[0], ext[1], aux[0], aux[1], alphas, (x, 0), db)
        zh_inv = pow((pow(x, n, P) - 1) % P, P - 2, P)
        for a in range(len(alphas)):
            assert acc[a][1] == 0
            out[a, i] = acc[a][0] * zh_inv % P
    return np.stack([oracle.coset_ifft(out[a], g) for a in range(len(alphas))])


def _ev(oracle, commit, z):
    return np.array([oracle.eval_poly_base_at_ext(p, z) for p in commit.coeffs], dtype=np.uint64).reshape(-1, 2)


def twin_prove(oracle, stark, config, trace, public_inputs):
    """prove (prover.rs:40-484) from the oracle's pieces and the product's host evaluator of the constraints. Returns the
    proof's parts (what the verifier reads) plus the intermediate values the GPU tests compare."""
    from plonky2_b200 import field as F
    from plonky2_b200.proof import StarkOpeningSet

    S = _stark_mod()
    trace = np.ascontiguousarray(trace, dtype=np.uint64)
    n = trace.shape[1]
    db = n.bit_length() - 1
    f = config.fri_config
    nc = config.num_challenges
    fri_params = config.fri_params(db)
    trace_c = oracle.Commit(trace, f.rate_bits, f.cap_height)
    ch = oracle.Challenger()
    ch.observe_elements(public_inputs)
    observe_config(ch, config)
    ch.observe_cap(trace_c.cap)
    lc, aux_c, helpers = None, None, None
    if stark.uses_lookups():
        lc = [ch.get_n_challenges(2)[0] for _ in range(nc)]
        helpers = oracle_helper_columns(stark, trace, lc)
        aux_c = oracle.Commit(helpers, f.rate_bits, f.cap_height)
        ch.observe_cap(aux_c.cap)
    alphas_prime = ch.get_n_challenges(nc)
    dummy = dummy_openings(ch, stark.COLUMNS, aux_c.B if aux_c else 0, stark.constraint_degree())
    zeta_prime = ch.get_extension_challenge()
    constraints = S.compute_eval_vanishing_poly(stark, dummy, lc, public_inputs, alphas_prime, zeta_prime, db)
    ch.observe_elements(np.array(constraints, dtype=np.uint64).reshape(-1))
    alphas = ch.get_n_challenges(nc)
    qdf = stark.quotient_degree_factor()
    q_c, q, chunks = None, None, None
    if qdf:
        q = host_quotient(stark, trace_c, aux_c, public_inputs, alphas, lc)
        assert not q[:, qdf * n:].any(), "Quotient has failed, the vanishing polynomial is not divisible by Z_H"
        chunks = np.concatenate([q[i, :qdf * n].reshape(qdf, n) for i in range(nc)])
        q_c = oracle.Commit(chunks, f.rate_bits, f.cap_height, is_coeffs=True)
        ch.observe_cap(q_c.cap)
    zeta = ch.get_extension_challenge()
    assert F.ext_pow(zeta, n) != (1, 0)
    g = F.primitive_root_of_unity(db)
    gz = F.ext_mul((g, 0), zeta)
    openings = StarkOpeningSet(_ev(oracle, trace_c, zeta), _ev(oracle, trace_c, gz),
                               _ev(oracle, aux_c, zeta) if aux_c else None, _ev(oracle, aux_c, gz) if aux_c else None,
                               _ev(oracle, q_c, zeta) if q_c else None)
    for batch in openings.to_fri_openings():
        ch.observe_elements(batch.reshape(-1))
    inst = stark.fri_instance(zeta, g, config)
    batches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in inst.batches]
    commits = [c for c in (trace_c, aux_c, q_c) if c is not None]
    params = oracle.make_params(f.rate_bits, f.cap_height, f.proof_of_work_bits, f.num_query_rounds,
                                fri_params.reduction_arity_bits)
    fri_bytes = oracle.prove_openings(commits, batches, ch, params)
    return dict(trace_cap=trace_c.cap, auxiliary_polys_cap=aux_c.cap if aux_c else None,
                quotient_polys_cap=q_c.cap if q_c else None, openings=openings, fri_bytes=fri_bytes,
                public_inputs=[int(x) % P for x in public_inputs], helpers=helpers, lookup_challenges=lc, alphas=alphas,
                quotient=q, chunks=chunks, commits=commits)


def verify_stark_proof(oracle, stark, config, parts):
    """verify_stark_proof (verifier.rs:30-330) without CTLs: the shape rules, the transcript replayed with the
    constraint-binding step (get_challenges.rs:30-190), the vanishing polynomial with lookup terms at zeta in F_{p^2}
    against Z_H(zeta) * sum_k zeta^{nk} chunk_k(zeta), then verify_fri_proof. Returns None or the reason it rejects."""
    from plonky2_b200 import field as F

    S = _stark_mod()
    f = config.fri_config
    nc = config.num_challenges
    o = parts["openings"]
    pis = parts["public_inputs"]
    # validate_proof_shape / check_lookup_options (verifier.rs:254-330)
    ncap = 1 << f.cap_height
    if len(pis) != stark.PUBLIC_INPUTS:
        return "public inputs"
    if np.asarray(parts["trace_cap"]).shape != (ncap, 4):
        return "trace cap height"
    if parts["quotient_polys_cap"] is not None and np.asarray(parts["quotient_polys_cap"]).shape != (ncap, 4):
        return "quotient cap height"
    if len(o.local_values) != stark.COLUMNS or len(o.next_values) != stark.COLUMNS:
        return "trace openings"
    nq = stark.num_quotient_polys(config)
    if (o.quotient_polys is None and nq) or (o.quotient_polys is not None and len(o.quotient_polys) != nq):
        return "quotient openings"
    if stark.uses_lookups():
        na = stark.num_lookup_helper_columns(config)
        if parts["auxiliary_polys_cap"] is None or o.auxiliary_polys is None or o.auxiliary_polys_next is None:
            return "missing auxiliary polynomials"
        if np.asarray(parts["auxiliary_polys_cap"]).shape != (ncap, 4):
            return "auxiliary cap height"
        if len(o.auxiliary_polys) != na or len(o.auxiliary_polys_next) != na:
            return "auxiliary openings"
    elif parts["auxiliary_polys_cap"] is not None or o.auxiliary_polys is not None or o.auxiliary_polys_next is not None:
        return "unexpected auxiliary polynomials"
    if parts["quotient_polys_cap"] is None and nq:
        return "missing quotient cap"
    db = parts["degree_bits"]   # recover_degree_bits reads it from the FRI proof; the test knows it from the trace
    n_rows = 1 << db
    ch = oracle.Challenger()
    ch.observe_elements(pis)
    observe_config(ch, config)
    ch.observe_cap(parts["trace_cap"])
    lc = None
    if parts["auxiliary_polys_cap"] is not None:
        lc = [ch.get_n_challenges(2)[0] for _ in range(nc)]
        ch.observe_cap(parts["auxiliary_polys_cap"])
    if not stark.uses_lookups():
        lc = None
    alphas_prime = ch.get_n_challenges(nc)
    dummy = dummy_openings(ch, stark.COLUMNS, len(o.auxiliary_polys) if o.auxiliary_polys is not None else 0,
                           stark.constraint_degree())
    zeta_prime = ch.get_extension_challenge()
    constraints = S.compute_eval_vanishing_poly(stark, dummy, lc, pis, alphas_prime, zeta_prime, db)
    ch.observe_elements(np.array(constraints, dtype=np.uint64).reshape(-1))
    alphas = ch.get_n_challenges(nc)
    if parts["quotient_polys_cap"] is not None:
        ch.observe_cap(parts["quotient_polys_cap"])
    zeta = ch.get_extension_challenge()
    for batch in o.to_fri_openings():
        ch.observe_elements(batch.reshape(-1))
    vanishing = S.compute_eval_vanishing_poly(stark, o, lc, pis, alphas, zeta, db)
    zeta_n = F.ext_pow(zeta, n_rows)
    z_h = F.ext_sub(zeta_n, (1, 0))
    qdf = stark.quotient_degree_factor()
    if o.quotient_polys is not None:
        for i in range(len(o.quotient_polys) // qdf):
            red = (0, 0)
            for v in reversed(o.quotient_polys[i * qdf:(i + 1) * qdf]):     # reduce_with_powers(chunk, zeta^n)
                red = F.ext_add(F.ext_mul(red, zeta_n), (int(v[0]), int(v[1])))
            if vanishing[i] != F.ext_mul(z_h, red):
                return "Mismatch between evaluation and opening of quotient polynomial"
    g = F.primitive_root_of_unity(db)
    inst = stark.fri_instance(zeta, g, config)
    batches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in inst.batches]
    caps = [c for c in (parts["trace_cap"], parts["auxiliary_polys_cap"], parts["quotient_polys_cap"]) if c is not None]
    num_polys = [oi.num_polys for oi in inst.oracles]
    params = oracle.make_params(f.rate_bits, f.cap_height, f.proof_of_work_bits, f.num_query_rounds,
                                config.fri_params(db).reduction_arity_bits)
    opened = np.concatenate([b.reshape(-1) for b in o.to_fri_openings()])
    rc = oracle.verify_fri_proof(caps, num_polys, num_polys, batches, opened, db, ch, params, parts["fri_bytes"])
    return None if rc == 0 else "FRI proof rejected (rc=%d)" % rc


def _twin(oracle, name, num_rows=None):
    st, cfg, tr, pis = case(name, num_rows)
    parts = twin_prove(oracle, st, cfg, tr, pis)
    parts["degree_bits"] = tr.shape[1].bit_length() - 1
    return st, cfg, tr, pis, parts


# ============================================================================= CPU tests
@pytest.mark.parametrize("name", LOOKUP_CASES)
def test_oracle_helper_columns_satisfy_the_logup_identities(name):
    """h_k * prod(f + gamma) = the filtered sum for each row and chunk; Z(0) = 0; the wrap-around Z step closes exactly
    when the multiset matches, and fails to close with a frequency off by one or a looking value outside the table."""
    from plonky2_b200 import field as F

    st, cfg, tr, _ = case(name)
    n = tr.shape[1]
    gammas = [0x1234567, P - 0x89ABCDE]
    out = oracle_helper_columns(st, tr, gammas)
    cs = max(1, st.constraint_degree() - 1)

    def closes(trace, h):
        col = 0
        res = []
        for lk in st.lookups():
            nh = lk.num_helper_columns(st.constraint_degree())
            for g in gammas:
                z = h[col + nh - 1]
                assert z[0] == 0
                last = sum(int(h[col + k, n - 1]) for k in range(nh - 1)) - lk.frequencies_column.eval_table(trace, n - 1) * \
                    F.inverse(lk.table_column.eval_table(trace, n - 1) + g)
                res.append((int(z[n - 1]) + last) % P == 0)
                col += nh
        return res

    col = 0
    for lk in st.lookups():
        nh = lk.num_helper_columns(st.constraint_degree())
        for g in gammas:
            for r in (0, 1, n // 2, n - 1):
                for k in range(nh - 1):
                    idx = range(k * cs, min((k + 1) * cs, len(lk.columns)))
                    dens = [(lk.columns[i].eval_table(tr, r) + g) % P for i in idx]
                    prod = 1
                    for d in dens:
                        prod = prod * d % P
                    want = sum(_filter_table(lk.filter_columns[i], tr, r) * prod * F.inverse(d) for i, d in zip(idx, dens)) % P
                    assert int(out[col + k, r]) * prod % P == want
            col += nh
    assert all(closes(tr, out))
    bad = tr.copy()
    fcol = 2 if name == "permutation" else 1
    bad[fcol, 3] = (int(bad[fcol, 3]) + 1) % P                    # one frequency off by one
    assert not all(closes(bad, oracle_helper_columns(st, bad, gammas)))
    bad = tr.copy()
    bad[st.first if name != "permutation" else 0, 5] = n + 7     # a looking value outside the table
    assert not all(closes(bad, oracle_helper_columns(st, bad, gammas)))
    with pytest.raises(ZeroDivisionError, match="Tried to invert zero"):
        col0 = st.lookups()[0].columns[0].eval_table(tr, 0)
        oracle_helper_columns(st, tr, [(P - col0) % P])


@pytest.mark.parametrize("name", LOOKUP_CASES)
def test_logup_row_source_on_host_matches_the_column_wise_oracle(logup_libs, name):
    """gl_logup.cuh compiled for the host (one loop iteration per device thread, the scan as a loop) equals the
    column-wise restatement bit for bit."""
    st, cfg, tr, _ = case(name)
    gammas = [0xDEADBEEF, 0x7777777777, 12345]
    want = _run_helper(logup_libs["logup_oracle"].oracle_logup_helper_columns, st, tr, gammas)
    got = _run_helper(logup_libs["logup_emu"].emu_logup_helper_columns, st, tr, gammas)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("name", ALL_CASES)
def test_cpu_twin_proof_is_accepted_and_tampering_is_rejected(oracle, name):
    """The CPU twin's proof passes the restated verifier; it fails after changing one opened value, a cap, a public
    input, or one byte of the FRI proof."""
    st, cfg, tr, pis, parts = _twin(oracle, name)
    assert verify_stark_proof(oracle, st, cfg, parts) is None
    from plonky2_b200.proof import StarkOpeningSet

    o = parts["openings"]
    lv = o.local_values.copy()
    lv[0, 0] ^= np.uint64(1)
    bad = dict(parts, openings=StarkOpeningSet(lv, o.next_values, o.auxiliary_polys, o.auxiliary_polys_next, o.quotient_polys))
    assert verify_stark_proof(oracle, st, cfg, bad) is not None
    cap = np.array(parts["trace_cap"]).copy()
    cap[0, 0] ^= np.uint64(1)
    assert verify_stark_proof(oracle, st, cfg, dict(parts, trace_cap=cap)) is not None
    assert verify_stark_proof(oracle, st, cfg, dict(parts, public_inputs=[(pis[0] + 1) % P] + list(pis[1:]))) is not None
    fb = bytearray(parts["fri_bytes"])
    fb[len(fb) // 2] ^= 1
    assert verify_stark_proof(oracle, st, cfg, dict(parts, fri_bytes=bytes(fb))) is not None
    if parts["auxiliary_polys_cap"] is not None:
        cap = np.array(parts["auxiliary_polys_cap"]).copy()
        cap[1, 2] ^= np.uint64(1)
        assert verify_stark_proof(oracle, st, cfg, dict(parts, auxiliary_polys_cap=cap)) is not None


def test_constraint_programs_fit_and_overflow_is_a_shape_error():
    """The test STARKs' programs fit in GL_STARK_MAX_INSTR instructions; a larger one raises ShapeError."""
    from plonky2_b200 import ShapeError

    for name in ALL_CASES:
        st, cfg, _, _ = case(name)
        b = st.constraint_program(cfg.num_challenges if st.uses_lookups() else 0)
        assert 0 < len(b.instrs) <= 256
        b.program()
    big = RangeCheckStark(1 << 7, 3, num_looking=30)
    with pytest.raises(ShapeError):
        big.constraint_program(2).program()


@pytest.mark.parametrize("name", ALL_CASES)
def test_prove_host_logic_with_cpu_backends(oracle, name, monkeypatch):
    """The HOST side of stark.prove -- shape checks, transcript order, lookup challenges, the simulated opening set and
    the binding step, oracle order, FRI instance -- with the oracle standing in for the device calls (commitments, helper
    columns, quotient, evaluations, prove_openings): every field equals the twin's."""
    import plonky2_b200.challenger as challenger_mod
    import plonky2_b200.fri as fri_mod
    import plonky2_b200.proof as proof_mod

    S = _stark_mod()
    st, cfg, tr, pis, parts = _twin(oracle, name)
    f = cfg.fri_config

    class Cap:
        def __init__(self, hashes):
            self.hashes = hashes

    class Tree:
        def __init__(self, commit):
            self.cap = Cap(commit.cap)

    class Batch:
        def __init__(self, commit):
            self.o, self.merkle_tree, self.num_polys, self.degree_log = commit, Tree(commit), commit.B, commit.log_n

        def close(self):
            pass

    class Ctx:
        device, h = 0, None

    def quotient(stark, trace_c, pis_, alphas, aux=None, lookup_challenges=None):
        return host_quotient(stark, trace_c.o, aux.o if aux is not None else None, pis_, alphas, lookup_challenges)

    def commit_quotient(stark, q, degree_bits, rate_bits, cap_height, ctx=None):
        qdf, n = stark.quotient_degree_factor(), 1 << degree_bits
        chunks = np.concatenate([q[i, :qdf * n].reshape(qdf, n) for i in range(q.shape[0])])
        return Batch(oracle.Commit(chunks, rate_bits, cap_height, is_coeffs=True))

    def evals(requests):
        return [_ev(oracle, b.o, z) for b, z in requests]

    class FriBytes:
        def __init__(self, b):
            self.b = b

        def to_bytes(self):
            return self.b

    class LoggingChallenger(challenger_mod.Challenger):
        def __init__(self):
            super().__init__()
            self.log = []

        def observe_element(self, element):
            self.log.append(("observe", int(element)))
            super().observe_element(element)

        def get_challenge(self):
            v = super().get_challenge()
            self.log.append(("challenge", v))
            return v

    def prove_openings(instance, oracles, challenger, fri_params):
        och = oracle.Challenger()
        for kind, v in challenger.log:
            if kind == "observe":
                och.observe_element(v)
            else:
                assert och.get_challenge() == v
        batches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in instance.batches]
        assert [o.num_polys for o in instance.oracles] == [b.num_polys for b in oracles]
        params = oracle.make_params(f.rate_bits, f.cap_height, f.proof_of_work_bits, f.num_query_rounds,
                                    fri_params.reduction_arity_bits)
        return FriBytes(oracle.prove_openings([b.o for b in oracles], batches, och, params))

    monkeypatch.setattr(challenger_mod, "Challenger", LoggingChallenger)
    monkeypatch.setattr(S, "_to_device", lambda columns, ctx: np.ascontiguousarray(columns, dtype=np.uint64))
    monkeypatch.setattr(S, "_commit_values", lambda v, rate_bits, cap_height, ctx: Batch(oracle.Commit(v, rate_bits, cap_height)))
    monkeypatch.setattr(S, "lookup_helper_columns", lambda stark, t, lc, ctx=None: oracle_helper_columns(stark, t, lc))
    monkeypatch.setattr(S, "compute_quotient_polys", quotient)
    monkeypatch.setattr(S, "commit_quotient_polys", commit_quotient)
    monkeypatch.setattr(proof_mod, "eval_commitments", evals)
    monkeypatch.setattr(fri_mod, "prove_openings", prove_openings)
    proof = S.prove(st, cfg, tr, pis, ctx=Ctx())
    _assert_same_proof(proof, parts)


def _assert_same_proof(proof, parts):
    p = proof.proof
    assert proof.public_inputs == parts["public_inputs"]
    assert np.array_equal(p.trace_cap.hashes, parts["trace_cap"])
    for mine, key in ((p.auxiliary_polys_cap, "auxiliary_polys_cap"), (p.quotient_polys_cap, "quotient_polys_cap")):
        assert (mine is None) == (parts[key] is None)
        if mine is not None:
            assert np.array_equal(mine.hashes, parts[key])
    for fld in ("local_values", "next_values", "auxiliary_polys", "auxiliary_polys_next", "quotient_polys"):
        a, b = getattr(p.openings, fld), getattr(parts["openings"], fld)
        assert (a is None) == (b is None), fld
        if a is not None:
            assert np.array_equal(np.asarray(a, dtype=np.uint64), b), fld
    assert p.opening_proof.to_bytes() == parts["fri_bytes"]


def test_prove_rejects_bad_shapes():
    """prove's shape asserts (prover.rs:55-59,153-156) and the trace shape raise ShapeError before any device work."""
    from plonky2_b200 import ShapeError

    S = _stark_mod()
    st, cfg, tr, pis = case("range3")
    with pytest.raises(ShapeError):
        S.prove(st, cfg, tr[:-1], pis)
    with pytest.raises(ShapeError):
        S.prove(st, cfg, tr, pis + [1])
    hi = RangeCheckStark(1 << 7, 4)                             # degree 4 > 2^rate_bits + 1 = 3
    with pytest.raises(ShapeError, match="blowup_factor"):
        S.prove(hi, cfg, tr, pis)


# ============================================================================= GPU tests
@pytest.fixture(scope="module")
def pb():
    import torch

    if not torch.cuda.is_available():
        if os.environ.get("GL_REQUIRE_GPU") == "1":
            raise AssertionError("GPU tests need a CUDA device")
        pytest.skip("no CUDA device (gpu-marked tests run on the B200 box)")
    import plonky2_b200 as p

    return p


def _dev_helpers(st, tr, challenges):
    S = _stark_mod()
    return S.lookup_helper_columns(st, tr, challenges).cpu().numpy().view(np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("name,num_rows", [("permutation", None), ("range3", None), ("range2", None),
                                           ("range3", 1 << 16), ("range3", 1 << 20)])
def test_helper_columns_on_device_match_the_oracle(pb, name, num_rows):
    """gl_stark_lookup_helper_columns equals the column-wise restatement bit for bit (the 2^20 case runs the multi-CTA
    scan over 512 chunks)."""
    st, cfg, tr, _ = case(name, num_rows)
    gammas = [0xDEADBEEF, 0x7777777777]
    assert np.array_equal(_dev_helpers(st, tr, gammas), oracle_helper_columns(st, tr, gammas))


@pytest.mark.gpu
def test_helper_columns_zero_denominator_is_an_error(pb):
    from plonky2_b200 import NativeError

    st, cfg, tr, _ = case("range3")
    col0 = st.lookups()[0].columns[0].eval_table(tr, 5)
    with pytest.raises((NativeError, ZeroDivisionError), match="Tried to invert zero"):
        _dev_helpers(st, tr, [3, (P - col0) % P])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["range3", "range2", "fibonacci"])
def test_aux_quotient_on_device_matches_the_twin(pb, oracle, name):
    """compute_quotient_polys with the auxiliary commitment equals the twin's host quotient bit for bit, and its
    commitment's cap equals from_coeffs of the twin's chunks."""
    S = _stark_mod()
    st, cfg, tr, pis, parts = _twin(oracle, name)
    f = cfg.fri_config
    trace_c = pb.PolynomialBatch.from_values(tr, f.rate_bits, False, f.cap_height)
    aux_c = None
    if parts["helpers"] is not None:
        aux_c = pb.PolynomialBatch.from_values(parts["helpers"], f.rate_bits, False, f.cap_height)
        assert np.array_equal(aux_c.merkle_tree.cap.hashes, parts["auxiliary_polys_cap"])
    q = S.compute_quotient_polys(st, trace_c, pis, parts["alphas"], aux_c, parts["lookup_challenges"])
    assert np.array_equal(q.cpu().numpy().view(np.uint64), parts["quotient"])
    qc = S.commit_quotient_polys(st, q, tr.shape[1].bit_length() - 1, f.rate_bits, f.cap_height)
    assert np.array_equal(qc.merkle_tree.cap.hashes, parts["quotient_polys_cap"])
    for c in (trace_c, aux_c, qc):
        if c is not None:
            c.close()


def _proof_parts(proof, degree_bits):
    """What verify_stark_proof reads, from a StarkProofWithPublicInputs."""
    p = proof.proof
    return dict(trace_cap=p.trace_cap.hashes, auxiliary_polys_cap=p.auxiliary_polys_cap.hashes if p.auxiliary_polys_cap else None,
                quotient_polys_cap=p.quotient_polys_cap.hashes if p.quotient_polys_cap else None, openings=p.openings,
                fri_bytes=p.opening_proof.to_bytes(), public_inputs=proof.public_inputs, degree_bits=degree_bits)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL_CASES)
def test_prove_on_device_equals_the_twin(pb, oracle, name):
    """stark.prove on the device equals the CPU twin in every field (caps, openings, opening_proof.to_bytes()), and the
    restated verifier accepts it."""
    S = _stark_mod()
    st, cfg, tr, pis, parts = _twin(oracle, name)
    proof = S.prove(st, cfg, tr, pis)
    _assert_same_proof(proof, parts)
    assert verify_stark_proof(oracle, st, cfg, _proof_parts(proof, parts["degree_bits"])) is None


@pytest.mark.gpu
def test_a_wrong_frequency_is_refused(pb, oracle):
    """One frequency off by one leaves the Z column open at the wrap-around. With quotient degree factor 3 (constraint
    degree 4 at rate_bits 2, a coset of 4n points) prove() refuses the trace with "Quotient has failed"
    (prover.rs:396-401). With factor 2, as with the reference, the coset of 2n points leaves no coefficient to check:
    prove() returns a proof and the verifier rejects it."""
    from plonky2_b200 import NativeError

    S = _stark_mod()
    st = RangeCheckStark(1 << 7, 4, num_looking=2, second_lookup=False)
    cfg, tr, pis = fast_config(2), st.generate_trace(5), [(1 << 7) - 1]
    assert verify_stark_proof(oracle, st, cfg, _proof_parts(S.prove(st, cfg, tr, pis), 7)) is None
    bad = tr.copy()
    bad[1, 9] = (int(bad[1, 9]) + 1) % P
    with pytest.raises((NativeError, ValueError), match="Quotient has failed"):
        S.prove(st, cfg, bad, pis)
    st, cfg, tr, pis = case("range3")
    bad = tr.copy()
    bad[1, 9] = (int(bad[1, 9]) + 1) % P
    assert verify_stark_proof(oracle, st, cfg, _proof_parts(S.prove(st, cfg, bad, pis), 7)) is not None
