"""starky's prover (SURVEY.md section 8f row 1): Stark constraints, logUp lookups, the quotient polynomials and their
commitment, and prove(), mirroring starky/src/{stark.rs, config.rs, constraint_consumer.rs, lookup.rs, vanishing_poly.rs,
prover.rs, fibonacci_stark.rs, permutation_stark.rs}. The constraints of a Stark -- its own, then the lookups' -- are
recorded ONCE as a straight-line program (ConstraintBuilder) and evaluated by gl_stark_quotient_aux on every point of the
quotient coset, reading the trace and auxiliary LDEs in place on the device; the same program is evaluated on the host over
F_{p^2} for the constraint-binding step. The logUp helper columns are computed on the device from the uploaded trace
(gl_stark_lookup_helper_columns)."""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _native as N
from . import field as F
from .polynomial_batch import PolynomialBatch

OP_LOCAL, OP_NEXT, OP_CONST, OP_ADD, OP_SUB, OP_MUL, OP_EMIT, OP_AUX_LOCAL, OP_AUX_NEXT = range(9)
MAX_INSTR = 256  # GL_STARK_MAX_INSTR
KIND_CONSTRAINT, KIND_TRANSITION, KIND_FIRST_ROW, KIND_LAST_ROW = range(4)


class StarkInstr(C.Structure):
    _fields_ = [("op", C.c_uint16), ("a", C.c_uint16), ("b", C.c_uint16), ("pad_", C.c_uint16)]


class Expr:
    """A value of the constraint program (the P: PackedField of eval_packed_generic)."""

    def __init__(self, b, idx):
        self.b, self.idx = b, idx

    def _bin(self, op, other):
        other = other if isinstance(other, Expr) else self.b.constant(other)
        return self.b._push(op, self.idx, other.idx)

    def __add__(self, o):
        return self._bin(OP_ADD, o)

    def __sub__(self, o):
        return self._bin(OP_SUB, o)

    def __mul__(self, o):
        return self._bin(OP_MUL, o)

    __radd__, __rmul__ = __add__, __mul__


class ConstraintBuilder:
    """Records eval_packed_generic as instructions; doubles as the ConstraintConsumer (constraint_consumer.rs:46-84)."""

    def __init__(self, num_columns, num_public_inputs, num_aux=0, num_lookup_challenges=0):
        # consts[0:num_pi] (public inputs) and consts[num_pi:num_bound] (lookup challenges) are bound at evaluation time
        self.num_bound = num_public_inputs + num_lookup_challenges
        self.instrs, self.consts = [], [None] * self.num_bound
        self.num_columns, self.num_pi, self.num_aux = num_columns, num_public_inputs, num_aux
        self._cache = {}

    def _push(self, op, a=0, b=0):
        key = (op, a, b)
        if op != OP_EMIT and key in self._cache:
            return self._cache[key]
        self.instrs.append((op, a, b))
        e = Expr(self, len(self.instrs) - 1)
        if op != OP_EMIT:
            self._cache[key] = e
        return e

    # StarkEvaluationFrame (evaluation_frame.rs:12-40)
    def local(self, col):
        assert 0 <= col < self.num_columns
        return self._push(OP_LOCAL, col)

    def next(self, col):
        assert 0 <= col < self.num_columns
        return self._push(OP_NEXT, col)

    def aux_local(self, k):
        assert 0 <= k < self.num_aux
        return self._push(OP_AUX_LOCAL, k)

    def aux_next(self, k):
        assert 0 <= k < self.num_aux
        return self._push(OP_AUX_NEXT, k)

    def public_input(self, k):
        assert 0 <= k < self.num_pi
        return self._push(OP_CONST, k)

    def lookup_challenge(self, j):
        """The j-th lookup challenge (the `beta` of get_grand_product_challenge_set, lookup.rs:525-543)."""
        assert 0 <= j < self.num_bound - self.num_pi
        return self._push(OP_CONST, self.num_pi + j)

    def constant(self, v):
        v = int(v) % F.ORDER
        if v not in self.consts[self.num_bound:]:
            self.consts.append(v)
        return self._push(OP_CONST, self.num_bound + self.consts[self.num_bound:].index(v))

    def bind(self, public_inputs, lookup_challenges=()):
        """consts of the program: the public inputs, the lookup challenges, then the program's constants."""
        if len(public_inputs) != self.num_pi or len(lookup_challenges) != self.num_bound - self.num_pi:
            raise N.ShapeError("expected %d public inputs and %d lookup challenges" % (self.num_pi, self.num_bound - self.num_pi))
        return np.array([int(x) % F.ORDER for x in list(public_inputs) + list(lookup_challenges)] + self.consts[self.num_bound:],
                        dtype=np.uint64)

    # ConstraintConsumer
    def constraint(self, e):
        self._push(OP_EMIT, e.idx, KIND_CONSTRAINT)

    def constraint_transition(self, e):
        self._push(OP_EMIT, e.idx, KIND_TRANSITION)

    def constraint_first_row(self, e):
        self._push(OP_EMIT, e.idx, KIND_FIRST_ROW)

    def constraint_last_row(self, e):
        self._push(OP_EMIT, e.idx, KIND_LAST_ROW)

    def program(self):
        if len(self.instrs) > MAX_INSTR:
            raise N.ShapeError("constraint program of %d instructions (max %d)" % (len(self.instrs), MAX_INSTR))
        arr = (StarkInstr * len(self.instrs))()
        for i, (op, a, b) in enumerate(self.instrs):
            arr[i].op, arr[i].a, arr[i].b = op, a, b
        return arr


# ------------------------------------------------------------------ logUp lookups (starky/src/lookup.rs:33-416)
class Column:
    """Column<F> (lookup.rs:132-399): sum of coeff * local[c], plus sum of coeff * next[c], plus a constant."""

    def __init__(self, linear_combination=(), next_row_linear_combination=(), constant=0):
        self.linear_combination = [(int(c), int(f) % F.ORDER) for c, f in linear_combination]
        self.next_row_linear_combination = [(int(c), int(f) % F.ORDER) for c, f in next_row_linear_combination]
        self.constant = int(constant) % F.ORDER

    @classmethod
    def single(cls, c):
        return cls([(c, 1)])

    @classmethod
    def single_next_row(cls, c):
        return cls((), [(c, 1)])

    @classmethod
    def constant_column(cls, v):
        """Column::constant"""
        return cls((), (), v)

    @classmethod
    def linear_combination_with_constant(cls, terms, constant):
        terms = list(terms)
        assert terms
        return cls(terms, (), constant)

    @classmethod
    def linear_combination_and_next_row_with_constant(cls, terms, next_terms, constant):
        terms, next_terms = list(terms), list(next_terms)
        assert terms or next_terms
        return cls(terms, next_terms, constant)

    def _lc(self, b, terms, read):
        acc = None
        for c, f in terms:
            t = read(c) if f == 1 else read(c) * f
            acc = t if acc is None else acc + t
        return acc

    def _finish(self, b, acc):
        if acc is None:
            return b.constant(self.constant)
        return acc + self.constant if self.constant else acc

    def eval(self, b):
        """eval (lookup.rs:290-300): local terms only."""
        return self._finish(b, self._lc(b, self.linear_combination, b.local))

    def eval_with_next(self, b):
        """eval_with_next (lookup.rs:302-316)."""
        a = self._lc(b, self.linear_combination, b.local)
        n = self._lc(b, self.next_row_linear_combination, b.next)
        return self._finish(b, n if a is None else (a if n is None else a + n))

    def eval_table(self, table, row):
        """eval_table (lookup.rs:318-329) on a host (columns, n) array."""
        n = table.shape[1]
        acc = self.constant
        for c, f in self.linear_combination:
            acc += int(table[c, row]) * f
        for c, f in self.next_row_linear_combination:
            acc += int(table[c, (row + 1) % n]) * f
        return acc % F.ORDER


class Filter:
    """Filter<F> (lookup.rs:33-126): sum of Column * Column products plus sum of Columns; the default is always on."""

    def __init__(self, products=(), constants=None):
        self.products = list(products)
        self.constants = [Column.constant_column(1)] if constants is None else list(constants)

    @classmethod
    def new_simple(cls, col):
        return cls((), [col])

    def eval_filter(self, b):
        """eval_filter (lookup.rs:68-84)."""
        acc = None
        for c1, c2 in self.products:
            t = c1.eval_with_next(b) * c2.eval_with_next(b)
            acc = t if acc is None else acc + t
        for c in self.constants:
            t = c.eval_with_next(b)
            acc = t if acc is None else acc + t
        return b.constant(0) if acc is None else acc


class Lookup:
    """Lookup<F> (lookup.rs:403-427): looking columns with their filters, a table column and its frequencies."""

    def __init__(self, columns, table_column, frequencies_column, filter_columns):
        assert len(columns) == len(filter_columns)
        self.columns, self.table_column = list(columns), table_column
        self.frequencies_column, self.filter_columns = frequencies_column, list(filter_columns)

    def num_helper_columns(self, constraint_degree):
        """One helper column per chunk of max(1, constraint_degree - 1) looking columns, plus Z."""
        return -(-len(self.columns) // _chunk_size(constraint_degree)) + 1


def _chunk_size(constraint_degree):
    """constraint_degree.checked_sub(1).unwrap_or(1); degree 1 would ask for chunks of 0 columns."""
    if constraint_degree == 1:
        raise N.ShapeError("lookups need a constraint degree other than 1")
    return max(1, constraint_degree - 1)


def eval_packed_lookups(stark, b, num_challenges):
    """eval_packed_lookups_generic (lookup.rs:804-863) with eval_helper_columns (lookup.rs:653-700) into the builder:
    for every lookup and challenge gamma, the chunk constraints of the helper columns, Z(0) = 0, and the Z step."""
    degree = stark.constraint_degree()
    start = 0
    for lookup in stark.lookups():
        nh = lookup.num_helper_columns(degree)
        cs = _chunk_size(degree)
        for j in range(num_challenges):
            gamma = b.lookup_challenge(j)
            cols = [c.eval_with_next(b) for c in lookup.columns]   # combine with beta = 1: f + gamma below
            helpers = [b.aux_local(start + k) for k in range(nh - 1)]
            for k, h in enumerate(helpers):
                chunk, fs = cols[k * cs:(k + 1) * cs], lookup.filter_columns[k * cs:(k + 1) * cs]
                if len(chunk) == 2:
                    c0, c1 = chunk[0] + gamma, chunk[1] + gamma
                    f0, f1 = fs[0].eval_filter(b), fs[1].eval_filter(b)
                    b.constraint(c1 * c0 * h - f0 * c1 - f1 * c0)
                elif len(chunk) == 1:
                    b.constraint((chunk[0] + gamma) * h - fs[0].eval_filter(b))
                else:
                    raise N.ShapeError("Allow other constraint degrees")
            z, next_z = b.aux_local(start + nh - 1), b.aux_next(start + nh - 1)
            table_with_challenge = lookup.table_column.eval(b) + gamma
            acc = b.constant(0)
            for h in helpers:
                acc = acc + h
            y = acc * table_with_challenge - lookup.frequencies_column.eval(b)
            b.constraint_first_row(z)
            b.constraint((next_z - z) * table_with_challenge - y)
            start += nh


class LogupTerm(C.Structure):
    _fields_ = [("col", C.c_uint32), ("next", C.c_uint32), ("coeff", C.c_uint64)]


class LogupColumn(C.Structure):
    _fields_ = [("term_begin", C.c_uint32), ("n_terms", C.c_uint32), ("constant", C.c_uint64)]


class LogupFilter(C.Structure):
    _fields_ = [("prod_begin", C.c_uint32), ("n_prods", C.c_uint32), ("sum_begin", C.c_uint32), ("n_sums", C.c_uint32)]


class LogupLookup(C.Structure):
    _fields_ = [("looking_begin", C.c_uint32), ("n_looking", C.c_uint32), ("table", C.c_uint32), ("frequencies", C.c_uint32)]


class LogupDesc(C.Structure):
    _fields_ = [("terms", C.POINTER(LogupTerm)), ("columns", C.POINTER(LogupColumn)), ("filter_columns", N.u32p),
                ("filters", C.POINTER(LogupFilter)), ("lookups", C.POINTER(LogupLookup)), ("n_terms", C.c_uint32),
                ("n_columns", C.c_uint32), ("n_filter_columns", C.c_uint32), ("n_lookups", C.c_uint32)]


def logup_descriptor(lookups):
    """The flat gl_logup_desc of a list of Lookups (include/plonky2_b200.h). Returns (desc, arrays it points into)."""
    main, filt = [], []              # main: every lookup's looking columns, table, frequencies; then the filters' columns
    lks = []
    for lk in lookups:
        lks.append((len(main), len(lk.columns), len(main) + len(lk.columns), len(main) + len(lk.columns) + 1))
        main += list(lk.columns) + [lk.table_column, lk.frequencies_column]
    columns = list(main)
    fdesc, fcols = [(0, 0, 0, 0)] * len(main), []
    for lk, (lb, nl, _, _) in zip(lookups, lks):
        for k, f in enumerate(lk.filter_columns):
            pb = len(fcols)
            for c1, c2 in f.products:
                fcols += [len(columns), len(columns) + 1]
                columns += [c1, c2]
            sb = len(fcols)
            for c in f.constants:
                fcols.append(len(columns))
                columns.append(c)
            fdesc[lb + k] = (pb, len(f.products), sb, len(f.constants))
    fdesc += [(0, 0, 0, 0)] * (len(columns) - len(fdesc))
    terms = []
    carr = (LogupColumn * max(1, len(columns)))()
    for i, c in enumerate(columns):
        tb = len(terms)
        terms += [(col, 0, f) for col, f in c.linear_combination] + [(col, 1, f) for col, f in c.next_row_linear_combination]
        carr[i].term_begin, carr[i].n_terms, carr[i].constant = tb, len(terms) - tb, c.constant
    tarr = (LogupTerm * max(1, len(terms)))(*[LogupTerm(*t) for t in terms])
    farr = (LogupFilter * max(1, len(fdesc)))(*[LogupFilter(*f) for f in fdesc])
    larr = (LogupLookup * max(1, len(lks)))(*[LogupLookup(*t) for t in lks])
    fc = np.array(fcols + [0], dtype=np.uint32)
    d = LogupDesc(tarr, carr, fc.ctypes.data_as(N.u32p), farr, larr, len(terms), len(columns), len(fcols), len(lks))
    return d, (tarr, carr, farr, larr, fc)


# ------------------------------------------------------------------ Stark, StarkConfig (stark.rs, config.rs)
@dataclass
class StarkConfig:
    """StarkConfig (starky/src/config.rs:20-108)."""
    security_bits: int
    num_challenges: int
    fri_config: object

    @classmethod
    def standard_fast_config(cls):
        """config.rs:52-64"""
        from .fri import starky_standard_fast_fri_config

        return cls(100, 2, starky_standard_fast_fri_config())

    def fri_params(self, degree_bits):
        """config.rs:66-68"""
        return self.fri_config.fri_params(degree_bits, False)

    def observe(self, challenger):
        """config.rs:102-108"""
        challenger.observe_element(self.security_bits)
        challenger.observe_element(self.num_challenges)
        self.fri_config.observe(challenger)


class Stark:
    """Stark<F, D> (starky/src/stark.rs:24-279): COLUMNS, PUBLIC_INPUTS, eval (eval_packed_generic), constraint_degree,
    lookups."""
    COLUMNS = 0
    PUBLIC_INPUTS = 0

    def eval(self, vars, yield_constr):
        raise NotImplementedError

    def constraint_degree(self):
        raise NotImplementedError

    def quotient_degree_factor(self):
        """stark.rs:87-92"""
        d = self.constraint_degree()
        return 0 if d == 0 else max(1, d - 1)

    def num_quotient_polys(self, config):
        """stark.rs:94-96"""
        return self.quotient_degree_factor() * config.num_challenges

    def lookups(self):
        """stark.rs:254-256: none by default."""
        return []

    def uses_lookups(self):
        return bool(self.lookups())

    def num_lookup_helper_columns(self, config, num_challenges=None):
        """stark.rs:258-265"""
        nc = config.num_challenges if num_challenges is None else num_challenges
        return sum(lk.num_helper_columns(self.constraint_degree()) for lk in self.lookups()) * nc

    def fri_instance(self, zeta, g, config):
        """fri_instance (stark.rs:101-172) without cross-table lookups: trace, auxiliary and quotient polynomials at zeta;
        trace and auxiliary polynomials at g * zeta."""
        from .fri import FriBatchInfo, FriInstanceInfo, FriOracleInfo, FriPolynomialInfo

        oracles = [FriOracleInfo(self.COLUMNS, False)]
        trace_info = FriPolynomialInfo.from_range(0, range(self.COLUMNS))
        aux_info = []
        if self.uses_lookups():
            na = self.num_lookup_helper_columns(config)
            aux_info = FriPolynomialInfo.from_range(len(oracles), range(na))
            oracles.append(FriOracleInfo(na, False))
        quot_info = []
        nq = self.num_quotient_polys(config)
        if nq > 0:
            quot_info = FriPolynomialInfo.from_range(len(oracles), range(nq))
            oracles.append(FriOracleInfo(nq, False))
        g_zeta = F.ext_mul((int(g) % F.ORDER, 0), zeta)
        return FriInstanceInfo(oracles, [FriBatchInfo(zeta, trace_info + aux_info + quot_info),
                                         FriBatchInfo(g_zeta, trace_info + aux_info)])

    def constraint_program(self, num_lookup_challenges=0):
        """eval_vanishing_poly (vanishing_poly.rs:28-63) as a program: the STARK's constraints, then -- with lookup
        challenges -- eval_packed_lookups_generic, in that order (the consumer reduces with Horner)."""
        nlc = num_lookup_challenges if self.uses_lookups() else 0
        b = ConstraintBuilder(self.COLUMNS, self.PUBLIC_INPUTS, self.num_lookup_helper_columns(None, nlc) if nlc else 0, nlc)
        self.eval(b, b)
        if nlc:
            eval_packed_lookups(self, b, nlc)
        return b


class FibonacciStark(Stark):
    """FibonacciStark (starky/src/fibonacci_stark.rs:19-120): columns (x0, x1), x0' = x1, x1' = x0 + x1; public inputs
    x0, x1 of the first row and x1 of the last row."""
    COLUMNS = 2
    PUBLIC_INPUTS = 3
    PI_INDEX_X0, PI_INDEX_X1, PI_INDEX_RES = 0, 1, 2

    def __init__(self, num_rows):
        self.num_rows = num_rows

    def generate_trace(self, x0, x1):
        """generate_trace (fibonacci_stark.rs:42-53): two columns of num_rows values."""
        cols = np.empty((2, self.num_rows), dtype=np.uint64)
        a, b = int(x0) % F.ORDER, int(x1) % F.ORDER
        for i in range(self.num_rows):
            cols[0, i], cols[1, i] = a, b
            a, b = b, (a + b) % F.ORDER
        return cols

    def eval(self, vars, yield_constr):
        """eval_packed_generic (fibonacci_stark.rs:73-95)."""
        l0, l1, n0, n1 = vars.local(0), vars.local(1), vars.next(0), vars.next(1)
        yield_constr.constraint_first_row(l0 - vars.public_input(self.PI_INDEX_X0))
        yield_constr.constraint_first_row(l1 - vars.public_input(self.PI_INDEX_X1))
        yield_constr.constraint_last_row(l1 - vars.public_input(self.PI_INDEX_RES))
        yield_constr.constraint_transition(n0 - l1)           # x0' <- x1
        yield_constr.constraint_transition(n1 - l0 - l1)      # x1' <- x0 + x1

    def constraint_degree(self):
        return 2


def compute_quotient_polys(stark, trace_commitment, public_inputs, alphas, auxiliary_polys_commitment=None,
                           lookup_challenges=None):
    """compute_quotient_polys (prover.rs:488-668) on the device. Returns a torch int64 CUDA tensor (num_challenges, size)
    of quotient-polynomial coefficients, size = n << log2_ceil(quotient_degree_factor), or None if the Stark has no
    quotient. Raises if the vanishing polynomial is not divisible by Z_H. With lookup_challenges the lookups' constraints
    are included; they read the helper columns from auxiliary_polys_commitment."""
    import torch

    qdf = stark.quotient_degree_factor()
    if qdf == 0:
        return None
    lc = list(lookup_challenges) if lookup_challenges is not None and stark.uses_lookups() else []
    b = stark.constraint_program(len(lc))
    if len(public_inputs) != stark.PUBLIC_INPUTS:
        raise N.ShapeError("expected %d public inputs" % stark.PUBLIC_INPUTS)
    if b.num_aux and (auxiliary_polys_commitment is None or auxiliary_polys_commitment.num_polys < b.num_aux):
        raise N.ShapeError("the lookups need %d auxiliary polynomials" % b.num_aux)
    consts = b.bind(public_inputs, lc)
    al = np.array([int(a) % F.ORDER for a in alphas], dtype=np.uint64)
    qd_bits = (qdf - 1).bit_length()
    size = (1 << trace_commitment.degree_log) << qd_bits
    ctx = trace_commitment.ctx
    out = torch.empty((len(al), size), dtype=torch.int64, device="cuda:%d" % ctx.device)
    prog = b.program()
    aux_h = auxiliary_polys_commitment.h if auxiliary_polys_commitment is not None else None
    N.check(N.lib().gl_stark_quotient_aux(ctx.h, trace_commitment.h, aux_h, prog, len(b.instrs), N.np_ptr(consts),
                                          len(consts), N.np_ptr(al), len(al), qdf, N.vp(out.data_ptr())), ctx.h)
    ctx.synchronize()
    return out


def commit_quotient_polys(stark, quotient_polys, degree_bits, rate_bits, cap_height, ctx=None):
    """'split quotient polys' + 'compute quotient commitment' (prover.rs:391-421): every polynomial is cut into
    quotient_degree_factor chunks of n coefficients, all chunks are committed with from_coeffs -- straight from the
    device tensor compute_quotient_polys returned."""
    ctx = ctx or N.default_context()
    qdf = stark.quotient_degree_factor()
    n = 1 << degree_bits
    num, size = quotient_polys.shape
    B = num * qdf
    L = N.lib()
    h = N.vp()
    N.check(L.gl_commit_begin(ctx.h, B, degree_bits, rate_bits, cap_height, 0, 0, 1, None, C.byref(h)), ctx.h)
    try:
        for j in range(num):
            N.check(L.gl_commit_add_columns(h, j * qdf, qdf, N.vp(quotient_polys[j].data_ptr()), n, N.COLS_COEFFS,
                                            N.MEM_DEVICE), ctx.h)
        N.check(L.gl_commit_finish(h, None, N.MEM_DEVICE), ctx.h)
        ctx.synchronize()
    except Exception:
        L.gl_commit_destroy(h)
        raise
    return PolynomialBatch(h, ctx, B, degree_bits, rate_bits, cap_height, False)


class PermutationStark(Stark):
    """PermutationStark (starky/src/permutation_stark.rs:17-90): columns (x, x + 1 rotated, 1) where column 0 looks up
    column 1 with frequencies column 2; no constraints of its own and constraint degree 0, so no quotient."""
    COLUMNS = 3
    PUBLIC_INPUTS = 1

    def __init__(self, num_rows):
        self.num_rows = num_rows

    def generate_trace(self, x0):
        """generate_trace (permutation_stark.rs:32-44)."""
        x0 = int(x0) % F.ORDER
        cols = np.empty((3, self.num_rows), dtype=np.uint64)
        for i in range(self.num_rows):
            cols[0, i], cols[1, i], cols[2, i] = (x0 + i) % F.ORDER, (x0 + 1 + i) % F.ORDER, 1
        cols[1, self.num_rows - 1] = x0
        return cols

    def eval(self, vars, yield_constr):
        pass

    def constraint_degree(self):
        return 0

    def lookups(self):
        return [Lookup([Column.single(0)], Column.single(1), Column.single(2), [Filter()])]


def eval_l_0_and_l_last(log_n, x):
    """eval_l_0_and_l_last (vanishing_poly.rs:89-97) at x in F_{p^2}."""
    n = 1 << log_n
    g = F.primitive_root_of_unity(log_n)
    z_x = F.ext_sub(F.ext_pow(x, n), (1, 0))
    a = F.ext_mul((n % F.ORDER, 0), F.ext_sub(x, (1, 0)))
    c = F.ext_mul((n % F.ORDER, 0), F.ext_sub(F.ext_mul((g, 0), x), (1, 0)))
    return F.ext_mul(z_x, F.ext_inverse(a)), F.ext_mul(z_x, F.ext_inverse(c))


def eval_program_ext(b, consts, local_values, next_values, aux, aux_next, alphas, zeta, degree_bits):
    """The constraint program at one point zeta of F_{p^2} with the ConstraintConsumer of vanishing_poly.rs:124-137:
    returns one accumulator per alpha (consumer.accumulators())."""
    l_0, l_last = eval_l_0_and_l_last(degree_bits, zeta)
    last = F.inverse(F.primitive_root_of_unity(degree_bits))
    z_last = F.ext_sub(zeta, (last, 0))
    em = {KIND_CONSTRAINT: None, KIND_TRANSITION: z_last, KIND_FIRST_ROW: l_0, KIND_LAST_ROW: l_last}
    acc = [(0, 0)] * len(alphas)
    v = []

    def e(x):
        return (int(x[0]) % F.ORDER, int(x[1]) % F.ORDER)

    for op, a, c in b.instrs:
        r = None
        if op == OP_LOCAL:
            r = e(local_values[a])
        elif op == OP_NEXT:
            r = e(next_values[a])
        elif op == OP_AUX_LOCAL:
            r = e(aux[a])
        elif op == OP_AUX_NEXT:
            r = e(aux_next[a])
        elif op == OP_CONST:
            r = (int(consts[a]) % F.ORDER, 0)
        elif op == OP_ADD:
            r = F.ext_add(v[a], v[c])
        elif op == OP_SUB:
            r = F.ext_sub(v[a], v[c])
        elif op == OP_MUL:
            r = F.ext_mul(v[a], v[c])
        else:
            t = v[a] if em[c] is None else F.ext_mul(v[a], em[c])
            acc = [F.ext_add(F.ext_mul(x, (int(al) % F.ORDER, 0)), t) for x, al in zip(acc, alphas)]
        v.append(r)
    return acc


def compute_eval_vanishing_poly(stark, opening_set, lookup_challenges, public_inputs, alphas, zeta, degree_bits):
    """compute_eval_vanishing_poly (vanishing_poly.rs:109-170) without CTLs: the vanishing polynomial, lookups included,
    at zeta from (simulated or opened) values -- the constraint-binding step of the prover and the verifier's check."""
    lc = list(lookup_challenges) if lookup_challenges is not None else []
    b = stark.constraint_program(len(lc))
    return eval_program_ext(b, b.bind(public_inputs, lc), opening_set.local_values, opening_set.next_values,
                            opening_set.auxiliary_polys, opening_set.auxiliary_polys_next, alphas, zeta, degree_bits)


def lookup_helper_columns(stark, trace, lookup_challenges, ctx=None):
    """Every lookup's helper columns for every challenge (prover.rs:159-173 over lookup_helper_columns, lookup.rs:579-652),
    lookup-major, challenge-minor, on the device from a (COLUMNS, n) trace -- a torch CUDA tensor (as _to_device returns)
    or a host array. Returns a torch int64 CUDA tensor (num_lookup_helper_columns, n) of values."""
    import torch

    ctx = ctx or N.default_context()
    lookups = stark.lookups()
    if not isinstance(trace, torch.Tensor):
        trace = _to_device(trace, ctx)
    ncols, n = trace.shape
    log_n = F.log2_strict(n)
    nc = len(lookup_challenges)
    out = torch.empty((stark.num_lookup_helper_columns(None, nc), n), dtype=torch.int64, device=trace.device)
    desc, keep = logup_descriptor(lookups)
    ch = np.array([int(x) % F.ORDER for x in lookup_challenges] + [0], dtype=np.uint64)
    N.check(N.lib().gl_stark_lookup_helper_columns(ctx.h, N.vp(trace.data_ptr()), trace.stride(0), ncols, log_n,
                                                   C.addressof(desc), N.np_ptr(ch), nc, stark.constraint_degree(),
                                                   N.vp(out.data_ptr()), N.MEM_DEVICE), ctx.h)
    ctx.synchronize()
    return out


def _to_device(columns, ctx):
    """Host (columns, n) values -> torch int64 tensor on the context's GPU, uploaded once."""
    import torch

    dev = "cuda:%d" % ctx.device
    t = torch.from_numpy(np.ascontiguousarray(columns, dtype=np.uint64).view(np.int64)).to(dev)
    torch.cuda.synchronize(dev)
    return t


def _commit_values(values, rate_bits, cap_height, ctx):
    """from_values (oracle.rs:57-79, no blinding) of a device tensor (B, n) without a host round trip."""
    B, n = values.shape
    degree_bits = F.log2_strict(n)
    L = N.lib()
    h = N.vp()
    N.check(L.gl_commit_begin(ctx.h, B, degree_bits, rate_bits, cap_height, 0, 0, 1, None, C.byref(h)), ctx.h)
    try:
        N.check(L.gl_commit_add_columns(h, 0, B, N.vp(values.data_ptr()), values.stride(0), N.COLS_VALUES, N.MEM_DEVICE),
                ctx.h)
        N.check(L.gl_commit_finish(h, None, N.MEM_DEVICE), ctx.h)
        ctx.synchronize()
    except Exception:
        L.gl_commit_destroy(h)
        raise
    return PolynomialBatch(h, ctx, B, degree_bits, rate_bits, cap_height, False)


def simulated_opening_set(challenger, num_columns, num_aux, constraint_degree):
    """The simulated opening set of the constraint-binding step (prover.rs:266-319, get_dummy_polys in
    get_challenges.rs): ceil(total / num_extension_powers) extension challenges c, each giving c, c^d, c^{d^2}, ...
    (d = max(2, constraint_degree + 1)), sliced into local, next, auxiliary and (the whole rest) auxiliary-next values."""
    from .proof import StarkOpeningSet

    total = 2 * num_columns + 2 * num_aux
    pow_degree = max(2, constraint_degree + 1)
    num_extension_powers = max(1, 50 // (pow_degree - 1).bit_length() - 1)   # log2_ceil(pow_degree)
    zetas = challenger.get_n_extension_challenges(-(-total // num_extension_powers))
    per = min(num_extension_powers + 1, total)
    evals = []
    for z in zetas:
        for _ in range(per):
            evals.append(z)
            z = F.ext_pow(z, pow_degree)
    arr = np.array(evals, dtype=np.uint64).reshape(-1, 2)
    a0, a1 = 2 * num_columns, 2 * num_columns + num_aux
    return StarkOpeningSet(arr[:num_columns], arr[num_columns:a0], arr[a0:a1] if num_aux else None,
                           arr[a1:] if num_aux else None)


def prove(stark, config, trace, public_inputs, ctx=None):
    """prove (starky/src/prover.rs:40-484) without cross-table lookups: trace (COLUMNS, n) values to a
    StarkProofWithPublicInputs. The trace is uploaded once; its commitment, the lookups' helper columns and their
    commitment, the quotient and its commitment, the openings and the FRI proof run on the device, the transcript on the
    host in the reference's order."""
    from . import challenger as challenger_mod
    from . import fri as fri_mod
    from .proof import StarkOpeningSet, StarkProof, StarkProofWithPublicInputs

    trace = np.ascontiguousarray(trace, dtype=np.uint64)
    if trace.ndim != 2 or trace.shape[0] != stark.COLUMNS:
        raise N.ShapeError("the trace must be (%d, n)" % stark.COLUMNS)
    if len(public_inputs) != stark.PUBLIC_INPUTS:
        raise N.ShapeError("expected %d public inputs" % stark.PUBLIC_INPUTS)
    public_inputs = [int(x) % F.ORDER for x in public_inputs]
    n = trace.shape[1]
    degree_bits = F.log2_strict(n)
    fri_params = config.fri_params(degree_bits)
    rate_bits, cap_height = config.fri_config.rate_bits, config.fri_config.cap_height
    if fri_params.total_arities() > degree_bits + rate_bits - cap_height:
        raise N.ShapeError("FRI total reduction arity is too large.")
    if stark.constraint_degree() > (1 << rate_bits) + 1:
        raise N.ShapeError("The degree of the Stark constraints must be <= blowup_factor + 1")
    nc = config.num_challenges
    ctx = ctx or N.default_context()
    commitments = []
    try:
        trace_dev = _to_device(trace, ctx)
        trace_commitment = _commit_values(trace_dev, rate_bits, cap_height, ctx)
        commitments.append(trace_commitment)
        challenger = challenger_mod.Challenger()
        challenger.observe_elements(public_inputs)
        config.observe(challenger)
        challenger.observe_cap(trace_commitment.merkle_tree.cap)
        lookup_challenges, aux = None, None
        if stark.uses_lookups():
            # get_grand_product_challenge_set (lookup.rs:525-543): (beta, gamma) pairs, the betas are kept
            lookup_challenges = [challenger.get_n_challenges(2)[0] for _ in range(nc)]
            aux = _commit_values(lookup_helper_columns(stark, trace_dev, lookup_challenges, ctx), rate_bits, cap_height, ctx)
            commitments.append(aux)
            challenger.observe_cap(aux.merkle_tree.cap)
        del trace_dev
        alphas_prime = challenger.get_n_challenges(nc)
        poly_evals = simulated_opening_set(challenger, stark.COLUMNS, aux.num_polys if aux else 0, stark.constraint_degree())
        zeta_prime = challenger.get_extension_challenge()
        constraints = compute_eval_vanishing_poly(stark, poly_evals, lookup_challenges, public_inputs, alphas_prime,
                                                  zeta_prime, degree_bits)
        challenger.observe_extension_elements(constraints)                # bind the constraints
        alphas = challenger.get_n_challenges(nc)
        quotient_commitment = None
        if stark.quotient_degree_factor() > 0:
            q = compute_quotient_polys(stark, trace_commitment, public_inputs, alphas, aux, lookup_challenges)
            quotient_commitment = commit_quotient_polys(stark, q, degree_bits, rate_bits, cap_height, ctx)
            del q
            commitments.append(quotient_commitment)
            challenger.observe_cap(quotient_commitment.merkle_tree.cap)
        zeta = challenger.get_extension_challenge()
        if F.ext_pow(zeta, n) == (1, 0):
            raise N.NativeError("Opening point is in the subgroup.")
        g = F.primitive_root_of_unity(degree_bits)
        openings = StarkOpeningSet.new(zeta, g, trace_commitment, aux, quotient_commitment)
        challenger.observe_openings(openings.to_fri_openings())
        opening_proof = fri_mod.prove_openings(stark.fri_instance(zeta, g, config), commitments, challenger, fri_params)
        proof = StarkProof(trace_commitment.merkle_tree.cap, aux.merkle_tree.cap if aux else None,
                           quotient_commitment.merkle_tree.cap if quotient_commitment else None, openings, opening_proof)
        return StarkProofWithPublicInputs(proof, public_inputs)
    finally:
        for c in commitments:
            c.close()
