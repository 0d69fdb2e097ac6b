"""plonky2's compute_quotient_polys and the prover around it (SURVEY.md section 8f row 1).

CPU (`-m "not gpu"`):
  * the oracle's restatement of the quotient is pinned by the verifier's own check (plonky2/src/plonk/verifier.rs:85-107):
    vanishing_polys_zeta[i] == Z_H(zeta) * reduce_with_powers(quotient chunks at zeta, zeta^n), with the vanishing
    polynomial re-evaluated at zeta in plain Python (vanishing_poly.rs:29-164), for circuits holding rows of every gate
    type and a lookup table; a witness that breaks any one gate, a copy constraint, a looking pair or a table row fails it;
  * the product's vanishing PROGRAM (plonky2_b200/plonk.py) run by the kernel's own per-point source
    (plonky2_b200/csrc/gl_vanishing.cuh compiled for the host) equals the oracle bit for bit;
  * a whole ProofWithPublicInputs assembled from the oracle's pieces is accepted by a restated verify() (transcript
    replay, vanishing identity in F_{p^2}, FRI) and rejected after tampering; the product's prover host logic, proof
    readers, get_challenges and compression are run against it with the oracle standing in for the device calls.
GPU (`-m gpu`): gl_plonk_quotient through the C ABI equals the oracle bit for bit, chained after the device-resident
Z / partial-products commitment; the quotient commitment equals from_coeffs of the oracle's chunks; prove_with_witness
produces the CPU prover's bytes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import P, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P_ = int(P)

# (num_wires, num_routed_wires, max_quotient_degree_factor, rate_bits, degree_bits)
SHAPES = [
    (12, 8, 4, 2, 4),     # two selector groups, partial-product chunks of 4
    (13, 8, 3, 2, 4),     # quotient_degree_factor 3: coset of 4n points, the top n coefficients must vanish
    (24, 16, 8, 3, 3),    # one selector for all gates, chunks of 8
    (135, 80, 8, 3, 5),   # CircuitConfig::standard_recursion_config
    (135, 80, 8, 3, 5, 9),  # ... with nine PoseidonGate rows (a hash chain): two selector groups, 123 gate constraints
    # ... and a row of every other gate type built so far: three selector groups
    (135, 80, 8, 3, 5, 4, ("ArithmeticExtensionGate", "MulExtensionGate", "BaseSumGate", "BaseSumGate4", "ReducingGate",
                           "ReducingExtensionGate", "PoseidonMdsGate", "RandomAccessGate", "ExponentiationGate",
                           "CosetInterpolationGate")),
]
NUM_EXTRA = len(SHAPES[5][6])
# ... plus a lookup table of 30 entries on two LookupTableGate rows and 80 lookups on two LookupGate rows
SHAPES.append(SHAPES[5] + (True,))
LOOKUP_SHAPE_64 = SHAPES[6][:4] + (6,) + SHAPES[6][5:]     # the same circuit on 64 rows (the GPU cases use this one)


def _plonk():
    from plonky2_b200 import plonk   # importing the host layer does not need the CUDA library

    return plonk


def _circuit(shape, **kw):
    import plonk_circuits as PC

    plonk = _plonk()
    nw, nr, qdf, rate_bits, degree_bits = shape[:5]
    if len(shape) > 5:
        kw.setdefault("poseidon_rows", shape[5])
    if len(shape) > 6:
        kw.setdefault("extra", shape[6])
    if len(shape) > 7:
        kw.setdefault("lookups", shape[7])
    cfg = plonk.CircuitConfig(num_wires=nw, num_routed_wires=nr, max_quotient_degree_factor=qdf, rate_bits=rate_bits,
                              cap_height=1, num_challenges=kw.pop("num_challenges", 2))
    return PC.FibonacciCircuit(plonk, cfg, degree_bits, seed=nw + qdf + len(shape), **kw)


def _challenges(seed, nc):
    v = [int(x) for x in synth(seed, (3 * nc,))]
    return v[:nc], v[nc:2 * nc], v[2 * nc:]


def _deltas(c, seed):
    """NUM_COINS_LOOKUP lookup challenges per challenge round, none for circuits without lookups."""
    return [int(x) for x in synth(seed ^ 0xD17A, (4 * c.config.num_challenges,))] if c.common.luts else []


def _oracle_commits(oracle, c, betas, gammas, deltas=()):
    cfg = c.config
    cs = oracle.Commit(c.constants_sigmas, cfg.rate_bits, cfg.cap_height)
    w = oracle.Commit(c.wires, cfg.rate_bits, cfg.cap_height)
    z = oracle.Commit(c.oracle_zs_partial_products(oracle, betas, gammas, deltas), cfg.rate_bits, cfg.cap_height)
    return cs, w, z


def _ev(coeffs, x):
    acc = 0
    for v in coeffs[::-1]:
        acc = (acc * x + int(v)) % P_
    return acc


def _vanishing_at(c, cs, w, z, zeta, betas, gammas, alphas, deltas=()):
    """eval_vanishing_poly (vanishing_poly.rs:29-164) at a base-field point, from the committed polynomials."""
    import plonk_circuits as PC

    cd, cfg = c.common, c.config
    n = c.n
    g = PC.root_of_unity(cd.degree_bits)
    consts_sigmas = [_ev(p, zeta) for p in cs.coeffs]
    wires = [_ev(p, zeta) for p in w.coeffs]
    zs_pp = [_ev(p, zeta) for p in z.coeffs]
    zs_pp_next = [_ev(p, zeta * g % P_) for p in z.coeffs]
    nsel = cd.selectors_info.num_selectors()
    circuit = c.oracle_circuit()
    constraint_terms = [0] * cd.num_gate_constraints
    for i, (kind, param, sel, g0, g1, *_) in enumerate(circuit["gates"]):
        s = consts_sigmas[sel]
        filt = 1
        for j in list(range(g0, g1)) + ([0xFFFFFFFF] if nsel > 1 else []):
            if j != i:
                filt = filt * (j - s) % P_
        k = consts_sigmas[nsel + cd.num_lookup_selectors:]
        if kind == 1:
            res = [k[t] - wires[t] for t in range(param)]
        elif kind == 2:
            res = [wires[t] - c.public_inputs_hash[t] for t in range(4)]
        elif kind == 3:
            res = [wires[4 * t + 3] - (wires[4 * t] * wires[4 * t + 1] * k[0] + wires[4 * t + 2] * k[1]) for t in range(param)]
        elif kind == 0:
            res = []
        else:   # the product's own gate code, over numbers (the oracle restates these gates independently in C++)
            pv = PC.PointVars(consts_sigmas, wires, c.public_inputs_hash).remove_prefix(nsel + cd.num_lookup_selectors)
            res = [int(v) for v in cd.gates[i].eval_unfiltered(pv)]
        for t, r in enumerate(res):
            constraint_terms[t] = (constraint_terms[t] + r * filt) % P_
    zh = (pow(zeta, n, P_) - 1) % P_
    l_0 = zh * pow(n * (zeta - 1) % P_, P_ - 2, P_) % P_     # eval_l_0(n, x), plonk_common.rs:69-79
    nc, nr, qdf, nprod = cfg.num_challenges, cfg.num_routed_wires, cd.quotient_degree_factor, cd.num_partial_products
    z1, pp = [], []
    for i in range(nc):
        z_x, z_gx = zs_pp[i], zs_pp_next[i]
        z1.append(l_0 * (z_x - 1) % P_)
        num = [(wires[j] + betas[i] * (cd.k_is[j] * zeta % P_) + gammas[i]) % P_ for j in range(nr)]
        den = [(wires[j] + betas[i] * consts_sigmas[cd.num_constants + j] + gammas[i]) % P_ for j in range(nr)]
        accs = [z_x] + zs_pp[nc + i * nprod: nc + (i + 1) * nprod] + [z_gx]
        for k in range(nprod + 1):
            a = b = 1
            for j in range(k * qdf, min((k + 1) * qdf, nr)):
                a, b = a * num[j] % P_, b * den[j] % P_
            pp.append((accs[k] * a - accs[k + 1] * b) % P_)
    lk = []
    for i in range(nc if cd.luts else 0):   # the product's check_lookup_constraints over numbers (the oracle restates it in C++)
        def product(vs):
            acc = PC.Fp(1)
            for v in vs:
                acc = acc * v
            return acc
        plonk = _plonk()
        rng = cd.lookup_range(i)
        d = deltas[4 * i:4 * i + 4]
        lk += [int(v) for v in plonk.check_lookup_constraints(
            cd, PC.PointVars(consts_sigmas, wires, c.public_inputs_hash), [PC.Fp(zs_pp[k]) for k in rng],
            [PC.Fp(zs_pp_next[k]) for k in rng], [PC.Fp(consts_sigmas[nsel + r]) for r in range(cd.num_lookup_selectors)],
            d, cd.lut_re_poly_evals(d), product)]
    terms = z1 + pp + lk + constraint_terms
    return [sum(pow(al, t, P_) * v for t, v in enumerate(terms)) % P_ for al in alphas], zh


@pytest.mark.parametrize("shape", SHAPES)
def test_oracle_quotient_passes_the_verifier_identity(oracle, shape):
    c = _circuit(shape)
    nc = c.config.num_challenges
    betas, gammas, alphas = _challenges(0x510 + shape[0], nc)
    deltas = _deltas(c, 0x511)
    cs, w, z = _oracle_commits(oracle, c, betas, gammas, deltas)
    q = oracle.plonk_quotient(c.oracle_circuit(), cs, w, z, c.public_inputs_hash, betas, gammas, alphas, deltas)
    qdf, n = c.common.quotient_degree_factor, c.n
    assert q.shape == (nc, n << (qdf - 1).bit_length())
    assert not q[:, qdf * n:].any()      # trim_to_len(quotient_degree) succeeds (prover.rs:327-331)
    for zeta in (int(synth(0x520 + shape[0], (1,))[0]), 3):
        want, zh = _vanishing_at(c, cs, w, z, zeta, betas, gammas, alphas, deltas)
        for i in range(nc):
            # reduce_with_powers(chunks at zeta, zeta^n) == the unsplit polynomial at zeta
            chunks = [_ev(q[i, k * n:(k + 1) * n], zeta) for k in range(qdf)]
            zn = pow(zeta, n, P_)
            assert sum(ch * pow(zn, k, P_) for k, ch in enumerate(chunks)) % P_ == _ev(q[i], zeta)
            assert want[i] == zh * _ev(q[i], zeta) % P_


def test_poseidon_gate_rows_hold_the_pinned_permutation(oracle):
    """The PoseidonGate rows of the test circuit are true Poseidon traces: their output wires equal the KAT-pinned
    permutation of the (swapped) inputs -- so the gate constraints that vanish on them are the reference's."""
    c = _circuit(SHAPES[4])
    assert len(c.poseidon_io) == 9
    for inputs, swap, outputs in c.poseidon_io:
        st = list(inputs)
        if swap:
            st[0:4], st[4:8] = st[4:8], st[0:4]
        assert [int(v) for v in oracle.poseidon(np.array(st, dtype=np.uint64))] == outputs


@pytest.mark.parametrize("broken", ["break_gate", "break_copy", "break_poseidon"])
def test_oracle_quotient_of_a_bad_witness_fails_the_verifier_identity(oracle, broken):
    for shape in (SHAPES[4:5] if broken == "break_poseidon" else SHAPES[:2]):
        c = _circuit(shape, **{broken: True})
        nc = c.config.num_challenges
        betas, gammas, alphas = _challenges(0x530, nc)
        cs, w, z = _oracle_commits(oracle, c, betas, gammas)
        q = oracle.plonk_quotient(c.oracle_circuit(), cs, w, z, c.public_inputs_hash, betas, gammas, alphas)
        zeta = int(synth(0x531, (1,))[0])
        want, zh = _vanishing_at(c, cs, w, z, zeta, betas, gammas, alphas)
        qdf, n = c.common.quotient_degree_factor, c.n
        trimmed = [_ev(q[i, :qdf * n], zeta) for i in range(nc)]
        assert any(want[i] != zh * trimmed[i] % P_ for i in range(nc))
        if qdf & (qdf - 1):   # a trimmed region exists: "Quotient has failed" (prover.rs:327-331)
            assert q[:, qdf * n:].any()


def test_selector_groups_follow_the_reference_rule():
    """selector_polynomials (gates/selectors.rs:114-194): one selector when max_gate_degree + num_gates - 1 <= max_degree,
    else greedy groups with |G| + max degree in G <= max_degree; UNUSED_SELECTOR outside a row's group."""
    plonk = _plonk()
    c = _circuit(SHAPES[3])
    info = c.common.selectors_info
    assert [g.id() for g in c.common.gates] == ["NoopGate", "ConstantGate { num_consts: 2 }", "PublicInputGate",
                                                "ArithmeticGate { num_ops: 20 }"]
    assert info.num_selectors() == 1 and list(info.groups[0]) == [0, 1, 2, 3] and c.common.num_constants == 3
    assert c.common.num_partial_products == 9 and c.common.num_gate_constraints == 20
    c = _circuit(SHAPES[0])
    info = c.common.selectors_info
    assert [list(g) for g in info.groups] == [[0, 1, 2], [3]] and info.selector_indices == [0, 0, 0, 1]
    s0, s1 = c.constant_vecs[0], c.constant_vecs[1]
    assert s0[0] == 2 and s0[1] == 1 and s0[2] == plonk.UNUSED_SELECTOR and s1[2] == 3 and s1[0] == plonk.UNUSED_SELECTOR
    assert s0[c.n - 1] == 0 and s1[c.n - 1] == plonk.UNUSED_SELECTOR     # NoopGate padding
    with pytest.raises(ValueError, match="too high degree"):
        _circuit((12, 8, 2, 1, 3))


@pytest.mark.parametrize("nc", [1, 3, 4])
def test_other_challenge_counts_through_the_kernel_source(oracle, emu_lib, nc):
    """num_challenges = 1, 3, 4 (the kernel's accumulator bound): identity for the oracle, bit-exactness for the program."""
    for shape in (SHAPES[1], SHAPES[6]):
        c = _circuit(shape, num_challenges=nc)
        betas, gammas, alphas = _challenges(0x5A0 + nc, nc)
        deltas = _deltas(c, 0x5A1)
        cs, w, z = _oracle_commits(oracle, c, betas, gammas, deltas)
        q = oracle.plonk_quotient(c.oracle_circuit(), cs, w, z, c.public_inputs_hash, betas, gammas, alphas, deltas)
        zeta = int(synth(0x5A2, (1,))[0])
        want, zh = _vanishing_at(c, cs, w, z, zeta, betas, gammas, alphas, deltas)
        assert all(want[i] == zh * _ev(q[i], zeta) % P_ for i in range(nc))
        assert np.array_equal(_emu_quotient(emu_lib, oracle, c, cs, w, z, betas, gammas, alphas, deltas), q)


@pytest.fixture(scope="module")
def emu_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu") / "libgl_vanishing_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-DGL_FORCE_32BIT_PATH", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "emu", "vanishing_emu.cpp")])
    return C.CDLL(out)


def _emu_quotient(L, oracle, c, cs, w, z, betas, gammas, alphas, deltas):
    """The product's program interpreted by the kernel's per-point source on the host, then coset_ifft."""
    cfg, cd = c.config, c.common
    nc = cfg.num_challenges
    b = cd.vanishing_program()
    prog, n_regs = b.compile()
    assert n_regs <= 64            # the schedule keeps the register set small (L1-resident on the device)
    consts = _plonk().program_constants(cd, b, c.public_inputs_hash, betas, gammas, deltas)
    ldes = [np.ascontiguousarray(o.leaves.T) for o in (cs, w, z)]     # column-major LDE in leaf order, like the device
    ptrs = (C.POINTER(C.c_uint64) * 3)(*[a.ctypes.data_as(C.POINTER(C.c_uint64)) for a in ldes])
    strides = (C.c_size_t * 3)(*[a.shape[1] for a in ldes])
    qd_bits = (cd.quotient_degree_factor - 1).bit_length()
    size = c.n << qd_bits
    vals = np.zeros((nc, size), dtype=np.uint64)
    al = np.array(alphas, dtype=np.uint64)
    L.emu_plonk_quotient_values.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                            C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    rc = L.emu_plonk_quotient_values(ptrs, strides, 3, cfg.rate_bits, cd.degree_bits, qd_bits, prog, len(prog),
                                     consts.ctypes.data, al.ctypes.data, nc, cd.num_vanishing_terms(), vals.ctypes.data)
    assert rc == 0
    return np.stack([oracle.coset_ifft(v, 14293326489335486720) for v in vals])   # .coset_ifft(F::coset_shift())


@pytest.mark.parametrize("shape", SHAPES + [LOOKUP_SHAPE_64, (135, 80, 8, 3, 6, 20), (135, 80, 8, 3, 7)])
def test_vanishing_program_through_the_kernel_source_on_host_matches_oracle(oracle, emu_lib, shape):
    c = _circuit(shape)
    nc = c.config.num_challenges
    betas, gammas, alphas = _challenges(0x540 + shape[0], nc)
    deltas = _deltas(c, 0x541)
    cs, w, z = _oracle_commits(oracle, c, betas, gammas, deltas)
    want = oracle.plonk_quotient(c.oracle_circuit(), cs, w, z, c.public_inputs_hash, betas, gammas, alphas, deltas)
    assert np.array_equal(_emu_quotient(emu_lib, oracle, c, cs, w, z, betas, gammas, alphas, deltas), want)


@pytest.mark.parametrize("broken", ["pair", "table"])
def test_lookup_argument_rejects_a_wrong_witness(oracle, broken):
    """A looking pair that is not in the table, or a table row that differs from the committed table (get_lut_poly): the
    oracle's quotient no longer satisfies the verifier identity."""
    c = _circuit(SHAPES[6], break_lookup=broken)
    nc = c.config.num_challenges
    betas, gammas, alphas = _challenges(0x580, nc)
    deltas = _deltas(c, 0x581)
    cs, w, z = _oracle_commits(oracle, c, betas, gammas, deltas)
    q = oracle.plonk_quotient(c.oracle_circuit(), cs, w, z, c.public_inputs_hash, betas, gammas, alphas, deltas)
    zeta = int(synth(0x582, (1,))[0])
    want, zh = _vanishing_at(c, cs, w, z, zeta, betas, gammas, alphas, deltas)
    assert any(want[i] != zh * _ev(q[i], zeta) % P_ for i in range(nc))


def test_coset_interpolation_row_holds_the_true_interpolant():
    """The CosetInterpolationGate row's evaluation_value is the Lagrange interpolant of its 16 F_{p^2} values on the coset
    shift*H at the evaluation point (computed here directly from the definition) -- so the barycentric recurrences the
    gate constrains (and the oracle restates) compute what the reference's gate is documented to compute."""
    import plonk_circuits as PC

    plonk = _plonk()
    c = _circuit(SHAPES[5])
    info = [i for i in c.extra_info if i][0]
    xs = [info["shift"] * x % P_ for x in plonk.two_adic_subgroup(4)]
    z = plonk.Ext2(PC.Fp(info["point"][0]), PC.Fp(info["point"][1]))
    total = plonk.Ext2(PC.Fp(0), PC.Fp(0))
    for i, v in enumerate(info["values"]):
        term = plonk.Ext2(PC.Fp(v[0]), PC.Fp(v[1]))
        den = 1
        for j, xj in enumerate(xs):
            if j != i:
                term = term * (z - xj)
                den = den * (xs[i] - xj) % P_
        total = total + term.scalar_mul(pow(den, P_ - 2, P_))
    assert [int(total.a), int(total.b)] == info["value"]


@pytest.mark.parametrize("which", range(NUM_EXTRA))
def test_each_gate_type_rejects_a_wrong_witness(oracle, which):
    """One wire of the `which`-th extra gate row off by one: the oracle's quotient no longer satisfies the verifier
    identity (the gate's constraints are not vacuous)."""
    shape = SHAPES[5]
    c = _circuit(shape, break_extra=which)
    nc = c.config.num_challenges
    betas, gammas, alphas = _challenges(0x570 + which, nc)
    cs, w, z = _oracle_commits(oracle, c, betas, gammas)
    q = oracle.plonk_quotient(c.oracle_circuit(), cs, w, z, c.public_inputs_hash, betas, gammas, alphas)
    zeta = int(synth(0x571, (1,))[0])
    want, zh = _vanishing_at(c, cs, w, z, zeta, betas, gammas, alphas)
    assert any(want[i] != zh * _ev(q[i], zeta) % P_ for i in range(nc))


# ----------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def pb():
    import torch

    if not torch.cuda.is_available():
        if os.environ.get("GL_REQUIRE_GPU") == "1":
            raise AssertionError("GPU tests need a CUDA device")
        pytest.skip("no CUDA device (gpu-marked tests run on the B200 box)")
    import plonky2_b200 as p

    p.default_context()
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [SHAPES[0], SHAPES[1], (135, 80, 8, 3, 7), (135, 80, 8, 3, 6, 20), SHAPES[5], LOOKUP_SHAPE_64])
def test_plonk_quotient_on_device_matches_oracle(pb, oracle, shape):
    """The prover's third phase without leaving the device (plonk/prover.rs:220-352): wires + constants_sigmas
    commitments -> Z / partial products commitment (device) -> quotient polynomials (device, LDEs read in place) ->
    quotient commitment; coefficients and cap bit for bit equal to the oracle's."""
    import torch

    from plonky2_b200 import plonk
    from plonky2_b200.prover import commit_zs_partial_products

    c = _circuit(shape)
    cfg, cd = c.config, c.common
    nc, nr = cfg.num_challenges, cfg.num_routed_wires
    betas, gammas, alphas = _challenges(0x550 + shape[0], nc)
    deltas = _deltas(c, 0x551)
    ocs, ow, oz = _oracle_commits(oracle, c, betas, gammas, deltas)
    want = oracle.plonk_quotient(c.oracle_circuit(), ocs, ow, oz, c.public_inputs_hash, betas, gammas, alphas, deltas)
    cs = pb.PolynomialBatch.from_values(c.constants_sigmas, cfg.rate_bits, False, cfg.cap_height)
    w = pb.PolynomialBatch.from_values(c.wires, cfg.rate_bits, False, cfg.cap_height)
    wires_dev = torch.from_numpy(c.wires[:nr].view(np.int64)).cuda()
    sigmas_dev = torch.from_numpy(c.sigmas.view(np.int64)).cuda()
    if cd.luts:
        # with lookups the second commitment also holds the RE / Sum / LDC columns (prover.rs:227-245): Z and partial
        # products from gl_partial_products_and_zs, the lookup columns from gl_lookup_polys, committed together
        from plonky2_b200.prover import compute_all_lookup_polys, wires_permutation_partial_products_and_zs

        zs, pps = [], []
        for beta, gamma in zip(betas, gammas):
            out = wires_permutation_partial_products_and_zs(c.wires[:nr], c.sigmas, cd.k_is, beta, gamma, cd.quotient_degree_factor)
            zs.append(out[-1])
            pps += list(out[:-1])
        lk = compute_all_lookup_polys(c.wires, nr, cfg.max_quotient_degree_factor, deltas, c.lookup_rows, nc)
        z = pb.PolynomialBatch.from_values(np.concatenate([np.stack(zs + pps), lk]), cfg.rate_bits, False, cfg.cap_height)
    else:
        z = commit_zs_partial_products(wires_dev, sigmas_dev, cd.k_is, betas, gammas, cd.quotient_degree_factor, cfg.rate_bits,
                                       cfg.cap_height)
    assert np.array_equal(z.merkle_tree.cap.hashes, oz.cap)
    q = plonk.compute_quotient_polys(cd, cs, c.public_inputs_hash, w, z, betas, gammas, alphas, deltas)
    got = q.cpu().numpy().view(np.uint64)
    assert np.array_equal(got, want)
    qc = plonk.commit_quotient_polys(cd, q)
    qdf, n = cd.quotient_degree_factor, c.n
    chunks = np.concatenate([want[i, :qdf * n].reshape(qdf, n) for i in range(nc)])   # quotient_poly.chunks(degree)
    oq = oracle.Commit(chunks, cfg.rate_bits, cfg.cap_height, is_coeffs=True)
    assert np.array_equal(qc.merkle_tree.cap.hashes, oq.cap)
    for b in (cs, w, z, qc):
        b.close()


@pytest.mark.gpu
def test_plonk_quotient_of_a_bad_witness_is_rejected(pb):
    """quotient_degree_factor 3: the coset has 4n points and trim_to_len(3n) must find zeros; a broken gate leaves a
    non-zero tail -> "Quotient has failed" (prover.rs:327-331)."""
    import torch

    from plonky2_b200 import NativeError, plonk
    from plonky2_b200.prover import commit_zs_partial_products

    c = _circuit(SHAPES[1], break_gate=True)
    cfg, cd = c.config, c.common
    betas, gammas, alphas = _challenges(0x560, cfg.num_challenges)
    cs = pb.PolynomialBatch.from_values(c.constants_sigmas, cfg.rate_bits, False, cfg.cap_height)
    w = pb.PolynomialBatch.from_values(c.wires, cfg.rate_bits, False, cfg.cap_height)
    wires_dev = torch.from_numpy(c.wires[:cfg.num_routed_wires].view(np.int64)).cuda()
    sigmas_dev = torch.from_numpy(c.sigmas.view(np.int64)).cuda()
    z = commit_zs_partial_products(wires_dev, sigmas_dev, cd.k_is, betas, gammas, cd.quotient_degree_factor, cfg.rate_bits,
                                   cfg.cap_height)
    with pytest.raises((NativeError, ValueError), match="Quotient has failed"):
        plonk.compute_quotient_polys(cd, cs, c.public_inputs_hash, w, z, betas, gammas, alphas)
    for b in (cs, w, z):
        b.close()


# ----------------------------------------------------------------------------- the whole proof
def _fri_cfg(c):
    from plonky2_b200.fri import FriConfig

    # standard_recursion_config's FRI shape with fewer queries / grinding bits so that the CPU twin stays quick
    return FriConfig(rate_bits=c.config.rate_bits, cap_height=c.config.cap_height, proof_of_work_bits=6,
                     reduction_strategy=("ConstantArityBits", 2, 2), num_query_rounds=6)


PROOF_SHAPES = [SHAPES[0], SHAPES[3], LOOKUP_SHAPE_64]


@pytest.mark.parametrize("shape", PROOF_SHAPES)
def test_whole_proof_is_accepted_by_the_restated_verifier(oracle, shape):
    """prove (plonk/prover.rs:132-360) assembled from the oracle's restatements produces a ProofWithPublicInputs that
    verify (plonk/verifier.rs:20-120) accepts: transcript replay, the vanishing-polynomial identity at zeta in F_{p^2},
    the FRI opening proof; and rejects after tampering with an opening or with the public inputs."""
    import plonk_circuits as PC

    plonk = _plonk()
    c = _circuit(shape, public_inputs=[3, 1, 4, 1, 5])
    digest = [int(x) for x in synth(0x590, (4,))]
    fri_cfg = _fri_cfg(c)
    proof_bytes, parts = PC.oracle_prove(oracle, c, digest, fri_cfg, c.public_inputs)
    assert PC.oracle_verify(oracle, plonk, c, digest, fri_cfg, parts) is None
    bad = dict(parts, openings=dict(parts["openings"]))
    w = bad["openings"]["wires"].copy()
    w[0, 0] ^= np.uint64(1)
    bad["openings"]["wires"] = w
    assert PC.oracle_verify(oracle, plonk, c, digest, fri_cfg, bad) is not None
    bad = dict(parts, public_inputs=[3, 1, 4, 1, 6])
    assert PC.oracle_verify(oracle, plonk, c, digest, fri_cfg, bad) is not None
    assert PC.oracle_verify(oracle, plonk, c, [digest[0] ^ 1] + digest[1:], fri_cfg, parts) is not None


@pytest.mark.parametrize("shape", PROOF_SHAPES)
def test_prove_host_logic_with_cpu_backends(oracle, shape, monkeypatch):
    """The HOST side of plonk.prove_with_witness -- transcript order, challenge bookkeeping, ranges, FRI instance, proof
    serialisation -- run on the CPU by standing the oracle's pieces in for the device calls (commitments, Z / partial
    products, lookup columns, quotient, evaluations, prove_openings): the bytes must equal the CPU twin's. The device calls
    themselves are compared with the same oracle pieces one by one in the `-m gpu` tests."""
    import plonk_circuits as PC

    import plonky2_b200.fri as fri_mod
    import plonky2_b200.hash as hash_mod
    import plonky2_b200.proof as proof_mod
    import plonky2_b200.prover as prover_mod
    from plonky2_b200 import plonk

    c = _circuit(shape, public_inputs=[3, 1, 4, 1, 5])
    cfg, cd = c.config, c.common
    digest = [int(x) for x in synth(0x590, (4,))]
    fri_cfg = _fri_cfg(c)
    want, _ = PC.oracle_prove(oracle, c, digest, fri_cfg, c.public_inputs)

    class Cap:
        def __init__(self, hashes):
            self.hashes = hashes

    class Tree:
        def __init__(self, commit):
            self.cap = Cap(commit.cap)

    class Batch:   # a PolynomialBatch whose device work is done by the oracle
        def __init__(self, commit):
            self.o, self.merkle_tree, self.num_polys, self.degree_log = commit, Tree(commit), commit.B, commit.log_n
            self.ctx = ctx

        @classmethod
        def from_values(cls, values, rate_bits, blinding, cap_height, ctx=None):
            assert not blinding
            return cls(oracle.Commit(values, rate_bits, cap_height))

        def close(self):
            pass

    class Ctx:
        device, h = 0, None

    ctx = Ctx()

    def commit_zs(wires_dev, sigmas_dev, k_is, betas, gammas, degree, rate_bits, cap_height, ctx=None):
        assert np.array_equal(wires_dev, c.wires[:cfg.num_routed_wires]) and np.array_equal(sigmas_dev, c.sigmas)
        return Batch(oracle.Commit(c.oracle_zs_partial_products(oracle, betas, gammas), rate_bits, cap_height))

    def quotient(cd_, cs, pih, w, z, betas, gammas, alphas, deltas=()):
        return oracle.plonk_quotient(c.oracle_circuit(), cs.o, w.o, z.o, pih, betas, gammas, alphas, deltas)

    def commit_quotient(cd_, q, ctx=None):
        qdf, n = cd.quotient_degree_factor, c.n
        chunks = np.concatenate([q[i, :qdf * n].reshape(qdf, n) for i in range(q.shape[0])])
        return Batch(oracle.Commit(chunks, cfg.rate_bits, cfg.cap_height, is_coeffs=True))

    def evals(requests):
        return [np.array([oracle.eval_poly_base_at_ext(p, z) for p in b.o.coeffs], dtype=np.uint64).reshape(-1, 2)
                for b, z in requests]

    class FriBytes:
        def __init__(self, b):
            self.b = b

        def to_bytes(self):
            return self.b

    import plonky2_b200.challenger as challenger_mod

    class LoggingChallenger(challenger_mod.Challenger):   # the product's host transcript, with a log to replay
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
        och = oracle.Challenger()     # continue the product transcript inside the oracle's prover: replay it
        for kind, v in challenger.log:
            if kind == "observe":
                och.observe_element(v)
            else:
                assert och.get_challenge() == v
        batches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in instance.batches]
        assert [o.num_polys for o in instance.oracles] == [b.num_polys for b in oracles]
        params = oracle.make_params(cfg.rate_bits, cfg.cap_height, fri_cfg.proof_of_work_bits, fri_cfg.num_query_rounds,
                                    fri_params.reduction_arity_bits)
        return FriBytes(oracle.prove_openings([b.o for b in oracles], batches, och, params))

    monkeypatch.setattr(challenger_mod, "Challenger", LoggingChallenger)
    monkeypatch.setattr(plonk, "PolynomialBatch", Batch)
    monkeypatch.setattr(plonk, "_to_device", lambda columns, ctx: np.ascontiguousarray(columns, dtype=np.uint64))
    monkeypatch.setattr(plonk, "compute_quotient_polys", quotient)
    monkeypatch.setattr(plonk, "commit_quotient_polys", commit_quotient)
    monkeypatch.setattr(prover_mod, "commit_zs_partial_products", commit_zs)
    monkeypatch.setattr(prover_mod, "wires_permutation_partial_products_and_zs",
                        lambda w, s, k, beta, gamma, degree, ctx=None: oracle.partial_products_and_zs(w, s, k, beta, gamma, degree))
    monkeypatch.setattr(prover_mod, "compute_all_lookup_polys",
                        lambda w, nr, qdf, deltas, rows, nc, ctx=None: np.concatenate(
                            [oracle.lookup_polys(w, nr, qdf, deltas[4 * k:4 * k + 4], rows) for k in range(nc)]))
    monkeypatch.setattr(proof_mod, "eval_commitments", evals)
    monkeypatch.setattr(fri_mod, "prove_openings", prove_openings)
    monkeypatch.setattr(hash_mod.PoseidonHash, "hash_no_pad", staticmethod(lambda x, ctx=None: oracle.hash_no_pad(x)))
    cs = Batch(oracle.Commit(c.constants_sigmas, cfg.rate_bits, cfg.cap_height))
    prover_data = plonk.ProverOnlyCircuitData(cs, c.sigmas, digest, fri_cfg.fri_params(cd.degree_bits, False))
    proof = plonk.prove_with_witness(prover_data, cd, c.wires, c.public_inputs, ctx=ctx)
    assert proof.to_bytes() == want


@pytest.mark.gpu
@pytest.mark.parametrize("shape", PROOF_SHAPES)
def test_prove_on_device_is_byte_identical_to_the_cpu_prover(pb, oracle, shape):
    """plonk.prove_with_witness: wires commitment, Z / partial products (+ lookups), quotient, openings and FRI on the
    device, the transcript on the host -- write_proof_with_public_inputs equals the CPU twin's bytes, which the restated
    verifier accepts."""
    import plonk_circuits as PC

    from plonky2_b200 import plonk

    c = _circuit(shape, public_inputs=[3, 1, 4, 1, 5])
    cfg, cd = c.config, c.common
    digest = [int(x) for x in synth(0x590, (4,))]
    fri_cfg = _fri_cfg(c)
    want, parts = PC.oracle_prove(oracle, c, digest, fri_cfg, c.public_inputs)
    assert PC.oracle_verify(oracle, plonk, c, digest, fri_cfg, parts) is None
    cs = pb.PolynomialBatch.from_values(c.constants_sigmas, cfg.rate_bits, False, cfg.cap_height)
    prover_data = plonk.ProverOnlyCircuitData(cs, c.sigmas, digest, fri_cfg.fri_params(cd.degree_bits, False))
    proof = plonk.prove_with_witness(prover_data, cd, c.wires, c.public_inputs)
    assert proof.to_bytes() == want
    cs.close()


@pytest.mark.parametrize("shape", PROOF_SHAPES)
def test_proof_bytes_round_trip_challenges_and_compression(oracle, shape):
    """read_proof_with_public_inputs / write_... round trip on the CPU prover's bytes; get_challenges replayed by the
    product's host code gives the prover's own query indices and grinding witness; Proof::compress shrinks the proof and
    keeps one initial-tree proof per distinct index."""
    import plonk_circuits as PC

    plonk = _plonk()
    c = _circuit(shape, public_inputs=[3, 1, 4, 1, 5])
    digest = [int(x) for x in synth(0x590, (4,))]
    fri_cfg = _fri_cfg(c)
    fri_params = fri_cfg.fri_params(c.common.degree_bits, False)
    data, parts = PC.oracle_prove(oracle, c, digest, fri_cfg, c.public_inputs, taps=True)
    proof = plonk.ProofWithPublicInputs.from_bytes(data, c.common, fri_params)
    assert proof.to_bytes() == data and proof.public_inputs == [3, 1, 4, 1, 5]
    assert proof.get_public_inputs_hash() == c.public_inputs_hash
    ch = proof.get_challenges(digest, c.common, fri_params)
    assert ch["fri_query_indices"] == [int(i) for i in parts["taps"]["query_indices"]]
    assert proof.proof.opening_proof.pow_witness == parts["taps"]["pow_witness"]
    assert [tuple(int(x) for x in b) for b in parts["taps"]["betas"]] == [tuple(b) for b in ch["fri_betas"]]
    lz = 64 - int(ch["fri_pow_response"]).bit_length()
    assert lz >= fri_cfg.proof_of_work_bits                                   # the grinding check of the verifier
    comp = proof.compress(digest, c.common, fri_params)
    cbytes = comp.to_bytes()
    assert len(cbytes) < len(data)
    distinct = sorted(set(ch["fri_query_indices"]))
    assert sorted(comp.proof.opening_proof.initial_trees_proofs) == distinct
    # the caps, openings, final polynomial and witness are carried over untouched
    head = 3 * 4 * 8 * (1 << c.config.cap_height)
    assert cbytes[:head] == data[:head]


# ----------------------------------------------------------------------------- the reference's own gate test
def _all_gates():
    plonk = _plonk()
    cfg = plonk.CircuitConfig()
    return [plonk.NoopGate(), plonk.ConstantGate(2), plonk.PublicInputGate(), plonk.ArithmeticGate.new_from_config(cfg),
            plonk.ArithmeticExtensionGate.new_from_config(cfg), plonk.MulExtensionGate.new_from_config(cfg),
            plonk.BaseSumGate.new_from_config(cfg, 2), plonk.BaseSumGate(31, 4), plonk.ReducingGate(43),
            plonk.ReducingExtensionGate(32), plonk.ExponentiationGate.new_from_config(cfg),
            plonk.RandomAccessGate.new_from_config(cfg, 4), plonk.RandomAccessGate.new_from_config(cfg, 1),
            plonk.PoseidonMdsGate(), plonk.PoseidonGate(), plonk.CosetInterpolationGate(4, 8), plonk.CosetInterpolationGate(2),
            plonk.LookupGate.new_from_config(cfg), plonk.LookupTableGate.new_from_config(cfg)]


@pytest.mark.parametrize("k", range(19))
def test_low_degree_like_the_reference_gate_tests(oracle, k):
    """test_low_degree (plonky2/src/gates/gate_testing.rs:22-68), which every gate file of the reference runs: the
    constraints applied to random witness polynomials of degree < 32 are polynomials of degree <= 31 * gate.degree()
    (the value the selector grouping relies on) and there are num_constraints() of them. Beyond the reference: the bound
    is attained, so no gate over-declares its degree."""
    import plonk_circuits as PC

    gate = _all_gates()[k]
    WITNESS_SIZE = 32
    rate_bits = gate.degree().bit_length()            # log2_ceil(degree + 1)
    size = WITNESS_SIZE << rate_bits
    rng = np.random.default_rng(1000 + k)

    def random_low_degree_matrix(num_polys):
        cols = []
        for _ in range(num_polys):
            coeffs = np.zeros(size, dtype=np.uint64)
            coeffs[:WITNESS_SIZE] = PC.rnd(rng, WITNESS_SIZE)
            cols.append(oracle.fft(coeffs))            # .lde(rate_bits).fft()
        return np.stack(cols) if cols else np.zeros((0, size), dtype=np.uint64)

    wires, constants = random_low_degree_matrix(gate.num_wires()), random_low_degree_matrix(gate.num_constants())
    pih = [int(x) for x in PC.rnd(rng, 4)]
    evals = np.zeros((gate.num_constraints(), size), dtype=np.uint64)
    for p in range(size):
        res = gate.eval_unfiltered(PC.PointVars(constants[:, p], wires[:, p], pih))
        assert len(res) == gate.num_constraints(), "eval should return num_constraints() constraints"
        evals[:, p] = [int(v) for v in res]
    degrees = []
    for row in evals:
        co = oracle.ifft(row)
        nz = np.nonzero(co)[0]
        degrees.append(int(nz[-1]) if len(nz) else 0)
    expected = (WITNESS_SIZE - 1) * gate.degree()
    assert all(d <= expected for d in degrees), (gate.id()[:40], expected, degrees)
    if degrees:
        assert max(degrees) == expected, (gate.id()[:40], expected, max(degrees))


def test_coset_shifts_are_distinct_cosets():
    """field/src/cosets.rs:26-55 (`distinct_cosets`): the shifts k_i = g^i of get_unique_coset_shifts give pairwise
    different cosets of the size-2^n subgroup, i.e. (k_i / k_j)^(2^n) != 1 -- what the permutation argument's identity
    polynomials k_i * x rely on."""
    plonk = _plonk()
    shifts = plonk.get_unique_coset_shifts(80)
    for bits in (5, 12, 20):
        powered = [pow(k, 1 << bits, P_) for k in shifts]
        assert len(set(powered)) == len(shifts)
