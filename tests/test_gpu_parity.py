"""GPU parity tests (run with `-m gpu` on the B200 box): every call goes through the C ABI
(libplonky2_b200.so) and is compared bit-for-bit with the CPU oracle on the same seeded inputs,
plus size-independent properties at larger sizes. /root/reference is never read here."""
import json
import os

import numpy as np
import pytest

from conftest import EDGE, P, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pb():
    import torch

    if not torch.cuda.is_available():
        # on the B200 box (GL_REQUIRE_GPU=1) a missing device is a loud failure, elsewhere the gpu tests skip
        if os.environ.get("GL_REQUIRE_GPU") == "1":
            raise AssertionError("GPU tests need a CUDA device")
        pytest.skip("no CUDA device (gpu-marked tests run on the B200 box)")
    import plonky2_b200 as p

    p.default_context()  # fails loudly if the CUDA extension is missing
    return p


# ----------------------------------------------------------------------------- NTT
@pytest.mark.parametrize("log_n", [0, 1, 2, 3, 4, 5, 7, 8, 10, 12, 13, 14, 16])
def test_fft_ifft_match_oracle(pb, oracle, log_n):
    n = 1 << log_n
    x = synth(0x01 + log_n, (3, n), canonical=False)
    got = pb.fft(x)
    for b in range(3):
        assert np.array_equal(got[b], oracle.fft(x[b])), (log_n, b)
    goti = pb.ifft(x)
    for b in range(3):
        assert np.array_equal(goti[b], oracle.ifft(x[b]))
    assert np.array_equal(pb.ifft(got), x % np.uint64(P))  # round trip returns the (canonical) input


def test_fft_reference_test_vector(pb, oracle):
    # field/src/fft.rs:215-249: deterministic i*1337 % 100, degree 200 padded to 256, zero_factor 0..3
    coeffs = np.array([(i * 1337) % 100 for i in range(200)] + [0] * 56, dtype=np.uint64)
    pts = pb.fft(coeffs)
    assert np.array_equal(pts, oracle.naive_coset_eval(coeffs, 1))
    assert np.array_equal(pb.ifft(pts), coeffs)
    for r in range(4):
        ext = pb.lde(coeffs, r)
        assert np.array_equal(pb.fft_with_options(ext, zero_factor=r), pb.fft(ext))
        assert np.array_equal(pb.fft(ext), oracle.fft(ext))


def test_edge_values_and_single_column(pb, oracle):
    x = np.array((EDGE * 6)[:64], dtype=np.uint64)
    assert np.array_equal(pb.fft(x), oracle.fft(x))
    assert np.array_equal(pb.ifft(x), oracle.ifft(x))


@pytest.mark.parametrize("log_n", [1, 4, 9, 13])
def test_coset_fft_and_ifft(pb, oracle, log_n):
    n = 1 << log_n
    x = synth(0x21 + log_n, (2, n))
    shift = int(synth(0x22, (1,))[0]) | 1
    got = pb.coset_fft(x, shift)
    for b in range(2):
        assert np.array_equal(got[b], oracle.coset_fft(x[b], shift))
    back = pb.coset_ifft(got, shift)
    assert np.array_equal(back, x)
    for b in range(2):
        assert np.array_equal(pb.coset_ifft(x, shift)[b], oracle.coset_ifft(x[b], shift))


def test_cfg1_2pow16_roundtrip(pb, oracle):
    # BASELINE.json configs[0]: 2^16-point forward + inverse NTT, single column, bit-exact vs CPU reference
    x = synth(0x01, (1 << 16,))
    y = pb.fft(x)
    assert np.array_equal(y, oracle.fft(x))
    assert np.array_equal(pb.ifft(y), x)
    assert np.array_equal(pb.ifft(x), oracle.ifft(x))


def test_ntt_linearity_large(pb):
    # size-independent property at 2^20 x 4 columns: NTT(a + c*b) = NTT(a) + c*NTT(b)
    n = 1 << 20
    a, b = synth(0x31, (2, n)), synth(0x32, (2, n))
    c = 0x1234567
    P_ = int(P)
    comb = ((a.astype(object) + c * b.astype(object)) % P_).astype(np.uint64)
    fa, fb, fc = pb.fft(a), pb.fft(b), pb.fft(comb)
    want = ((fa.astype(object) + c * fb.astype(object)) % P_).astype(np.uint64)
    assert np.array_equal(fc, want)
    assert np.array_equal(pb.ifft(fa), a)


def test_ntt_shape_errors(pb):
    with pytest.raises(ValueError):
        pb.fft(np.zeros(12, dtype=np.uint64))


# ----------------------------------------------------------------------------- Poseidon / Merkle
def test_poseidon_kats_on_device(pb, oracle):
    # the reference's 4 stored known-answer vectors (plonky2/src/hash/poseidon_goldilocks.rs:466-487) straight
    # through the DEVICE permutation (FP64-pipe formulation), 12 lanes in, 12 lanes out
    kat = json.load(open(os.path.join(ROOT, "tests", "golden", "poseidon_kat.json")))
    ins = np.array([[int(x) for x in v["input"]] for v in kat["vectors"]], dtype=np.uint64)
    exp = np.array([[int(x) for x in v["output"]] for v in kat["vectors"]], dtype=np.uint64)
    assert len(ins) == 4
    got = pb.PoseidonHash.permute_many(ins)
    assert np.array_equal(got, exp)
    # a few thousand random / non-canonical states against the oracle permutation (both forms agree on the KATs)
    st = synth(0x4B, (3000, 12), canonical=False)
    st[:len(EDGE)] = np.array([EDGE] * 12, dtype=np.uint64).T[:, :12]
    got = pb.PoseidonHash.permute_many(st)
    for i in list(range(40)) + list(range(2990, 3000)):
        assert got[i].tolist() == (oracle.poseidon(st[i]) % np.uint64(P)).tolist(), i
    # host transcript permutation = the same function
    h = st[17].copy()
    pb._native.lib().gl_poseidon_permute_host(pb._native.np_ptr(h))
    assert h.tolist() == got[17].tolist()


@pytest.mark.parametrize("W", [0, 1, 3, 4, 5, 7, 8, 9, 12, 16, 17, 33, 135])
def test_hash_many_matches_oracle(pb, oracle, W):
    rows = synth(0x41 + W, (257, W), canonical=False) if W else np.zeros((5, 0), dtype=np.uint64)
    got = pb.PoseidonHash.hash_many(rows)
    want = oracle.hash_many(rows) if W else np.zeros((5, 4), dtype=np.uint64)
    assert np.array_equal(got, want)
    if W:
        g2 = pb.PoseidonHash.hash_no_pad_many(rows[:9])
        for i in range(9):
            assert np.array_equal(g2[i], oracle.hash_no_pad(rows[i]))


def test_hash_extreme_inputs(pb, oracle):
    rows = np.array([(EDGE * 3)[i:i + 12] for i in range(12)], dtype=np.uint64)
    assert np.array_equal(pb.PoseidonHash.hash_many(rows), oracle.hash_many(rows))
    rows = np.full((4, 20), 2**64 - 1, dtype=np.uint64)
    assert np.array_equal(pb.PoseidonHash.hash_many(rows), oracle.hash_many(rows))


def test_hash_fp64_limb_stress(pb, oracle):
    """Inputs that maximise the FP64-pipe limbs of the device Poseidon (both 32-bit halves of every word near
    2^32, non-canonical words, sparse states): the exactness bound of gl_poseidon.cuh must hold on the GPU as it
    does in tests/emu/poseidon_f64_emu.cpp."""
    rng = np.random.default_rng(0xF64)
    rows = rng.integers(0, 2**63, size=(4096, 16), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    rows[0::4] |= np.uint64(0xFFFFFFF0FFFFFFF0)
    rows[1::4] = np.uint64(2**64 - 1) - (rows[1::4] & np.uint64(7))
    rows[2::4, 1:] = 0
    assert np.array_equal(pb.PoseidonHash.hash_many(rows), oracle.hash_many(rows))
    pairs = rows[:, :8].copy()
    got = pb.PoseidonHash.two_to_one_many(pairs[:256])
    for i in range(256):
        assert np.array_equal(got[i], oracle.two_to_one(pairs[i, :4], pairs[i, 4:]))


def test_two_to_one(pb, oracle):
    pairs = synth(0x51, (100, 8), canonical=False)
    got = pb.PoseidonHash.two_to_one_many(pairs)
    for i in range(100):
        assert np.array_equal(got[i], oracle.two_to_one(pairs[i, :4], pairs[i, 4:]))


@pytest.mark.parametrize("log_n,W,cap_height", [(8, 7, 0), (8, 7, 1), (8, 7, 8), (0, 5, 0), (3, 2, 3),
                                                (10, 12, 4), (11, 135, 4), (6, 4, 2), (12, 32, 4)])
def test_merkle_tree_matches_oracle(pb, oracle, log_n, W, cap_height):
    N = 1 << log_n
    leaves = synth(0x61 + log_n, (N, W))
    t = pb.MerkleTree(leaves, cap_height)
    d, cap = oracle.merkle_build(leaves, cap_height)
    assert np.array_equal(t.cap.hashes, cap)
    assert np.array_equal(t.digests, d)
    idx = sorted(set([0, N - 1, N // 2, N // 3]))
    lv, paths = t.open_many(idx)
    for k, i in enumerate(idx):
        assert np.array_equal(lv[k], leaves[i])
        assert np.array_equal(paths[k], oracle.merkle_prove(i, N, cap_height, d))
        assert oracle.merkle_verify(lv[k], i, paths[k], cap, cap_height)


def test_merkle_every_leaf_proof_verifies(pb, oracle):
    # merkle_tree.rs:269-311 (random 256 x 7 leaves, every proof against the cap)
    leaves = synth(0x71, (256, 7))
    for cap_height in (1, 8):
        t = pb.MerkleTree(leaves, cap_height)
        lv, paths = t.open_many(np.arange(256))
        cap = t.cap.hashes
        for i in range(256):
            assert oracle.merkle_verify(lv[i], i, paths[i], cap, cap_height)
    pb.verify_merkle_proof_to_cap(leaves[5], 5, t.cap, t.prove(5))
    with pytest.raises(ValueError):
        pb.verify_merkle_proof_to_cap(leaves[6], 5, t.cap, t.prove(5))


def test_merkle_cap_too_big(pb):
    with pytest.raises(ValueError) as e:
        pb.MerkleTree(synth(1, (8, 5)), 4)
    assert "should be at most log2(leaves.len())" in str(e.value)
    with pytest.raises(ValueError):
        pb.MerkleTree(synth(1, (12, 5)), 1)


def test_merkle_large_cap_property(pb, oracle):
    # 2^18 leaves x 12 (config 3 shape, reduced): cap equals the fold of the digest array's top pairs and a
    # sample of proofs verifies; full 2^23 is covered by bench.py's checks.
    N, W, h = 1 << 18, 12, 4
    leaves = synth(0x03, (N, W))
    t = pb.MerkleTree(leaves, h)
    d, cap = oracle.merkle_build(leaves, h)
    assert np.array_equal(t.cap.hashes, cap)
    lv, paths = t.open_many([1, 77777, N - 2])
    for k, i in enumerate([1, 77777, N - 2]):
        assert oracle.merkle_verify(lv[k], i, paths[k], cap, h)


# ----------------------------------------------------------------------------- PolynomialBatch
@pytest.mark.parametrize("B,log_n,r,h", [(5, 4, 2, 1), (3, 0, 3, 0), (1, 1, 1, 2), (9, 6, 3, 4), (135, 10, 3, 4),
                                         (20, 13, 3, 4), (16, 14, 1, 4), (2, 12, 0, 0), (17, 9, 2, 11)])
def test_from_values_matches_oracle(pb, oracle, B, log_n, r, h):
    n = 1 << log_n
    vals = synth(0x02 + B, (B, n), canonical=(B % 2 == 0))
    c = pb.PolynomialBatch.from_values(vals, r, False, h)
    o = oracle.Commit(vals, r, h)
    assert np.array_equal(c.polynomials, o.coeffs)
    assert np.array_equal(c.merkle_tree.cap.hashes, o.cap)
    assert np.array_equal(c.merkle_tree.leaves, o.leaves)
    assert np.array_equal(c.merkle_tree.digests, o.digests)
    N = n << r
    for (idx, step) in [(0, 1), (N // 2 - 1 if N > 1 else 0, 2 if N > 1 else 1), (N - 1, 1)]:
        assert np.array_equal(c.get_lde_values(idx, step), o.get_lde_values(idx, step))
    lv, paths = c.merkle_tree.open_many([0, N - 1])
    assert np.array_equal(lv[1], o.leaves[N - 1])
    if N > (1 << h):
        assert np.array_equal(paths[1], oracle.merkle_prove(N - 1, N, h, o.digests))
    c.close()


def test_from_coeffs_and_blinding(pb, oracle):
    B, log_n, r, h = 6, 7, 3, 2
    n, N = 1 << log_n, 1 << (log_n + r)
    co = synth(0x81, (B, n))
    salt = synth(0x82, (4, N))
    c = pb.PolynomialBatch.from_coeffs(co, r, True, h, salt=salt)
    o = oracle.Commit(co, r, h, salt=salt, is_coeffs=True)
    assert c.leaf_width == B + 4
    assert np.array_equal(c.merkle_tree.leaves, o.leaves)
    assert np.array_equal(c.merkle_tree.cap.hashes, o.cap)
    assert np.array_equal(c.get_lde_values(3, 1), o.get_lde_values(3, 1))  # salt stripped
    # OsRng-salted commitment: different caps, same unsalted LDE values
    c2 = pb.PolynomialBatch.from_coeffs(co, r, True, h)
    assert not np.array_equal(c2.merkle_tree.cap.hashes, o.cap)
    assert np.array_equal(c2.get_lde_values(3, 1), o.get_lde_values(3, 1))


def test_commit_shape_errors(pb):
    with pytest.raises(ValueError):
        pb.PolynomialBatch.from_values(np.zeros((2, 12), dtype=np.uint64), 1, False, 0)
    with pytest.raises(ValueError) as e:
        pb.PolynomialBatch.from_values(np.zeros((2, 8), dtype=np.uint64), 1, False, 5)
    assert "cap_height" in str(e.value)


def test_commit_lde_restricts_to_values(pb):
    # property at a larger size (B=8, n=2^16, r=3): LDE at rate 1 extends the same polynomial: the coeffs'
    # forward NTT returns the committed values, and the commitment of coeffs equals the commitment of values.
    B, log_n = 8, 16
    vals = synth(0x83, (B, 1 << log_n))
    c = pb.PolynomialBatch.from_values(vals, 3, False, 4)
    co = c.polynomials
    assert np.array_equal(pb.fft(co), vals)
    c2 = pb.PolynomialBatch.from_coeffs(co, 3, False, 4)
    assert np.array_equal(c2.merkle_tree.cap.hashes, c.merkle_tree.cap.hashes)


# ----------------------------------------------------------------------------- FRI
def _instance(pb, oracles_B, zeta, gzeta, z_polys):
    inst_batches = []
    all_polys = [pb.FriPolynomialInfo(o, i) for o, B in enumerate(oracles_B) for i in range(B)]
    inst_batches.append(pb.FriBatchInfo(zeta, all_polys))
    inst_batches.append(pb.FriBatchInfo(gzeta, [pb.FriPolynomialInfo(*p) for p in z_polys]))
    return pb.FriInstanceInfo([pb.FriOracleInfo(B, False) for B in oracles_B], inst_batches)


def _opened_values(oracle, ocommits, batches):
    vals = []
    for point, polys in batches:
        for (oi, pi) in polys:
            vals.append(oracle.eval_poly_base_at_ext(ocommits[oi].coeffs[pi], point))
    return np.array(vals, dtype=np.uint64)


@pytest.mark.parametrize("log_n,Bs,arity,pow_bits,nq", [(5, [3, 2], [1], 3, 4), (8, [4, 6, 2], [2, 2], 5, 6),
                                                       (10, [7, 9, 4, 3], [4], 8, 9),
                                                       (12, [20, 33, 20, 16], [4, 4], 16, 28),
                                                       (9, [5], [3, 1, 2], 4, 5), (7, [2, 2], [5], 2, 3),
                                                       (6, [3], [], 2, 3), (4, [1], [1, 1, 1], 0, 2)])
def test_prove_openings_bit_exact_and_verifies(pb, oracle, log_n, Bs, arity, pow_bits, nq):
    r, h = 3, (4 if log_n >= 8 else 1)
    n = 1 << log_n
    vals = [synth(0x04 + i, (B, n)) for i, B in enumerate(Bs)]
    commits = [pb.PolynomialBatch.from_values(v, r, False, h) for v in vals]
    ocommits = [oracle.Commit(v, r, h) for v in vals]
    zeta = (int(synth(0xA1, (1,))[0]), int(synth(0xA2, (1,))[0]))
    gz = pb.field.ext_mul(zeta, (pb.field.primitive_root_of_unity(log_n), 0))
    z_polys = [(len(Bs) - 1, i) for i in range(min(2, Bs[-1]))]
    inst = _instance(pb, Bs, zeta, gz, z_polys)
    obatches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in inst.batches]
    cfg = pb.FriConfig(r, h, pow_bits, ("Fixed", arity), nq)
    params = pb.FriParams(cfg, False, log_n, arity)
    oparams = oracle.make_params(r, h, pow_bits, nq, arity)

    # a transcript prefix both sides share
    ch, och = pb.Challenger(), oracle.Challenger()
    for c in commits:
        ch.observe_cap(c.merkle_tree.cap)
    for o in ocommits:
        och.observe_cap(o.cap)
    och_verify = och.clone()

    taps = {}
    proof = pb.prove_openings(inst, commits, ch, params, taps=taps)
    oproof, otaps = oracle.prove_openings(ocommits, obatches, och, oparams, taps=True)
    assert np.array_equal(taps["final_poly"], otaps["final_poly"])
    assert taps["pow_witness"] == otaps["pow_witness"]
    assert list(taps["query_indices"]) == otaps["query_indices"].tolist()
    assert proof.to_bytes() == oproof                      # bit-exact FRI proof bytes
    assert ch.get_challenge() == och.get_challenge()       # transcripts stay in sync
    # and the proof passes the restated verifier (fri/verifier.rs:62-241)
    opened = _opened_values(oracle, ocommits, obatches)
    rc = oracle.verify_fri_proof([o.cap for o in ocommits], Bs, [o.W for o in ocommits], obatches, opened,
                                 log_n, och_verify, oparams, proof.to_bytes())
    assert rc == 0
    # a corrupted proof must be rejected
    bad = bytearray(proof.to_bytes())
    bad[-9] ^= 1
    rc2 = oracle.verify_fri_proof([o.cap for o in ocommits], Bs, [o.W for o in ocommits], obatches, opened,
                                  log_n, oracle.Challenger(), oparams, bytes(bad))
    assert rc2 != 0


def test_fri_pow_smallest_nonce(pb, oracle):
    ctx = pb.default_context()
    st = synth(0xB1, (12,))
    for pos, bits in [(0, 0), (3, 7), (7, 10)]:
        nonce = np.zeros(1, dtype=np.uint64)
        pb._native.check(pb._native.lib().gl_fri_pow(ctx.h, pb._native.np_ptr(st), pos, bits,
                                                     pb._native.np_ptr(nonce)), ctx.h)
        # brute force on the oracle
        want = None
        for cand in range(1 << 14):
            s = st.copy()
            s[pos] = cand
            if (64 - int(oracle.poseidon(s)[7]).bit_length()) >= bits:
                want = cand
                break
        assert int(nonce[0]) == want


# ----------------------------------------------------------------------------- row-block sharding
@pytest.mark.parametrize("B,log_n,r,h,G", [(9, 8, 3, 4, 2), (9, 8, 3, 4, 8), (5, 10, 1, 4, 8), (5, 10, 1, 4, 16),
                                           (3, 13, 1, 3, 4), (4, 2, 1, 3, 8), (6, 6, 0, 2, 4)])
def test_sharded_commit_concatenates_to_single_device_commit(pb, oracle, B, log_n, r, h, G):
    # every shard is built on this one GPU; concatenated shards must equal the single-device commitment
    n, N = 1 << log_n, 1 << (log_n + r)
    vals = synth(0x05 + G, (B, n))
    salt = synth(0x06, (4, N)) if B == 9 else None
    o = oracle.Commit(vals, r, h, salt=salt)
    leaves, digests, caps = [], [], []
    for g in range(G):
        c = pb.PolynomialBatch.from_values(vals, r, salt is not None, h, salt=salt, shard=(g, G))
        assert np.array_equal(c.polynomials, o.coeffs)
        leaves.append(c.merkle_tree.leaves)
        digests.append(c.merkle_tree.digests)
        caps.append(c.merkle_tree.cap.hashes)
        # a local opening verifies against the local cap with the local index
        lv, paths = c.merkle_tree.open_many([0, c.local_rows - 1])
        assert oracle.merkle_verify(lv[1], c.local_rows - 1, paths[1], caps[-1], h - int(np.log2(G)))
        # and is the global opening of leaf g*rows + local
        gi = g * c.local_rows + c.local_rows - 1
        assert np.array_equal(lv[1], o.leaves[gi])
        assert np.array_equal(paths[1], oracle.merkle_prove(gi, N, h, o.digests))
        c.close()
    assert np.array_equal(np.concatenate(leaves), o.leaves)
    assert np.array_equal(np.concatenate(caps), o.cap)
    assert np.array_equal(np.concatenate(digests), o.digests)


def test_sharding_rejects_more_shards_than_cap_entries(pb):
    with pytest.raises(ValueError):
        pb.PolynomialBatch.from_values(synth(1, (2, 16)), 1, False, 1, shard=(0, 4))


# ----------------------------------------------------------------------------- large shapes (BASELINE configs)
@pytest.mark.parametrize("log_n", [17, 20, 22, 23, 24])
def test_large_ntt_against_oracle_and_roundtrip(pb, oracle, log_n):
    # exercises every tile size up to 2^12 x 2^12 (log_n = 24 is the per-transform maximum of this build)
    n = 1 << log_n
    x = synth(0x100 + log_n, (n,))
    y = pb.fft(x)
    assert np.array_equal(y, oracle.fft(x))
    assert np.array_equal(pb.ifft(y), x)


@pytest.mark.parametrize("log_n", [21, 22, 25])
def test_three_pass_ntt_spot_checks_and_roundtrip(pb, oracle, log_n):
    # n > 2^20 runs three passes (7+7+7 ... 9+8+8): a few outputs against Horner evaluation of the input polynomial
    # at w_n^k on the CPU (size-independent check), then ifft(fft(x)) == x
    n = 1 << log_n
    x = synth(0x90 + log_n, (n,))
    y = pb.fft(x)
    w = pb.field.primitive_root_of_unity(log_n)
    for k in (0, 1, 2, n // 2 + 5, n - 1, 0x12345 % n, (1 << (log_n - 7)) + 3):
        pt = (pow(w, k, P), 0)
        assert int(y[k]) == oracle.eval_poly_base_at_ext(x, pt)[0], (log_n, k)
    assert np.array_equal(pb.ifft(y), x)


def test_cfg3_merkle_2pow23_leaves_width12(pb, oracle):
    # BASELINE.json configs[2]: Poseidon Merkle commitment of 2^23 leaves x width 12, cap bit-exact vs CPU
    N, W, h = 1 << 23, 12, 4
    leaves = synth(0x03, (N, W))
    t = pb.MerkleTree(leaves, h)
    d, cap = oracle.merkle_build(leaves, h)
    assert np.array_equal(t.cap.hashes, cap)
    idx = [0, 12345, N - 1]
    lv, paths = t.open_many(idx)
    for k, i in enumerate(idx):
        assert np.array_equal(paths[k], oracle.merkle_prove(i, N, h, d))
        assert oracle.merkle_verify(lv[k], i, paths[k], cap, h)
    t.close()


def test_cfg5_shape_reduced_starky_commit_and_fri(pb, oracle):
    # starky standard_fast_config shape (rate_bits 1, cap 4, arity-16 rounds) at n = 2^16, 8 columns:
    # commitment vs oracle, then the FRI commit phase + proof bytes vs oracle.
    B, log_n, r, h = 8, 16, 1, 4
    vals = synth(0x05, (B, 1 << log_n))
    c = pb.PolynomialBatch.from_values(vals, r, False, h)
    o = oracle.Commit(vals, r, h)
    assert np.array_equal(c.merkle_tree.cap.hashes, o.cap)
    cfg = pb.starky_standard_fast_fri_config()
    params = cfg.fri_params(log_n, False)
    assert params.reduction_arity_bits == [4, 4, 4]
    zeta = (123456789, 987654321)
    inst = _instance(pb, [B], zeta, pb.field.ext_mul(zeta, (pb.field.primitive_root_of_unity(log_n), 0)), [(0, 0)])
    obatches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in inst.batches]
    ch, och = pb.Challenger(), oracle.Challenger()
    ch.observe_cap(c.merkle_tree.cap)
    och.observe_cap(o.cap)
    proof = pb.prove_openings(inst, [c], ch, params)
    oproof = oracle.prove_openings([o], obatches, och, oracle.make_params(r, h, 16, 84, [4, 4, 4]))
    assert proof.to_bytes() == oproof


def test_multi_gpu_sharded_prove(pb):
    """Needs >= 2 GPUs (skipped on the single-GPU test box): torchrun, one rank per GPU, NCCL cap all-gather,
    routed openings; rank 0 checks caps and proof bytes against the CPU oracle."""
    import subprocess
    import sys
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tests", "mgpu_prove_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MGPU_PROVE_CHECK OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("B,log_n", [(3, 0), (5, 1), (7, 9), (20, 13), (4, 16)])
def test_eval_commitment_at_extension_point(pb, oracle, B, log_n):
    # OpeningSet::new's eval_commitment (plonk/proof.rs:313-351) vs Horner evaluation on the CPU
    vals = synth(0xE0 + B, (B, 1 << log_n))
    c = pb.PolynomialBatch.from_values(vals, 1, False, 0)
    coeffs = c.polynomials
    for z in [(0, 0), (1, 0), (5, 7), (int(synth(0xE1, (1,))[0]), int(synth(0xE2, (1,))[0]))]:
        got = c.eval_commitment(z)
        for b in range(B):
            assert tuple(int(x) for x in got[b]) == oracle.eval_poly_base_at_ext(coeffs[b], z)


@pytest.mark.parametrize("R,log_n,deg", [(13, 4, 4), (80, 10, 8), (80, 14, 8), (5, 0, 2), (9, 12, 3)])
def test_partial_products_and_zs(pb, oracle, R, log_n, deg):
    # wires_permutation_partial_products_and_zs (plonk/prover.rs:387-449) vs the oracle restatement
    from plonky2_b200.prover import wires_permutation_partial_products_and_zs as gpu_pp

    n = 1 << log_n
    w, sg, k = synth(0xF0 + R, (R, n)), synth(0xF1 + R, (R, n)), synth(0xF2, (R,))
    beta, gamma = int(synth(0xF3, (1,))[0]), int(synth(0xF4, (1,))[0])
    got = gpu_pp(w, sg, k, beta, gamma, deg)
    want = oracle.partial_products_and_zs(w, sg, k, beta, gamma, deg)
    assert np.array_equal(got, want)
    # a valid permutation (sigma = identity: s_sigma = k_j * x) makes every quotient 1: Z == 1 everywhere
    wn = pb.field.primitive_root_of_unity(log_n)
    xs = np.array([pow(wn, i, P) for i in range(n)], dtype=object)
    ident = np.array([[int(k[j]) * int(x) % P for x in xs] for j in range(R)], dtype=np.uint64) if n <= 1024 else None
    if ident is not None:
        one = gpu_pp(w, ident, k, beta, gamma, deg)
        assert np.all(one == 1)
    # zero denominator -> the reference panics ("Tried to invert zero")
    if n >= 2:
        sg2 = sg.copy()
        # choose sigma so that w + beta*sigma + gamma == 0 at (row 1, col 0)
        sg2[0, 1] = (-(int(w[0, 1]) + gamma)) * pow(beta, P - 2, P) % P
        with pytest.raises(ZeroDivisionError):
            gpu_pp(w, sg2, k, beta, gamma, deg)


# ----------------------------------------------------------------------------- GL_MEM_DEVICE entry points
def test_device_memory_entry_points(pb, oracle):
    """The same ABI with device pointers (what a device-resident pipeline / bench.py uses): NTT with a column
    stride larger than n, commit from device columns, cap/leaves/coeffs to device buffers, Merkle and hashing
    on device leaves."""
    import ctypes as C

    import torch

    N_ = pb._native
    L, ctx = N_.lib(), pb.default_context()
    dev = torch.device("cuda", 0)

    def to_dev(a):
        return torch.from_numpy(a.view(np.int64).copy()).to(dev)

    def to_np(t):
        return t.cpu().numpy().view(np.uint64)

    # --- gl_ntt, stride > n, forward then inverse with a coset
    B, log_n, stride = 5, 13, (1 << 13) + 24
    x = synth(0xD1, (B, stride))
    d = to_dev(x)
    N_.check(L.gl_ntt(ctx.h, C.c_void_p(d.data_ptr()), log_n, B, stride, 0, 0, 7, N_.MEM_DEVICE), ctx.h)
    ctx.synchronize()
    got = to_np(d)
    for b in range(B):
        assert np.array_equal(got[b, :1 << log_n], oracle.coset_fft(x[b, :1 << log_n], 7))
        assert np.array_equal(got[b, 1 << log_n:], x[b, 1 << log_n:])  # padding untouched
    N_.check(L.gl_ntt(ctx.h, C.c_void_p(d.data_ptr()), log_n, B, stride, 1, 0, 7, N_.MEM_DEVICE), ctx.h)
    ctx.synchronize()
    assert np.array_equal(to_np(d)[:, :1 << log_n], x[:, :1 << log_n])

    # --- gl_commit_create from device columns; outputs into device buffers
    B, log_n, r, h = 11, 9, 2, 3
    n, NN = 1 << log_n, 1 << (log_n + r)
    vals = synth(0xD2, (B, n))
    dv = to_dev(vals)
    hnd = N_.vp()
    N_.check(L.gl_commit_create(ctx.h, C.c_void_p(dv.data_ptr()), n, B, log_n, r, h, None, 0, N_.MEM_DEVICE,
                                C.byref(hnd)), ctx.h)
    o = oracle.Commit(vals, r, h)
    cap = torch.empty(4 << h, dtype=torch.int64, device=dev)
    leaves = torch.empty(NN * B, dtype=torch.int64, device=dev)
    coeffs = torch.empty(B * n, dtype=torch.int64, device=dev)
    digs = torch.empty(8 * (NN - (1 << h)), dtype=torch.int64, device=dev)
    N_.check(L.gl_commit_cap(hnd, C.c_void_p(cap.data_ptr()), N_.MEM_DEVICE), ctx.h)
    N_.check(L.gl_commit_leaves(hnd, 0, NN, C.c_void_p(leaves.data_ptr()), N_.MEM_DEVICE), ctx.h)
    N_.check(L.gl_commit_coeffs(hnd, C.c_void_p(coeffs.data_ptr()), N_.MEM_DEVICE), ctx.h)
    N_.check(L.gl_commit_digests(hnd, C.c_void_p(digs.data_ptr()), N_.MEM_DEVICE), ctx.h)
    ctx.synchronize()
    assert np.array_equal(to_np(cap).reshape(-1, 4), o.cap)
    assert np.array_equal(to_np(leaves).reshape(NN, B), o.leaves)
    assert np.array_equal(to_np(coeffs).reshape(B, n), o.coeffs)
    assert np.array_equal(to_np(digs).reshape(-1, 4), o.digests)
    assert L.gl_commit_num_polys(hnd) == B and L.gl_commit_leaf_width(hnd) == B
    assert L.gl_commit_degree_log(hnd) == log_n and L.gl_commit_rate_bits(hnd) == r and L.gl_commit_cap_height(hnd) == h

    # --- MerkleTree::new and hashing directly on the device leaves
    mh = N_.vp()
    N_.check(L.gl_merkle_build(ctx.h, C.c_void_p(leaves.data_ptr()), NN, B, h, N_.MEM_DEVICE, C.byref(mh)), ctx.h)
    cap2 = np.empty((1 << h, 4), dtype=np.uint64)
    N_.check(L.gl_merkle_cap(mh, N_.np_ptr(cap2), N_.MEM_HOST), ctx.h)
    assert np.array_equal(cap2, o.cap)
    hashes = torch.empty(NN * 4, dtype=torch.int64, device=dev)
    N_.check(L.gl_poseidon_hash_many(ctx.h, C.c_void_p(leaves.data_ptr()), NN, B, C.c_void_p(hashes.data_ptr()),
                                     N_.MEM_DEVICE), ctx.h)
    ctx.synchronize()
    assert np.array_equal(to_np(hashes).reshape(NN, 4), oracle.hash_many(o.leaves))
    L.gl_merkle_destroy(mh)
    L.gl_commit_destroy(hnd)


def test_profiling_phases_and_launch_count(pb):
    ctx = pb.Context(0)
    ctx.set_profiling(True)
    l0 = ctx.launch_count
    c = pb.PolynomialBatch.from_values(synth(0xD5, (9, 1 << 12)), 3, False, 4, ctx=ctx)
    ph = ctx.phase_ms()
    assert ctx.launch_count > l0
    assert ph["leaf_hash"][1] == 1 and ph["leaf_hash"][0] > 0 and ph["lde"][1] >= 1 and ph["intt"][1] >= 1
    ctx.reset_phases()
    assert ctx.phase_ms()["leaf_hash"] == (0.0, 0)
    c.close()
    ctx.close()


def test_cpp_host_layer_parity(pb, tmp_path):
    """The compiled-language host layer (include/plonky2_b200.hpp, mirroring the reference's Rust interface)
    driven by tests/cpp/host_parity.cpp: NTT vs naive evaluation, commitment vs oracle, shape errors,
    byte-identical FriProof accepted by the restated verifier."""
    import subprocess

    exe = str(tmp_path / "gl_host_parity")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "host_parity.cpp"),
                           "-L" + os.path.join(ROOT, "plonky2_b200"), "-lplonky2_b200",
                           "-L" + os.path.join(ROOT, "oracle"), "-lgl_oracle",
                           "-Wl,-rpath," + os.path.join(ROOT, "plonky2_b200"), "-Wl,-rpath," + os.path.join(ROOT, "oracle")])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "CPP HOST PARITY OK" in r.stdout, r.stdout + r.stderr


def test_randomised_shapes_against_oracle(pb, oracle):
    """Seeded sweep over random (columns, degree, rate, cap, salt, coeffs/values, non-canonical inputs) shapes:
    commitment (coefficients, cap, a leaf block, an opening) bit-exact vs the oracle."""
    rng = np.random.RandomState(20260922)
    for case in range(40):
        log_n = int(rng.randint(0, 12))
        r = int(rng.randint(0, 4))
        B = int(rng.randint(1, 40))
        h = int(rng.randint(0, min(log_n + r, 5) + 1))
        blinding = bool(rng.randint(0, 4) == 0)
        is_coeffs = bool(rng.randint(0, 2))
        n, N = 1 << log_n, 1 << (log_n + r)
        vals = synth(1000 + case, (B, n), canonical=bool(rng.randint(0, 2)))
        salt = synth(2000 + case, (4, N)) if blinding else None
        mk = pb.PolynomialBatch.from_coeffs if is_coeffs else pb.PolynomialBatch.from_values
        c = mk(vals, r, blinding, h, salt=salt)
        o = oracle.Commit(vals, r, h, salt=salt, is_coeffs=is_coeffs)
        tag = (case, B, log_n, r, h, blinding, is_coeffs)
        assert np.array_equal(c.polynomials, o.coeffs), tag
        assert np.array_equal(c.merkle_tree.cap.hashes, o.cap), tag
        lo = int(rng.randint(0, N))
        cnt = min(N - lo, 7)
        assert np.array_equal(c.merkle_tree.get_rows(lo, cnt), o.leaves[lo:lo + cnt]), tag
        lv, pt = c.merkle_tree.open_many([lo])
        assert np.array_equal(pt[0], oracle.merkle_prove(lo, N, h, o.digests)), tag
        c.close()


# ----------------------------------------------------------------------------- round-2 ABI: multi-destination iNTT, incremental commit
@pytest.mark.parametrize("log_n", [3, 10, 13])
def test_ntt_bcast_writes_every_destination(pb, oracle, log_n):
    """gl_ntt_bcast: the natural-order pass stores each coefficient to all destinations (peer mappings in production)."""
    import ctypes as C

    import torch

    from plonky2_b200 import _native as N

    n, B = 1 << log_n, 5
    x = synth(0x90 + log_n, (B, n), canonical=False)
    ctx = pb.default_context()
    src = torch.from_numpy(x.view(np.int64).copy()).cuda()
    dests = [torch.zeros((B + 2, n), dtype=torch.int64, device="cuda") for _ in range(3)]
    torch.cuda.synchronize()
    outs = (N.vp * 3)(*[N.vp(d[1:].data_ptr()) for d in dests])  # column b lands at row b + 1 of each destination
    N.check(N.lib().gl_ntt_bcast(ctx.h, N.vp(src.data_ptr()), n, log_n, B, 1, outs, 3, n), ctx.h)
    ctx.synchronize()
    want = np.stack([oracle.ifft(x[b]) for b in range(B)])
    for d in dests:
        got = d.cpu().numpy().view(np.uint64)
        assert np.array_equal(got[1:B + 1], want)
        assert not got[0].any() and not got[B + 1].any()
    assert np.array_equal(src.cpu().numpy().view(np.uint64), x)  # out of place: the input is untouched


@pytest.mark.parametrize("external", [False, True])
def test_incremental_commit_matches_oracle(pb, oracle, external):
    """gl_commit_begin / add_columns (any order, mixed kinds, host and device sources) / finish == from_values."""
    import ctypes as C

    import torch

    from plonky2_b200 import _native as N

    B, log_n, r, h = 13, 11, 3, 4
    n = 1 << log_n
    vals = synth(0xA1, (B, n))
    o = oracle.Commit(vals, r, h)
    coeffs = o.coeffs
    ctx = pb.default_context()
    L = N.lib()
    storage = torch.zeros((B, n), dtype=torch.int64, device="cuda") if external else None
    hnd = N.vp()
    N.check(L.gl_commit_begin(ctx.h, B, log_n, r, h, 0, 0, 1, N.vp(storage.data_ptr()) if external else None, C.byref(hnd)), ctx.h)
    try:
        cap = np.empty((1 << h, 4), dtype=np.uint64)
        assert L.gl_commit_cap(hnd, N.np_ptr(cap), N.MEM_HOST) != 0  # not finished yet
        # columns 8..12 as canonical coefficients from the device (in place when the storage is external)
        if external:
            storage[8:13].copy_(torch.from_numpy(coeffs[8:13].view(np.int64).copy()))
            src = storage[8:13]
        else:
            src = torch.from_numpy(coeffs[8:13].view(np.int64).copy()).cuda()
        torch.cuda.synchronize()
        N.check(L.gl_commit_add_columns(hnd, 8, 5, N.vp(src.data_ptr()), n, N.COLS_COEFFS_CANONICAL, N.MEM_DEVICE), ctx.h)
        # columns 0..2 as values from the host, 3..7 as (non-canonical) coefficients from the host
        N.check(L.gl_commit_add_columns(hnd, 0, 3, N.np_ptr(np.ascontiguousarray(vals[0:3])), n, N.COLS_VALUES, N.MEM_HOST), ctx.h)
        nc = coeffs[3:8].copy()
        nc[:, 0] = np.where(nc[:, 0] < np.uint64(2**32 - 1), nc[:, 0] + np.uint64(P), nc[:, 0])  # same residues, >= p
        N.check(L.gl_commit_add_columns(hnd, 3, 5, N.np_ptr(nc), n, N.COLS_COEFFS, N.MEM_HOST), ctx.h)
        assert L.gl_commit_add_columns(hnd, 12, 2, N.np_ptr(nc), n, N.COLS_COEFFS, N.MEM_HOST) != 0  # outside the batch
        N.check(L.gl_commit_finish(hnd, None, N.MEM_HOST), ctx.h)
        N.check(L.gl_commit_cap(hnd, N.np_ptr(cap), N.MEM_HOST), ctx.h)
        assert np.array_equal(cap, o.cap)
        got = np.empty((B, n), dtype=np.uint64)
        N.check(L.gl_commit_coeffs(hnd, N.np_ptr(got), N.MEM_HOST), ctx.h)
        assert np.array_equal(got, coeffs)
        rows = np.empty((16, B), dtype=np.uint64)
        N.check(L.gl_commit_leaves(hnd, 100, 16, N.np_ptr(rows), N.MEM_HOST), ctx.h)
        assert np.array_equal(rows, o.leaves[100:116])
        assert L.gl_commit_finish(hnd, None, N.MEM_HOST) != 0  # already finished
    finally:
        L.gl_commit_destroy(hnd)


def test_opening_set_one_call_matches_oracle(pb, oracle):
    """OpeningSet::new (proof.rs:313-351) through gl_openings: four commitments, zeta and g*zeta, one native call;
    every value equals the oracle's Horner evaluation of the oracle's coefficients."""
    log_n, r, h = 9, 3, 2
    n = 1 << log_n
    Bs = [9, 7, 6, 4]  # constants+sigmas, wires, zs+partial products(+lookup), quotient
    data = [synth(0xB0 + i, (B, n)) for i, B in enumerate(Bs)]
    batches = [pb.PolynomialBatch.from_values(d, r, False, h) for d in data[:3]] + [pb.PolynomialBatch.from_coeffs(data[3], r, False, h)]
    ocoeffs = [oracle.Commit(d, r, h).coeffs for d in data[:3]] + [data[3]]
    zeta = (int(synth(0xB7, (1,))[0]), int(synth(0xB8, (1,))[0]))
    g = pb.field.primitive_root_of_unity(log_n)
    gz = pb.field.ext_mul((g, 0), zeta)
    os_ = pb.OpeningSet.new(zeta, g, batches[0], batches[1], batches[2], batches[3], constants_range=range(0, 4),
                            sigmas_range=range(4, 9), zs_range=range(0, 2), partial_products_range=range(2, 5),
                            lookup_range=range(5, 6))

    def ev(co, z):
        return np.array([oracle.eval_poly_base_at_ext(c, z) for c in co], dtype=np.uint64)

    assert np.array_equal(os_.constants, ev(ocoeffs[0][0:4], zeta))
    assert np.array_equal(os_.plonk_sigmas, ev(ocoeffs[0][4:9], zeta))
    assert np.array_equal(os_.wires, ev(ocoeffs[1], zeta))
    assert np.array_equal(os_.plonk_zs, ev(ocoeffs[2][0:2], zeta))
    assert np.array_equal(os_.plonk_zs_next, ev(ocoeffs[2][0:2], gz))
    assert np.array_equal(os_.partial_products, ev(ocoeffs[2][2:5], zeta))
    assert np.array_equal(os_.lookup_zs, ev(ocoeffs[2][5:6], zeta))
    assert np.array_equal(os_.lookup_zs_next, ev(ocoeffs[2][5:6], gz))
    assert np.array_equal(os_.quotient_polys, ev(ocoeffs[3], zeta))
    zb, nb = os_.to_fri_openings()
    assert zb.shape == (9 + 7 + 5 + 4 + 1, 2) and nb.shape == (3, 2)
    so = pb.StarkOpeningSet.new(zeta, g, batches[1], None, batches[3])
    assert np.array_equal(so.local_values, ev(ocoeffs[1], zeta)) and np.array_equal(so.next_values, ev(ocoeffs[1], gz))
    assert np.array_equal(so.quotient_polys, ev(ocoeffs[3], zeta))
    for b in batches:
        b.close()


def test_zs_partial_products_commit_stays_on_device(pb, oracle):
    """prover.rs:220-254 chained on the device: wires (device) -> partial products / Z per challenge -> Z's first ->
    from_values, compared with the oracle's partial_products_and_zs + Commit on the host-assembled columns."""
    import torch

    from plonky2_b200.prover import commit_zs_partial_products

    R, log_n, deg, r, h = 20, 10, 8, 3, 4
    n = 1 << log_n
    w = synth(0xC1, (R, n))
    sg = synth(0xC2, (R, n))
    k = synth(0xC3, (R,))
    betas, gammas = [int(x) for x in synth(0xC4, (2,))], [int(x) for x in synth(0xC5, (2,))]
    wd = torch.from_numpy(w.view(np.int64).copy()).cuda()
    sd = torch.from_numpy(sg.view(np.int64).copy()).cuda()
    torch.cuda.synchronize()
    batch = commit_zs_partial_products(wd, sd, k, betas, gammas, deg, r, h)
    per = [oracle.partial_products_and_zs(w, sg, k, betas[i], gammas[i], deg) for i in range(2)]  # pp..., Z
    cols = np.concatenate([np.stack([p[-1] for p in per])] + [p[:-1] for p in per])                # Z's first
    o = oracle.Commit(cols, r, h)
    assert batch.num_polys == cols.shape[0] == 2 * 3
    assert np.array_equal(batch.merkle_tree.cap.hashes, o.cap)
    assert np.array_equal(batch.polynomials, o.coeffs)
    batch.close()


# ----------------------------------------------------------------------------- SURVEY 8(f) row 1: STARK quotient on the device
@pytest.mark.parametrize("log_n,r,num_alphas", [(5, 1, 1), (10, 1, 2), (13, 2, 2)])
def test_stark_quotient_fibonacci_matches_oracle(pb, oracle, log_n, r, num_alphas):
    """compute_quotient_polys (starky/src/prover.rs:488-668) for FibonacciStark: constraint program evaluated on the
    device over the trace LDE in place, bit for bit equal to the oracle's restatement; then the quotient commitment
    (prover.rs:391-421) equals from_coeffs of the oracle's chunks."""
    h = 2
    n = 1 << log_n
    stark = pb.FibonacciStark(n)
    trace = stark.generate_trace(7, 11)
    pi = [7, 11, int(trace[1, n - 1])]
    alphas = [int(x) for x in synth(0xE0 + log_n, (num_alphas,))]
    tc = pb.PolynomialBatch.from_values(trace, r, False, h)
    q = pb.compute_quotient_polys(stark, tc, pi, alphas)
    want = oracle.stark_quotient_fibonacci(oracle.Commit(trace, r, h), pi, alphas)
    got = q.cpu().numpy().view(np.uint64)
    assert np.array_equal(got, want)
    qc = pb.commit_quotient_polys(stark, q, log_n, r, h)
    oq = oracle.Commit(want, r, h, is_coeffs=True)   # quotient_degree_factor = 1: one chunk per challenge
    assert np.array_equal(qc.merkle_tree.cap.hashes, oq.cap)
    assert np.array_equal(qc.polynomials, want)
    tc.close()
    qc.close()


def test_stark_quotient_generic_program_higher_degree(pb):
    """The constraint program is generic: a toy STARK with products (declared constraint degree 4: quotient_degree_factor
    3, coset of size 4n, three chunks per challenge) checked by the verifier's identity (starky/src/verifier.rs:150-190)
    at a random point, and rejected ("Quotient has failed", prover.rs:396-401) when the trace is wrong."""
    from plonky2_b200 import NativeError
    from plonky2_b200.stark import Stark

    P_ = int(P)

    class CubicStark(Stark):
        COLUMNS, PUBLIC_INPUTS = 2, 1

        def eval(self, v, y):
            a, b = v.local(0), v.local(1)
            y.constraint_first_row(a - v.public_input(0))
            y.constraint_transition(v.next(0) - (a * a * b + 1))     # a' = a^2 b + 1
            y.constraint_transition(v.next(1) - (b + a * 3))          # b' = b + 3a
            y.constraint(a * 0)                                       # an unfiltered (trivially satisfied) constraint

        def constraint_degree(self):
            return 4   # an upper bound is allowed: the quotient then has zero top chunks, which trim_to_len checks

    log_n, r, h = 8, 2, 1
    n = 1 << log_n
    tr = np.empty((2, n), dtype=np.uint64)
    a, b = 5, 9
    for i in range(n):
        tr[0, i], tr[1, i] = a, b
        a, b = (a * a * b + 1) % P_, (b + 3 * a) % P_
    stark = CubicStark()
    assert stark.quotient_degree_factor() == 3
    alphas = [int(x) for x in synth(0xE9, (2,))]
    tc = pb.PolynomialBatch.from_values(tr, r, False, h)
    q = pb.compute_quotient_polys(stark, tc, [5], alphas).cpu().numpy().view(np.uint64)
    assert q.shape == (2, 4 * n) and not q[:, 3 * n:].any()
    coeffs = tc.polynomials
    z = int(synth(0xEA, (1,))[0])
    w = pb.field.primitive_root_of_unity(log_n)
    last = pow(w, P_ - 2, P_)

    def ev(c, x):
        acc = 0
        for v in c[::-1]:
            acc = (acc * x + int(v)) % P_
        return acc

    la, lb = ev(coeffs[0], z), ev(coeffs[1], z)
    na, nb = ev(coeffs[0], z * w % P_), ev(coeffs[1], z * w % P_)
    zh = (pow(z, n, P_) - 1) % P_
    l_first = zh * pow(n * (z - 1) % P_, P_ - 2, P_) % P_
    z_last = (z - last) % P_
    cons = [(la - 5) * l_first, (na - (la * la * lb + 1)) * z_last, (nb - (lb + 3 * la)) * z_last, 0]
    for j, al in enumerate(alphas):
        acc = 0
        for c in cons:
            acc = (acc * al + c) % P_
        assert acc == zh * ev(q[j], z) % P_
    qc = pb.commit_quotient_polys(stark, pb.compute_quotient_polys(stark, tc, [5], alphas), log_n, r, h)
    assert qc.num_polys == 6 and np.array_equal(qc.polynomials, q[:, :3 * n].reshape(6, n))   # 3 chunks of n per challenge
    qc.close()
    tc.close()
    tr[1, n // 2] ^= np.uint64(1)   # one wrong cell: the vanishing polynomial is no longer divisible by Z_H
    tb = pb.PolynomialBatch.from_values(tr, r, False, h)
    with pytest.raises(NativeError, match="Quotient has failed"):
        pb.compute_quotient_polys(stark, tb, [5], alphas)
    tb.close()


def test_stark_prove_pipeline_on_device(pb, oracle):
    """The starky prover's commitment path end to end on the device (starky/src/prover.rs:83-94,391-470): trace
    commitment -> quotient polynomials from the LDE in place -> quotient commitment -> StarkOpeningSet (one call) ->
    prove_openings; the FRI proof is accepted by the restated verifier with exactly those openings."""
    log_n, r, h = 10, 1, 4
    n = 1 << log_n
    stark = pb.FibonacciStark(n)
    trace = stark.generate_trace(1, 1)
    pi = [1, 1, int(trace[1, n - 1])]
    cfg = pb.starky_standard_fast_fri_config()
    params = cfg.fri_params(log_n, False)
    ch, och = pb.Challenger(), oracle.Challenger()
    tc = pb.PolynomialBatch.from_values(trace, r, False, h)
    ch.observe_cap(tc.merkle_tree.cap)
    alphas = ch.get_n_challenges(2)
    q = pb.compute_quotient_polys(stark, tc, pi, alphas)
    qc = pb.commit_quotient_polys(stark, q, log_n, r, h)
    ch.observe_cap(qc.merkle_tree.cap)
    zeta = ch.get_extension_challenge()
    g = pb.field.primitive_root_of_unity(log_n)
    openings = pb.StarkOpeningSet.new(zeta, g, tc, None, qc)
    zb, nb = openings.to_fri_openings()
    for batch in (zb, nb):
        ch.observe_elements(batch.reshape(-1))
    gz = pb.field.ext_mul((g, 0), zeta)
    inst = pb.FriInstanceInfo([pb.FriOracleInfo(2, False), pb.FriOracleInfo(2, False)],
                              [pb.FriBatchInfo(zeta, [pb.FriPolynomialInfo(0, 0), pb.FriPolynomialInfo(0, 1),
                                                      pb.FriPolynomialInfo(1, 0), pb.FriPolynomialInfo(1, 1)]),
                               pb.FriBatchInfo(gz, [pb.FriPolynomialInfo(0, 0), pb.FriPolynomialInfo(0, 1)])])
    # the oracle verifier replays the transcript from the same state
    och.observe_cap(tc.merkle_tree.cap.hashes)
    assert och.get_n_challenges(2) == alphas
    och.observe_cap(qc.merkle_tree.cap.hashes)
    assert och.get_extension_challenge() == zeta
    for batch in (zb, nb):
        och.observe_elements(batch.reshape(-1))
    proof = pb.prove_openings(inst, [tc, qc], ch, params)
    obatches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in inst.batches]
    oparams = oracle.make_params(r, h, cfg.proof_of_work_bits, cfg.num_query_rounds, params.reduction_arity_bits)
    rc = oracle.verify_fri_proof([tc.merkle_tree.cap.hashes, qc.merkle_tree.cap.hashes], [2, 2], [2, 2], obatches,
                                 np.concatenate([zb.reshape(-1), nb.reshape(-1)]), log_n, och, oparams, proof.to_bytes())
    assert rc == 0
    # the verifier's quotient identity at zeta (starky/src/verifier.rs:150-190) with the opened values, in F_{p^2}
    E = pb.field
    lv, nv, qv = [tuple(int(x) for x in v) for v in openings.local_values], [tuple(int(x) for x in v) for v in openings.next_values], \
        [tuple(int(x) for x in v) for v in openings.quotient_polys]
    zn = E.ext_pow(zeta, n)
    zh = E.ext_sub(zn, (1, 0))
    last = pow(g, int(P) - 2, int(P))
    l_first = E.ext_mul(zh, E.ext_inverse(E.ext_mul((n, 0), E.ext_sub(zeta, (1, 0)))))
    l_last = E.ext_mul(E.ext_mul(zh, (last, 0)), E.ext_inverse(E.ext_mul((n, 0), E.ext_sub(zeta, (last, 0)))))
    z_last = E.ext_sub(zeta, (last, 0))
    cons = [E.ext_mul(E.ext_sub(lv[0], (pi[0], 0)), l_first), E.ext_mul(E.ext_sub(lv[1], (pi[1], 0)), l_first),
            E.ext_mul(E.ext_sub(lv[1], (pi[2], 0)), l_last), E.ext_mul(E.ext_sub(nv[0], lv[1]), z_last),
            E.ext_mul(E.ext_sub(E.ext_sub(nv[1], lv[0]), lv[1]), z_last)]
    for j, al in enumerate(alphas):
        acc = (0, 0)
        for c in cons:
            acc = E.ext_add(E.ext_mul(acc, (al, 0)), c)
        assert acc == E.ext_mul(zh, qv[j])
    tc.close()
    qc.close()


@pytest.mark.parametrize("routed,qdf,log_n,rows", [(12, 4, 8, [(10, 40, 60)]), (80, 8, 10, [(3, 300, 500), (600, 700, 900)]),
                                                   (6, 2, 6, [(5, 5, 5)])])
def test_lookup_polys_match_oracle(pb, oracle, routed, qdf, log_n, rows):
    """compute_lookup_polys (plonk/prover.rs:458-577): RE + partial Sum/LDC columns vs the oracle's literal restatement,
    one and two LookupWires, degenerate ranges; a zero denominator is reported like the reference's panic."""
    from plonky2_b200.prover import compute_all_lookup_polys, compute_lookup_polys

    n = 1 << log_n
    wires = synth(0xF8 + log_n, (routed, n))
    deltas = [int(x) for x in synth(0xF9, (8,))]
    got = compute_lookup_polys(wires, routed, qdf, deltas[:4], rows)
    want = oracle.lookup_polys(wires, routed, qdf, deltas[:4], rows)
    assert got.shape == want.shape and np.array_equal(got, want)
    both = compute_all_lookup_polys(wires, routed, qdf, deltas, rows, 2)
    assert np.array_equal(both[:len(want)], want)
    assert np.array_equal(both[len(want):], oracle.lookup_polys(wires, routed, qdf, deltas[4:], rows))
    # alpha = inp + A*out on one looked slot -> "Tried to invert zero"
    row = rows[0][2]
    bad = list(deltas[:4])
    bad[2] = (int(wires[0, row]) + bad[0] * int(wires[1, row])) % int(P)
    with pytest.raises(ZeroDivisionError):
        compute_lookup_polys(wires, routed, qdf, bad, rows)


@pytest.mark.parametrize("shards", [2, 8])
def test_fri_round_trees_row_block_sharded(pb, shards):
    """gl_fri_commit_round_sharded: every shard hashes its own block of a round's leaves; the shards' cap entries in
    shard order are the unsharded cap, round after round (values and folds are replicated)."""
    import ctypes as C

    from plonky2_b200 import _native as N

    log_n, r, h = 10, 2, 4
    n = 1 << log_n
    coeffs = synth(0xFA, (n, 2))
    betas = synth(0xFB, (3, 2))
    ctx = pb.default_context()
    L = N.lib()

    def begin():
        f = N.vp()
        N.check(L.gl_fri_begin_from_coeffs(ctx.h, N.np_ptr(coeffs.reshape(-1)), log_n, r, h, C.byref(f)), ctx.h)
        return f

    ref = begin()
    states = [begin() for _ in range(shards)]
    try:
        for rnd, arity_bits in enumerate([3, 2, 2]):   # 4096 -> 512 -> 128 -> 32 values: leaves 512, 128, 32
            want = np.empty(4 << h, dtype=np.uint64)
            N.check(L.gl_fri_commit_round(ref, arity_bits, N.np_ptr(want)), ctx.h)
            got = []
            for g, f in enumerate(states):
                loc = np.empty((4 << h) // shards, dtype=np.uint64)
                N.check(L.gl_fri_commit_round_sharded(f, arity_bits, g, shards, N.np_ptr(loc)), ctx.h)
                got.append(loc)
            assert np.array_equal(np.concatenate(got), want), rnd
            for f in [ref] + states:
                N.check(L.gl_fri_fold(f, N.np_ptr(np.ascontiguousarray(betas[rnd]))), ctx.h)
        out = [np.empty(2 * 16, dtype=np.uint64) for _ in range(1 + shards)]
        for f, o in zip([ref] + states, out):
            ln = C.c_size_t()
            N.check(L.gl_fri_final_poly(f, N.np_ptr(o), o.size, C.byref(ln)), ctx.h)
            assert ln.value == 32 >> r
        assert all(np.array_equal(o[:16], out[0][:16]) for o in out)
    finally:
        for f in [ref] + states:
            L.gl_fri_destroy(f)


def _fri_setup(pb, log_n=9, r=2, h=3, Bs=(5, 3)):
    n = 1 << log_n
    data = [synth(0x1A0 + i, (B, n)) for i, B in enumerate(Bs)]
    zeta = (int(synth(0x1A8, (1,))[0]), int(synth(0x1A9, (1,))[0]))
    gz = pb.field.ext_mul(zeta, (pb.field.primitive_root_of_unity(log_n), 0))
    inst = pb.FriInstanceInfo([pb.FriOracleInfo(B, False) for B in Bs],
                              [pb.FriBatchInfo(zeta, [pb.FriPolynomialInfo(o, i) for o, B in enumerate(Bs) for i in range(B)]),
                               pb.FriBatchInfo(gz, [pb.FriPolynomialInfo(0, 1), pb.FriPolynomialInfo(1, 0)])])
    cfg = pb.FriConfig(r, h, 4, ("Fixed", [3, 2]), 9)
    params = pb.FriParams(cfg, False, log_n, [3, 2])
    return data, inst, params, zeta, gz


def _openings_for(pb, inst, batches):
    req = []
    for b in inst.batches:
        for p in b.polynomials:
            req.append((batches[p.oracle_index], b.point))
    ev = pb.eval_commitments(req)
    out, k = [], 0
    for b in inst.batches:
        vals = []
        for p in b.polynomials:
            vals.append(ev[k][p.polynomial_index])
            k += 1
        out.append(np.array(vals, dtype=np.uint64))
    return out


def test_fri_value_domain_begin_gives_the_same_proof(pb):
    """gl_fri_begin_values (composition from the LDE rows + the openings) yields the codeword of gl_fri_begin: the
    whole FRI proof is byte-identical."""
    from plonky2_b200 import fri as F

    data, inst, params, zeta, gz = _fri_setup(pb)
    batches = [pb.PolynomialBatch.from_values(d, params.config.rate_bits, False, params.config.cap_height) for d in data]
    opened = _openings_for(pb, inst, batches)
    ch1, ch2 = pb.Challenger(), pb.Challenger()
    for ch in (ch1, ch2):
        for b in batches:
            ch.observe_cap(b.merkle_tree.cap)
    want = pb.prove_openings(inst, batches, ch1, params).to_bytes()
    st = F._begin_values(inst, batches, ch2.get_extension_challenge(), opened, params)
    try:
        caps, final = F.fri_committed_trees(st, ch2, params)
        poww = F.fri_proof_of_work(ch2, params.config, st.ctx)
        rounds, _ = F.fri_prover_query_rounds(batches, st, ch2, params.lde_size(), params)
        assert F.FriProof(caps, rounds, final, poww).to_bytes() == want
    finally:
        st.close()
    for b in batches:
        b.close()


@pytest.mark.parametrize("shards", [2, 8])
def test_fri_value_domain_row_block_sharded_rounds(pb, shards):
    """With row-block sharded commitments the value-domain state is rank-local: per round the shards' cap entries in
    shard order equal the unsharded cap, the gathered last codeword interpolates to the same final polynomial."""
    import ctypes as C

    from plonky2_b200 import _native as N
    from plonky2_b200 import fri as F

    data, inst, params, zeta, gz = _fri_setup(pb)
    r, h = params.config.rate_bits, params.config.cap_height
    whole = [pb.PolynomialBatch.from_values(d, r, False, h) for d in data]
    opened = _openings_for(pb, inst, whole)
    alpha = (int(synth(0x1AA, (1,))[0]), int(synth(0x1AB, (1,))[0]))
    ref = F._begin_values(inst, whole, alpha, opened, params)
    parts = [[pb.PolynomialBatch.from_values(d, r, False, h, shard=(g, shards)) for d in data] for g in range(shards)]
    states = [F._begin_values(inst, parts[g], alpha, opened, params) for g in range(shards)]
    L, ctx = N.lib(), ref.ctx
    betas = synth(0x1AC, (2, 2))
    try:
        for rnd, ab in enumerate(params.reduction_arity_bits):
            want = np.empty(4 << h, dtype=np.uint64)
            N.check(L.gl_fri_commit_round(ref.h, ab, N.np_ptr(want)), ctx.h)
            got = []
            for st in states:
                loc = np.empty((4 << h) // shards, dtype=np.uint64)
                N.check(L.gl_fri_commit_round(st.h, ab, N.np_ptr(loc)), ctx.h)
                got.append(loc)
            assert np.array_equal(np.concatenate(got), want), rnd
            for st in [ref] + states:
                N.check(L.gl_fri_fold(st.h, N.np_ptr(np.ascontiguousarray(betas[rnd]))), ctx.h)
        log_last = params.lde_bits() - params.total_arities()
        vals = []
        for st in states:
            loc = np.empty(2 * ((1 << log_last) // shards), dtype=np.uint64)
            ln = C.c_size_t()
            N.check(L.gl_fri_values_local(st.h, N.np_ptr(loc), loc.size, C.byref(ln)), ctx.h)
            assert ln.value == (1 << log_last) // shards
            vals.append(loc)
        shift = pow(pb.field.coset_shift(), 1 << params.total_arities(), int(P))
        coeffs = F._final_poly_from_values(np.concatenate(vals).reshape(-1, 2), log_last, shift, r, ctx)
        buf = np.empty(2 * (1 << log_last), dtype=np.uint64)
        ln = C.c_size_t()
        N.check(L.gl_fri_final_poly(ref.h, N.np_ptr(buf), buf.size, C.byref(ln)), ctx.h)
        assert np.array_equal(coeffs.reshape(-1), buf[:2 * ln.value])
    finally:
        for st in [ref] + states:
            st.close()
        for b in whole + [x for p in parts for x in p]:
            b.close()
