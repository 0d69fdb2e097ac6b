"""CPU-side checks of the product: the C-ABI library loads and exports every symbol the header
declares, fails loudly without a GPU, and the host-side mirror logic (transcript, parameters,
serialisation) agrees with the oracle. No GPU compute here."""
import os
import re

import numpy as np
import pytest

from conftest import P, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    import plonky2_b200.build as b

    b.build()
    from plonky2_b200 import _native

    return _native


def test_library_exports_every_declared_symbol(native):
    hdr = open(os.path.join(ROOT, "include", "plonky2_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(gl_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 35
    L = native.lib()
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, missing
    assert set(native.EXPORTS) <= declared


def test_no_cpu_fallback_without_gpu(native):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(native.NativeError) as e:
        native.Context(0)
    assert "no CPU fallback" in str(e.value)
    import plonky2_b200 as pb

    with pytest.raises(native.NativeError):
        pb.fft(np.arange(8, dtype=np.uint64))
    with pytest.raises(native.NativeError):
        pb.PolynomialBatch.from_values(np.zeros((2, 8), dtype=np.uint64), 1, False, 0)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "plonky2_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "gl_oracle" not in txt and "oracle_lib" not in txt and "glo_" not in txt, f


def test_host_permutation_matches_kats(native):
    import json

    kat = json.load(open(os.path.join(ROOT, "tests", "golden", "poseidon_kat.json")))
    for v in kat["vectors"]:
        s = np.array([int(x) for x in v["input"]], dtype=np.uint64)
        native.lib().gl_poseidon_permute_host(native.np_ptr(s))
        assert s.tolist() == [int(x) for x in v["output"]]


def test_challenger_matches_oracle(native, oracle):
    from plonky2_b200 import Challenger, MerkleCap

    ch, och = Challenger(), oracle.Challenger()
    xs = synth(0x91, (37,), canonical=False)
    ch.observe_elements([int(x) for x in xs[:5]])
    och.observe_elements(xs[:5])
    assert ch.get_challenge() == och.get_challenge()
    ch.observe_elements([int(x) for x in xs[5:30]])
    och.observe_elements(xs[5:30])
    assert ch.get_n_challenges(11) == och.get_n_challenges(11)
    cap = synth(0x92, (16, 4))
    ch.observe_cap(MerkleCap(cap))
    och.observe_cap(cap)
    assert ch.get_extension_challenge() == och.get_extension_challenge()
    st, ib = och.state()
    assert [int(x) for x in ch.sponge_state.state] == st.tolist()
    c2 = ch.clone()
    ch.observe_element(7)
    assert c2.get_challenge() == och.get_challenge()


def test_field_helpers(oracle):
    from plonky2_b200 import field as F

    L = oracle.lib()
    for k in range(0, 33):
        assert F.primitive_root_of_unity(k) == L.glo_primitive_root_of_unity(k)
        assert F.inverse_2exp(k) == L.glo_inverse_2exp(k)
    assert F.coset_shift() == L.glo_coset_shift()
    a, b = (123456789123456789 % P, 987654321987654321 % P), (5, P - 3)
    out = np.zeros(2, dtype=np.uint64)
    L.glo_ext2_mul(oracle.ptr(np.array(a, dtype=np.uint64)), oracle.ptr(np.array(b, dtype=np.uint64)),
                   oracle.ptr(out))
    assert F.ext_mul(a, b) == tuple(out.tolist())
    assert F.ext_mul(F.ext_inverse(a), a) == (1, 0)
    assert F.reverse_bits(0b01011, 5) == 0b11010
    with pytest.raises(ValueError):
        F.log2_strict(12)


def test_fri_params_and_reduction_strategy():
    from plonky2_b200.fri import (reduction_arity_bits, standard_recursion_fri_config,
                                  starky_standard_fast_fri_config)

    cfg = standard_recursion_fri_config()
    # SURVEY section 8: cfg4 arities [4,4,4] at n=2^14 and [4,4] at 2^12
    assert cfg.fri_params(14, False).reduction_arity_bits == [4, 4, 4]
    assert cfg.fri_params(12, False).reduction_arity_bits == [4, 4]
    assert cfg.fri_params(14, False).final_poly_len() == 4
    assert starky_standard_fast_fri_config().fri_params(24, False).reduction_arity_bits == [4, 4, 4, 4, 4]
    assert reduction_arity_bits(("Fixed", [3, 2]), 10, 1, 0, 5) == [3, 2]


def test_fri_proof_serialisation_layout():
    from plonky2_b200.fri import FriInitialTreeProof, FriProof, FriQueryRound, FriQueryStep
    from plonky2_b200.hash import MerkleCap

    cap = MerkleCap(np.arange(8, dtype=np.uint64).reshape(2, 4))
    init = FriInitialTreeProof([(np.array([9, 10, 11], dtype=np.uint64), np.arange(8, dtype=np.uint64).reshape(2, 4))])
    st = FriQueryStep(np.array([[1, 2], [3, 4]], dtype=np.uint64), np.arange(4, dtype=np.uint64).reshape(1, 4))
    pr = FriProof([cap], [FriQueryRound(init, [st])], np.array([[5, 6]], dtype=np.uint64), 77)
    b = pr.to_bytes()
    # 8 cap words + (3 leaf + 1 byte + 8 sib) + (4 evals + 1 byte + 4 sib) + 2 final + 1 pow
    assert len(b) == 8 * (8 + 3 + 8 + 4 + 4 + 2 + 1) + 2
    assert b[:8] == (0).to_bytes(8, "little") and b[-8:] == (77).to_bytes(8, "little")
    assert b[8 * 8 + 3 * 8] == 2


def test_cpp_host_layer_compiles_and_fails_loudly_without_gpu(native, oracle, tmp_path):
    """include/plonky2_b200.hpp (the C++ mirror of the reference's Rust interface) builds against the C ABI;
    without a GPU the program must abort with the library's "no CPU fallback" error, not compute anything."""
    import subprocess

    import torch

    exe = str(tmp_path / "gl_host_parity_cpu")
    subprocess.check_call(["g++", "-std=c++17", "-O0", "-Wall", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "host_parity.cpp"),
                           "-L" + os.path.join(ROOT, "plonky2_b200"), "-lplonky2_b200",
                           "-L" + os.path.join(ROOT, "oracle"), "-lgl_oracle",
                           "-Wl,-rpath," + os.path.join(ROOT, "plonky2_b200"), "-Wl,-rpath," + os.path.join(ROOT, "oracle")])
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
