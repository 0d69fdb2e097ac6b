"""plonky2_b200 -- B200-native (sm_100a CUDA) implementation of the plonky2 prover hot path:
Goldilocks NTT / coset-LDE, Poseidon Merkle commitment and the FRI commit phase, behind the C ABI in
include/plonky2_b200.h. This package is the host-side mirror of the reference's interface for that
path (same names, argument meaning and error behaviour); see DESIGN.md and INTEGRATION.md."""
from . import field  # noqa: F401
from ._native import Context, NativeError, ShapeError, default_context  # noqa: F401
from .challenger import Challenger  # noqa: F401
from .fft import (coset_fft, coset_fft_with_options, coset_ifft, fft, fft_with_options, ifft,  # noqa: F401
                  ifft_with_options, lde, lde_onto_coset)
from .fri import (FriBatchInfo, FriConfig, FriInstanceInfo, FriOracleInfo, FriParams,  # noqa: F401
                  FriPolynomialInfo, FriProof, prove_openings, standard_recursion_fri_config,
                  starky_standard_fast_fri_config)
from .hash import (MerkleCap, MerkleProof, MerkleTree, PoseidonHash, PoseidonPermutation,  # noqa: F401
                   verify_merkle_proof_to_cap)
from .polynomial_batch import SALT_SIZE, PolynomialBatch  # noqa: F401
from .proof import OpeningSet, StarkOpeningSet, StarkProof, StarkProofWithPublicInputs, eval_commitments  # noqa: F401
from .stark import (Column, FibonacciStark, Filter, Lookup, PermutationStark, Stark, StarkConfig,  # noqa: F401
                    commit_quotient_polys, compute_quotient_polys)
from . import plonk  # noqa: F401  (plonk.compute_quotient_polys: the plonky2 circuit quotient)
from .batch_merkle_tree import (BatchMerkleTree, compress_merkle_proofs, decompress_merkle_proofs,  # noqa: F401
                                verify_batch_merkle_proof_to_cap)
from .batch_fri import BatchFriOracle, batch_prove_openings  # noqa: F401
