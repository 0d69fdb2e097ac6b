"""OpeningSet / StarkOpeningSet mirroring plonky2/src/plonk/proof.rs:300-351 and starky/src/proof.rs:205-290: the
purported values of every committed polynomial at zeta (and g*zeta), computed on the device from the coefficient
matrices behind the PolynomialBatch handles in ONE native call (gl_openings): no coefficient D2H."""
import ctypes as C
from dataclasses import dataclass, field as dc_field

import numpy as np

from . import _native as N
from . import field as F


def eval_commitments(requests):
    """requests: [(PolynomialBatch, point)], point in F_{p^2} as (c0, c1). Returns a list of (num_polys, 2) uint64 arrays
    (eval_commitment, proof.rs:323-328), all from one gl_openings call."""
    if not requests:
        return []
    ctx = requests[0][0].ctx
    pts, idx = [], []
    for _, z in requests:
        z = (int(z[0]) % F.ORDER, int(z[1]) % F.ORDER)
        if z not in pts:
            pts.append(z)
        idx.append(pts.index(z))
    handles = (N.vp * len(requests))(*[b.h for b, _ in requests])
    pidx = np.array(idx, dtype=np.uint32)
    points = np.array(pts, dtype=np.uint64).reshape(-1)
    total = sum(b.num_polys for b, _ in requests)
    out = np.empty((total, 2), dtype=np.uint64)
    N.check(N.lib().gl_openings(ctx.h, handles, pidx.ctypes.data_as(N.u32p), len(requests), N.np_ptr(points), len(pts),
                                N.np_ptr(out), N.MEM_HOST), ctx.h)
    res, off = [], 0
    for b, _ in requests:
        res.append(out[off:off + b.num_polys].copy())
        off += b.num_polys
    return res


@dataclass
class OpeningSet:
    """OpeningSet<F, D> (proof.rs:300-311); every field is an (k, 2) uint64 array of F_{p^2} values."""
    constants: np.ndarray
    plonk_sigmas: np.ndarray
    wires: np.ndarray
    plonk_zs: np.ndarray
    plonk_zs_next: np.ndarray
    partial_products: np.ndarray
    quotient_polys: np.ndarray
    lookup_zs: np.ndarray
    lookup_zs_next: np.ndarray

    @classmethod
    def new(cls, zeta, g, constants_sigmas_commitment, wires_commitment, zs_partial_products_lookup_commitment,
            quotient_polys_commitment, constants_range, sigmas_range, zs_range, partial_products_range, lookup_range):
        """OpeningSet::new (proof.rs:313-351). The *_range arguments are the CommonCircuitData ranges
        (circuit_data.rs constants_range() ... lookup_range()) as Python ranges/slices."""
        g_zeta = F.ext_mul((int(g[0]), int(g[1])) if isinstance(g, (tuple, list, np.ndarray)) else (int(g), 0), zeta)
        cs, zs, zs_next, quot, wires = eval_commitments([
            (constants_sigmas_commitment, zeta), (zs_partial_products_lookup_commitment, zeta),
            (zs_partial_products_lookup_commitment, g_zeta), (quotient_polys_commitment, zeta), (wires_commitment, zeta)])

        def take(a, r):
            return a[r.start:r.stop] if isinstance(r, (range, slice)) else a[list(r)]

        return cls(constants=take(cs, constants_range), plonk_sigmas=take(cs, sigmas_range), wires=wires,
                   plonk_zs=take(zs, zs_range), plonk_zs_next=take(zs_next, zs_range),
                   partial_products=take(zs, partial_products_range), quotient_polys=quot,
                   lookup_zs=take(zs, lookup_range), lookup_zs_next=take(zs_next, lookup_range))

    def to_fri_openings(self):
        """to_fri_openings (proof.rs:352-400): [zeta batch values, zeta_next batch values] in the FRI instance's order."""
        has_lookup = len(self.lookup_zs) > 0
        zeta_batch = [self.constants, self.plonk_sigmas, self.wires, self.plonk_zs, self.partial_products, self.quotient_polys]
        if has_lookup:
            zeta_batch.append(self.lookup_zs)
        next_batch = [self.plonk_zs_next] + ([self.lookup_zs_next] if has_lookup else [])
        return [np.concatenate(zeta_batch), np.concatenate(next_batch)]


@dataclass
class StarkOpeningSet:
    """StarkOpeningSet<F, D> (starky/src/proof.rs:205-219) without cross-table lookups."""
    local_values: np.ndarray
    next_values: np.ndarray
    auxiliary_polys: np.ndarray = None
    auxiliary_polys_next: np.ndarray = None
    quotient_polys: np.ndarray = None

    @classmethod
    def new(cls, zeta, g, trace_commitment, auxiliary_polys_commitment=None, quotient_commitment=None):
        """StarkOpeningSet::new (starky/src/proof.rs:221-260): trace (and auxiliary) polynomials at zeta and g*zeta,
        quotient polynomials at zeta."""
        g_zeta = F.ext_mul((int(g), 0), zeta)
        req = [(trace_commitment, zeta), (trace_commitment, g_zeta)]
        if auxiliary_polys_commitment is not None:
            req += [(auxiliary_polys_commitment, zeta), (auxiliary_polys_commitment, g_zeta)]
        if quotient_commitment is not None:
            req.append((quotient_commitment, zeta))
        res = eval_commitments(req)
        k = 2
        aux = aux_next = quot = None
        if auxiliary_polys_commitment is not None:
            aux, aux_next = res[k], res[k + 1]
            k += 2
        if quotient_commitment is not None:
            quot = res[k]
        return cls(res[0], res[1], aux, aux_next, quot)

    def to_fri_openings(self):
        """to_fri_openings (starky/src/proof.rs:263-290), no CTLs: [zeta batch, zeta_next batch]."""
        zeta_batch = [self.local_values]
        if self.auxiliary_polys is not None:
            zeta_batch.append(self.auxiliary_polys)
        if self.quotient_polys is not None:
            zeta_batch.append(self.quotient_polys)
        next_batch = [self.next_values] + ([self.auxiliary_polys_next] if self.auxiliary_polys_next is not None else [])
        return [np.concatenate(zeta_batch), np.concatenate(next_batch)]


@dataclass
class StarkProof:
    """StarkProof<F, C, D> (starky/src/proof.rs:27-40) without cross-table lookups. The caps are MerkleCaps (None where
    the STARK has no auxiliary or no quotient polynomials); opening_proof is a FriProof, whose to_bytes() is
    write_fri_proof. The reference serialises a STARK proof with serde only, so there is no byte format here."""
    trace_cap: object
    auxiliary_polys_cap: object
    quotient_polys_cap: object
    openings: StarkOpeningSet
    opening_proof: object


@dataclass
class StarkProofWithPublicInputs:
    """StarkProofWithPublicInputs (starky/src/proof.rs:150-158)."""
    proof: StarkProof
    public_inputs: list
