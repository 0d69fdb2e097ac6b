"""Fiat-Shamir duplex challenger on the host (plonky2/src/iop/challenger.rs:16-153).
Inherently sequential (one permutation per <= 8 absorbed elements), so it stays on the CPU exactly as
in the reference; the permutation itself is gl_poseidon_permute_host (same source as the device one)."""
from .field import ORDER
from .hash import SPONGE_RATE, PoseidonPermutation


class Challenger:
    def __init__(self):
        self.sponge_state = PoseidonPermutation()
        self.input_buffer = []
        self.output_buffer = []

    def clone(self):
        c = Challenger()
        c.sponge_state = self.sponge_state.copy()
        c.input_buffer = list(self.input_buffer)
        c.output_buffer = list(self.output_buffer)
        return c

    def observe_element(self, element):
        self.output_buffer.clear()
        self.input_buffer.append(int(element) % ORDER)
        if len(self.input_buffer) == SPONGE_RATE:
            self.duplexing()

    def observe_elements(self, elements):
        for e in elements:
            self.observe_element(e)

    def observe_extension_element(self, element):
        self.observe_elements(element)

    def observe_extension_elements(self, elements):
        for e in elements:
            self.observe_extension_element(e)

    def observe_hash(self, h):
        self.observe_elements([int(x) for x in h])

    def observe_cap(self, cap):
        for h in cap.hashes:
            self.observe_hash(h)

    def observe_openings(self, openings):
        """observe_openings (plonky2/src/fri/challenges.rs:19-26): every batch's F_{p^2} values in order;
        `openings` is a list of (k, 2) arrays (OpeningSet / StarkOpeningSet .to_fri_openings())."""
        for batch in openings:
            self.observe_elements([int(x) for x in batch.reshape(-1)])

    def get_challenge(self):
        if self.input_buffer or not self.output_buffer:
            self.duplexing()
        return self.output_buffer.pop()

    def get_n_challenges(self, n):
        return [self.get_challenge() for _ in range(n)]

    def get_hash(self):
        return [self.get_challenge() for _ in range(4)]

    def get_extension_challenge(self):
        c = self.get_n_challenges(2)
        return (c[0], c[1])

    def get_n_extension_challenges(self, n):
        return [self.get_extension_challenge() for _ in range(n)]

    def duplexing(self):
        assert len(self.input_buffer) <= SPONGE_RATE
        self.sponge_state.set_from_iter(self.input_buffer, 0)
        self.input_buffer = []
        self.sponge_state.permute()
        self.output_buffer = [int(x) for x in self.sponge_state.squeeze()]

    def compact(self):
        if self.input_buffer:
            self.duplexing()
        self.output_buffer = []
        return self.sponge_state
