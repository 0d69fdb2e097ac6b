"""Phase times of stark.prove on one GPU: a range-check STARK with 16 looking columns (one lookup, constraint degree 3,
standard_fast_config, 2 challenges) at 2^20 and 2^22 rows. CUDA events on the library's stream time the helper columns,
the auxiliary commitment, the quotient (and its commitment), the openings, the FRI proof and the whole prove, after one
warm-up proof per size. The proof is checked with the restated verifier (tests/test_stark_prove.py) before any time is
printed. The card's name and power limit are read in the same run. No CPU comparison is made: the CPU twin in the tests
is a checker, not a tuned CPU prover.

    python tools/stark_prove_timing.py [--log-n 20 22] [--reps 3] [--out timings.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log-n", type=int, nargs="+", default=[20, 22])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    import oracle_lib
    import plonky2_b200 as pb
    from plonky2_b200 import stark as S
    from test_stark_prove import RangeCheckStark, fast_config, verify_stark_proof

    ctx = pb.default_context(0)
    stream = torch.cuda.ExternalStream(ctx.stream, device="cuda:0")
    name, limit = card()
    results = []
    for log_n in args.log_n:
        st = RangeCheckStark(1 << log_n, 3, num_looking=16, second_lookup=False)
        cfg = fast_config()
        tr = st.generate_trace(7)
        pis = [st.num_rows - 1]
        # the phases, each bracketed by events on the library's stream (every call is ordered on it)
        times = {}
        orig = {k: getattr(S, k) for k in ("lookup_helper_columns", "_commit_values", "compute_quotient_polys",
                                            "commit_quotient_polys")}
        import plonky2_b200.fri as fri_mod
        import plonky2_b200.proof as proof_mod

        orig_fri, orig_open = fri_mod.prove_openings, proof_mod.StarkOpeningSet.new

        def timed(key, fn):
            def wrap(*a, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                r = fn(*a, **k)
                e1.record(stream)
                e1.synchronize()
                times.setdefault(key, []).append(e0.elapsed_time(e1))
                return r
            return wrap

        commit_calls = []

        def commit_values(values, rate_bits, cap_height, ctx_):
            key = "trace_commitment" if not commit_calls else "aux_commitment"
            commit_calls.append(key)
            return timed(key, orig["_commit_values"])(values, rate_bits, cap_height, ctx_)

        S.lookup_helper_columns = timed("helper_columns", orig["lookup_helper_columns"])
        S._commit_values = commit_values
        S.compute_quotient_polys = timed("quotient", orig["compute_quotient_polys"])
        S.commit_quotient_polys = timed("quotient_commitment", orig["commit_quotient_polys"])
        fri_mod.prove_openings = timed("fri", orig_fri)
        proof_mod.StarkOpeningSet.new = classmethod(lambda cls, *a, **k: timed("openings", orig_open)(*a, **k))
        try:
            whole = []
            proof = None
            for rep in range(args.reps + 1):
                times.clear()
                commit_calls.clear()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                e0.record(stream)
                proof = S.prove(st, cfg, tr, pis, ctx=ctx)
                e1.record(stream)
                e1.synchronize()
                wall = time.perf_counter() - t0
                if rep == 0:
                    continue  # warm-up
                whole.append((e0.elapsed_time(e1), wall * 1e3, {k: v[0] for k, v in times.items()}))
        finally:
            for k, v in orig.items():
                setattr(S, k, v)
            fri_mod.prove_openings, proof_mod.StarkOpeningSet.new = orig_fri, orig_open
        p = proof.proof
        parts = dict(trace_cap=p.trace_cap.hashes, auxiliary_polys_cap=p.auxiliary_polys_cap.hashes,
                     quotient_polys_cap=p.quotient_polys_cap.hashes, openings=p.openings, fri_bytes=p.opening_proof.to_bytes(),
                     public_inputs=proof.public_inputs, degree_bits=log_n)
        reason = verify_stark_proof(oracle_lib, st, cfg, parts)
        if reason is not None:
            raise SystemExit("the proof at 2^%d does not verify: %s" % (log_n, reason))
        med = lambda xs: float(np.median(xs))  # noqa: E731
        phases = {k: med([w[2][k] for w in whole]) for k in whole[0][2]}
        res = dict(gpu=name, power_limit=limit, log_n=log_n, looking_columns=16, lookups=1, challenges=cfg.num_challenges,
                   constraint_degree=3, instructions=len(st.constraint_program(2).instrs), reps=args.reps,
                   prove_ms_events=med([w[0] for w in whole]), prove_ms_wall=med([w[1] for w in whole]),
                   phases_ms=phases, verified=True)
        print(json.dumps(res), flush=True)
        results.append(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
