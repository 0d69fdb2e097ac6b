#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native plonky2 prover hot path.

A "step" = one pass of the hot path over one batch of synthetic input: PolynomialBatch::from_values
(plonky2/src/fri/oracle.rs:57-112) = iNTT of every column -> rate-2^-r coset LDE -> Poseidon Merkle
commitment of the LDE rows.  Workload at N=1 = BASELINE.json configs[1]: 234 columns x 2^20 values,
rate_bits 3, cap_height 4 (2^23 leaves of 234 elements).  Metric = Goldilocks field-elements/s
(LDE output elements committed per second = B*N / t), whole job.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

N > 1: the SAME commitment is row-block sharded over the ranks (strong scaling): rank g builds leaf rows
[g*N/G, (g+1)*N/G) on its own coset and the ranks all-gather their Merkle-cap entries over NCCL.
Prints ONE JSON line on rank 0 (see DESIGN.md "Measurement").
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "goldilocks_field_elements_per_s_ntt_lde_merkle"
UNIT = "elements/s"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


PRESETS = {  # --config name: (columns, log_n, rate_bits, cap_height, generator seed, BASELINE.json configs index)
    "cfg2": (234, 20, 3, 4, 0x02, 1),
    "cfg5": (64, 24, 1, 4, 0x05, 4),
}


def preset_of(args):
    for name, (B, log_n, r, h, seed, idx) in PRESETS.items():
        if (args.cols, args.log_n, args.rate_bits, args.cap_height) == (B, log_n, r, h):
            return name, seed, idx
    return None, 0x02, None


def load_fixture(args):
    """Golden cap of this exact workload from the CPU oracle (tools/make_fullscale_fixtures.py), or None."""
    name, seed, _ = preset_of(args)
    path = os.path.join(ROOT, "tests", "golden", "fullscale_%s.json" % name) if name else None
    if path and os.path.exists(path) and args.seed == seed:
        return json.load(open(path))
    return None


def synth_torch(seed, shape, device):
    """tests/conftest.py synth() (the SURVEY 8(d) splitmix64 counter generator) on the device, bit for bit:
    int64 arithmetic wraps like uint64; logical shifts are emulated with masks."""
    import torch

    def s64(v):
        v &= (1 << 64) - 1
        return v - (1 << 64) if v >= (1 << 63) else v

    def lsr(z, k):
        return (z >> k) & ((1 << (64 - k)) - 1)

    n = 1
    for d in shape:
        n *= d
    z = torch.arange(n, dtype=torch.int64, device=device) + s64(seed * 0x1000000000 + 0x9E3779B97F4A7C15)
    z = (z ^ lsr(z, 30)) * s64(0xBF58476D1CE4E5B9)
    z = (z ^ lsr(z, 27)) * s64(0x94D049BB133111EB)
    z = z ^ lsr(z, 31)
    z = torch.where((z < 0) & (z >= -0xFFFFFFFF), z + 0xFFFFFFFF, z)  # z >= p (unsigned)  ->  z - p
    return z.reshape(shape)


def workload_config(args, world):
    n, N = 1 << args.log_n, 1 << (args.log_n + args.rate_bits)
    name = "from_values: %d columns x 2^%d values, rate_bits=%d, cap_height=%d (2^%d leaves x %d)" % (
        args.cols, args.log_n, args.rate_bits, args.cap_height, args.log_n + args.rate_bits, args.cols)
    pname, _, idx = preset_of(args)
    if getattr(args, "fri_commit", False):
        name += " + FRI commit phase of its opening proof"
    if pname:
        name = "BASELINE configs[%d]: " % idx + name
    return {
        "workload": name,
        "columns": args.cols, "log_n": args.log_n, "rate_bits": args.rate_bits, "cap_height": args.cap_height,
        "lde_elements": args.cols * N,
        "l2": "inputs %.2f GB + leaves %.2f GB per step, far larger than the 126 MB L2 (no flush needed)" % (
            args.cols * n * 8 / 1e9, args.cols * N * 8 / 1e9),
        "parallelism": ("column-sharded iNTT storing into every rank's coefficient matrix over NVLink (64-column "
                        "chunks), then row-block (coset) sharded LDE + Merkle x%d + NCCL all-gather of cap "
                        "entries" % world) if world > 1 else "single GPU",
    }


# ------------------------------------------------------------------------------------------------
# reference arm: the CPU path (oracle port; the Rust reference cannot be built in this image)
# ------------------------------------------------------------------------------------------------
CPU_STEP_SECONDS = 4.5  # one CPU step of the bounded sample: the SAME sample in the --impl reference arm (K steps) and the cpu_baseline leg


def cpu_sample(args, cores, target_seconds=CPU_STEP_SECONDS):
    """Rows per CPU step: the FULL workload when one step fits `target_seconds` on this box's cores, otherwise the
    largest power-of-two row count that does (same columns / rate / cap). Calibrated at 2^14 rows, where the CPU
    path is already bandwidth- and hash-bound like the full size, scaling n log n."""
    base = min(14, args.log_n)
    run_cpu_once(args, min(12, base), cores, 7)  # warm-up (thread pool, page faults)
    dt, _ = run_cpu_once(args, base, cores, 8)
    log_n_s = base
    while log_n_s < args.log_n and dt * 2.0 * (log_n_s + 1 + 8) / (log_n_s + 8) <= target_seconds:
        dt *= 2.0 * (log_n_s + 1 + 8) / (log_n_s + 8)
        log_n_s += 1
    avail = 0
    try:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    except (ValueError, OSError):
        pass
    while avail and log_n_s > base and 8 * args.cols * ((2 << (log_n_s + args.rate_bits)) + (2 << log_n_s)) > 0.7 * avail:
        log_n_s -= 1  # the oracle holds the column-major LDE and the row-major leaves at once
    return log_n_s


def cpu_threads():
    """Threads for the CPU arm: all hardware threads, or one per physical core when SMT siblings slow the
    hash-bound path down (measured on a small sample; the faster wins)."""
    import oracle_lib

    class A:  # small probe shape
        cols, log_n, rate_bits, cap_height = 64, 12, 3, 4

    full = oracle_lib.nproc()
    best, best_dt = full, None
    for c in sorted({full, max(1, full // 2)}, reverse=True):
        run_cpu_once(A, 12, c, 5)
        dt = min(run_cpu_once(A, 12, c, 6)[0] for _ in range(3))
        if best_dt is None or dt < 0.9 * best_dt:
            best, best_dt = c, dt
    return best


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def sample_text(args, log_n_s):
    if log_n_s == args.log_n:
        return "the full workload (n=2^%d rows per step)" % log_n_s
    return "same columns/rate/cap, n=2^%d rows per step (bounded sample: 1/%d of the n=2^%d workload)" % (
        log_n_s, 1 << (args.log_n - log_n_s), args.log_n)


def run_cpu_once(args, log_n_s, cores, seed):
    import oracle_lib

    from conftest import synth

    vals = synth(seed, (args.cols, 1 << log_n_s))  # seeds >= 7 are bench-only; a full-size run at args.seed is the fixture
    t0 = time.perf_counter()
    c = oracle_lib.Commit(vals, args.rate_bits, args.cap_height, nthreads=cores)
    dt = time.perf_counter() - t0
    cap = c.cap
    del c
    return dt, cap


def reference_arm(args, rank, world):
    if rank != 0:
        return
    import oracle_lib

    cores = cpu_threads()
    log_n_s = cpu_sample(args, cores)
    for w in range(args.warmup):
        run_cpu_once(args, min(log_n_s, 12), cores, 100 + w)
    times = []
    for k in range(args.steps):
        dt, _ = run_cpu_once(args, log_n_s, cores, 200 + k)
        times.append(dt)
    elems = args.cols * (1 << (log_n_s + args.rate_bits))
    total = sum(times)
    value = elems * len(times) / total
    sample = sample_text(args, log_n_s)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "cpu_model": cpu_model(), "sample_log_n": log_n_s,
                         "note": "C++ restatement of the reference CPU algorithm (oracle/) on a persistent thread "
                                 "pool; the Rust reference needs nightly cargo, absent from this image"},
        "sample": sample,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(device)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(",") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if sm:
            busy = sorted(sm)[len(sm) // 2:]  # samples under load are the upper half when idle ones exist
            out.update(sm_mhz=float(np.median(busy)), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step computed, for comparing two builds output for output
# ------------------------------------------------------------------------------------------------
DUMP_SEED = 0x0D
DUMP_LEAF_ROWS = 4096           # sampled Merkle leaves, each with its path
DUMP_LEAF_BYTES = 24 << 20      # fewer rows when the leaves are wide
DUMP_COEFFS = 1 << 20           # sampled coefficients
DUMP_MAX_BYTES = 64 << 20


def limbs(words):
    """Field words as float64, exactly: a trailing axis of 2 holds each word's low and high 32 bits."""
    w = np.ascontiguousarray(words, dtype=np.uint64)
    return np.stack([(w & np.uint64(0xFFFFFFFF)).astype(np.float64), (w >> np.uint64(32)).astype(np.float64)], axis=-1)


def dump_outputs(out_dir, hnd, cap, fri_result, ctx, dev):
    """Write what a caller of the timed commitment receives as DIR/<name>.npy (float64):
    merkle_cap (the whole cap), leaf_rows + merkle_paths (gl_commit_open of leaf_row_index, a fixed seeded sample of
    leaves), coeffs (the coefficient matrix, column-major, at the flat positions coeff_index, a fixed seeded sample),
    and with the FRI commit phase fri_caps (one cap per round) and fri_final_poly. Field words go through limbs();
    the index arrays are plain float64 (exact below 2^53)."""
    import torch

    from plonky2_b200 import _native as N

    L = N.lib()
    B, W, log_n = L.gl_commit_num_polys(hnd), L.gl_commit_leaf_width(hnd), L.gl_commit_degree_log(hnd)
    log_N, h = log_n + L.gl_commit_rate_bits(hnd), L.gl_commit_cap_height(hnd)
    rng = np.random.default_rng(DUMP_SEED)
    n_rows = min(1 << log_N, DUMP_LEAF_ROWS, max(1, DUMP_LEAF_BYTES // (16 * W)))
    rows = np.sort(rng.choice(1 << log_N, n_rows, replace=False)).astype(np.uint64)
    leaves = np.empty((n_rows, W), dtype=np.uint64)
    paths = np.empty((n_rows, log_N - h, 4), dtype=np.uint64)
    N.check(L.gl_commit_open(hnd, N.np_ptr(rows), n_rows, N.np_ptr(leaves), N.np_ptr(paths)), ctx.h)
    pos = np.sort(rng.choice(B << log_n, min(B << log_n, DUMP_COEFFS), replace=False))
    coeffs = torch.empty(B << log_n, dtype=torch.int64, device=dev)
    N.check(L.gl_commit_coeffs(hnd, C.c_void_p(coeffs.data_ptr()), N.MEM_DEVICE), ctx.h)
    picked = coeffs[torch.from_numpy(pos).to(dev)].cpu().numpy().view(np.uint64)
    del coeffs
    arrays = {"merkle_cap": limbs(cap), "leaf_row_index": rows.astype(np.float64), "leaf_rows": limbs(leaves),
              "merkle_paths": limbs(paths), "coeff_index": pos.astype(np.float64), "coeffs": limbs(picked)}
    if fri_result is not None:
        caps, final_poly = fri_result
        arrays["fri_caps"] = limbs(np.stack([c.hashes for c in caps]))
        arrays["fri_final_poly"] = limbs(final_poly)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, "output dump of %d bytes exceeds %d" % (total, DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def gpu_arm(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from plonky2_b200 import _native as N

    L = N.lib()
    stream = torch.cuda.Stream(device=dev)
    ctx = N.Context(local_rank, stream=stream.cuda_stream)
    ctx.set_profiling(True)
    if args.ntt_group:
        ctx.set_ntt_group(args.ntt_group)
    B, log_n, r, h = args.cols, args.log_n, args.rate_bits, args.cap_height
    n, NN = 1 << log_n, 1 << (log_n + r)
    cap_local_words = (4 << h) // world
    peak, peak_src = load_peaks()

    with torch.cuda.stream(stream):
        vals = synth_torch(args.seed, (B, n), dev)  # SURVEY 8(d) generator: the oracle can reproduce cap0 without torch
        fixture = load_fixture(args)
        cap_local = torch.empty(cap_local_words, dtype=torch.int64, device=dev)
        cap_full = torch.empty(cap_local_words * world, dtype=torch.int64, device=dev)

        committer = None
        if world >= 2:
            # column-sharded iNTT whose stores are the coefficient all-gather (NVLink), pipelined under the LDE
            from plonky2_b200.distributed import PipelinedCommitter

            committer = PipelinedCommitter(ctx, B, log_n, r, h, rank, world, dev, transport=args.transport)

        fri_ctx = None
        if args.fri_commit:
            # BASELINE configs[4] ("LDE + FRI commit"): after the trace commitment, the FRI commit phase of its opening
            # proof (starky/src/prover.rs:83-94 -> fri/oracle.rs:176-220 + fri/prover.rs:84-150) with the real host
            # transcript: observe cap -> alpha -> batch-combine at zeta / g*zeta -> fold rounds (arity 16 x5), caps out.
            import plonky2_b200 as pb
            from plonky2_b200 import fri as F

            cfg = pb.starky_standard_fast_fri_config() if r == 1 else pb.standard_recursion_fri_config()
            params = cfg.fri_params(log_n, False)
            zeta = (0x1122334455667788 % pb.field.ORDER, 0x99AABBCCDDEEFF00 % pb.field.ORDER)
            gz = pb.field.ext_mul(zeta, (pb.field.primitive_root_of_unity(log_n), 0))
            inst = pb.FriInstanceInfo([pb.FriOracleInfo(B, False)],
                                      [pb.FriBatchInfo(zeta, [pb.FriPolynomialInfo(0, i) for i in range(B)]),
                                       pb.FriBatchInfo(gz, [pb.FriPolynomialInfo(0, 0), pb.FriPolynomialInfo(0, 1)])])

            class _Oracle:  # what fri._begin / _begin_values / eval_commitments need of a PolynomialBatch
                def __init__(self, h):
                    self.h, self.ctx = h, ctx
                    self.num_polys, self.shard_index, self.num_shards = B, rank, world

            def gather_words(local):  # all-gather of the ranks' cap entries of one FRI round (NCCL)
                t_loc = torch.from_numpy(local.view(np.int64)).to(dev)
                t_all = torch.empty(t_loc.numel() * world, dtype=torch.int64, device=dev)
                dist.all_gather_into_tensor(t_all, t_loc)
                return t_all.cpu().numpy().view(np.uint64)

            def fri_commit_phase(hnd, cap_np):
                ch = pb.Challenger()
                ch.observe_cap(pb.MerkleCap(np.ascontiguousarray(cap_np).view(np.uint64).reshape(-1, 4)))
                if world > 1 and args.fri_values:
                    # N > 1: the codeword is composed in the VALUE domain from this rank's own LDE rows (and the openings,
                    # which a prover holds at this point: proof.rs:313-351), so every FRI round is rank-local
                    orc = _Oracle(hnd)
                    ev_z, ev_gz = pb.eval_commitments([(orc, zeta), (orc, gz)])
                    opened = [ev_z, ev_gz[:2]]
                    for o in opened:
                        ch.observe_elements(o.reshape(-1))
                    st = F._begin_values(inst, [orc], ch.get_extension_challenge(), opened, params)
                else:
                    st = F._begin(inst, [_Oracle(hnd)], ch.get_extension_challenge(), params)
                try:
                    caps, final = F.fri_committed_trees(st, ch, params, shard=(rank, world) if world > 1 else None,
                                                        gather=gather_words)
                finally:
                    st.close()
                return caps, final

            fri_ctx = fri_commit_phase
        fri_out = [None]
        fri_spans = []

        def step_device(keep=False):
            """One step; keep=True returns the commitment handle instead of destroying it."""
            if committer is not None:
                # column-sharded iNTT -> NCCL all-gather of coefficients -> row-block sharded LDE + Merkle
                hnd = committer.commit(vals, from_host=False)
            else:
                hnd = N.vp()
                N.check(L.gl_commit_create_sharded(ctx.h, C.c_void_p(vals.data_ptr()), n, B, log_n, r, h, None, 0,
                                                   N.MEM_DEVICE, rank, world, C.byref(hnd)), ctx.h)
            N.check(L.gl_commit_cap(hnd, C.c_void_p(cap_local.data_ptr()), N.MEM_DEVICE), ctx.h)
            if world > 1:
                dist.all_gather_into_tensor(cap_full, cap_local)
            else:
                cap_full.copy_(cap_local)
            if fri_ctx is not None:
                fa, fb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                fa.record(stream)
                fri_out[0] = fri_ctx(hnd, cap_full.cpu().numpy())
                fb.record(stream)
                fri_spans.append((fa, fb))
            if keep:
                return hnd
            L.gl_commit_destroy(hnd)

        def sync_all():
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize(dev)

        for _ in range(max(args.warmup, 3)):
            step_device()
        sync_all()
        ctx.reset_phases()
        del fri_spans[:]
        if committer is not None:
            committer.timing = True
            committer.transfer_ms()
        launches0 = ctx.launch_count
        sampler = ClockSampler(local_rank) if rank == 0 else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        marks = []
        last = None
        for k in range(args.steps):
            # with --dump-outputs the last step's commitment outlives the timed window (its free is stream-ordered)
            last = step_device(keep=bool(args.dump_outputs) and k == args.steps - 1)
            m = torch.cuda.Event(enable_timing=True)
            m.record(stream)
            marks.append(m)
        e1.record(stream)
        sync_all()
        ms = e0.elapsed_time(e1)
        step_ms = [a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks)]
        launches = ctx.launch_count - launches0
        side = committer.transfer_ms() if committer is not None else None
        if committer is not None:
            committer.timing = False
        clocks = sampler.stop() if sampler else None
        phases = ctx.phase_ms()
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_max = float(t.item())
        cap_dev = cap_full.cpu().numpy().view(np.uint64).reshape(-1, 4).copy()
        cap_ok = None
        if fixture is not None:  # golden cap of this exact workload from the CPU oracle (tests/golden/fullscale_*.json)
            cap_ok = bool(np.array_equal(cap_dev, np.array(fixture["cap"], dtype=np.uint64)))
            assert cap_ok, "rank %d: the gathered Merkle cap differs from the oracle fixture" % rank
        if last is not None:
            dump_outputs(args.dump_outputs, last, cap_dev, fri_out[0], ctx, dev)
            L.gl_commit_destroy(last)

        # ---- end to end through the C ABI with HOST buffers (pinned): H2D of the columns + D2H of the cap
        host_vals = torch.empty((B, n), dtype=torch.int64, pin_memory=True)
        host_vals.copy_(vals)
        torch.cuda.synchronize(dev)
        host_cap = np.empty(cap_local_words, dtype=np.uint64)

        def step_e2e():
            if committer is not None:
                hnd = committer.commit(host_vals, from_host=True)  # every rank uploads 1/G of the columns
            else:
                hnd = N.vp()
                N.check(L.gl_commit_create_sharded(ctx.h, C.c_void_p(host_vals.data_ptr()), n, B, log_n, r, h, None, 0,
                                                   N.MEM_HOST, rank, world, C.byref(hnd)), ctx.h)
            N.check(L.gl_commit_cap(hnd, N.np_ptr(host_cap), N.MEM_HOST), ctx.h)  # synchronises
            if world > 1:
                cap_local.copy_(torch.from_numpy(host_cap.view(np.int64)))
                dist.all_gather_into_tensor(cap_full, cap_local)
            if fri_ctx is not None:
                fri_ctx(hnd, cap_full.cpu().numpy() if world > 1 else host_cap)
            L.gl_commit_destroy(hnd)

        step_e2e()
        sync_all()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ke = max(1, min(args.steps, 3))
        e2.record(stream)
        for _ in range(ke):
            step_e2e()
        e3.record(stream)
        sync_all()
        t2 = torch.tensor([e2.elapsed_time(e3)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ms_e2e = float(t2.item()) / ke
        assert np.array_equal(host_cap.reshape(-1, 4), cap_dev[rank * (len(cap_dev) // world):(rank + 1) * (len(cap_dev) // world)])

        # ---- bare batched NTT roofline (the north star's "2^20-point NTT"): 64 columns, working set 512 MiB
        ntt = None
        if rank == 0 and not args.no_ntt:
            cols_ntt = args.ntt_cols
            buf = vals[:cols_ntt].clone() if cols_ntt <= B else torch.randint(0, 2**63 - 1, (cols_ntt, n), dtype=torch.int64, device=dev)
            for _ in range(3):
                N.check(L.gl_ntt(ctx.h, C.c_void_p(buf.data_ptr()), log_n, cols_ntt, n, 0, 0, 1, N.MEM_DEVICE), ctx.h)
            torch.cuda.synchronize(dev)
            l0 = ctx.launch_count
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            a.record(stream)
            for _ in range(reps):
                N.check(L.gl_ntt(ctx.h, C.c_void_p(buf.data_ptr()), log_n, cols_ntt, n, 0, 0, 1, N.MEM_DEVICE), ctx.h)
            b.record(stream)
            torch.cuda.synchronize(dev)
            ms_ntt = a.elapsed_time(b) / reps
            alg = 16.0 * n * cols_ntt
            ntt = {"workload": "forward NTT, %d columns x 2^%d, in place, device resident" % (cols_ntt, log_n),
                   "ms": ms_ntt, "elements_per_s": cols_ntt * n / (ms_ntt * 1e-3),
                   "algorithmic_bytes": alg, "achieved": alg / (ms_ntt * 1e-3) / 1e9, "unit": "GB/s",
                   "peak": peak, "frac": alg / (ms_ntt * 1e-3) / 1e9 / peak,
                   "launches_per_call": (ctx.launch_count - l0) // reps}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    steps = args.steps
    ms_step = ms_max / steps
    value = B * NN / (ms_step * 1e-3)
    N_loc = NN // world
    # dominant kernel = the Poseidon leaf hash (k_leaf_hash): algorithmic bytes = leaves read + digests written
    leaf_ms, leaf_cnt = phases["leaf_hash"]
    leaf_avg = leaf_ms / max(1, leaf_cnt)
    leaf_bytes = 8.0 * N_loc * B + 32.0 * N_loc
    perms = N_loc * ((B + 7) // 8 if B > 4 else 0)
    traffic, traffic_note = None, None
    try:  # DRAM bytes per launch from the committed ncu --set full capture (scaled by the algorithmic bytes)
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["k_leaf_hash"]
        traffic = tr["dram_bytes_per_algorithmic_byte"] * leaf_bytes
        traffic_note = "ncu dram read+write per algorithmic byte x this launch's algorithmic bytes; " + tr["source"]
    except Exception:
        pass
    roof = {
        "kernel": "k_leaf_hash (Poseidon sponge over each LDE row)", "bound": "hbm",
        "achieved": leaf_bytes / (leaf_avg * 1e-3) / 1e9 if leaf_avg else None, "peak": peak, "unit": "GB/s",
        "frac": (leaf_bytes / (leaf_avg * 1e-3) / 1e9 / peak) if leaf_avg else None,
        "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src, "avg_ms": leaf_avg, "launches": leaf_cnt,
        "algorithmic_bytes": leaf_bytes,
        "permutations_per_s": perms / (leaf_avg * 1e-3) if leaf_avg else None,
        "note": "instruction-issue bound (x^7 S-boxes on the integer pipes, MDS / partial rounds on the FP64 pipe), not HBM bound: see DESIGN.md",
    }
    # integer-issue roofline (what actually bounds these kernels): thread-instructions/s vs 128 lanes/clk/SM
    issue = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        sm_clk = (clocks or {}).get("sm_mhz") or 1965.0
        peak_issue = 148 * 128 * sm_clk * 1e6
        ipp = tr["k_leaf_hash"]["thread_instructions_per_permutation"]
        ach = ipp * roof["permutations_per_s"]
        issue = {"kernel": "k_leaf_hash", "bound": "instruction issue (4 warp-instructions/clk/SM)",
                 "achieved": ach, "peak": peak_issue, "unit": "thread-instructions/s", "frac": ach / peak_issue,
                 "thread_instructions_per_permutation": ipp, "source": tr["k_leaf_hash"]["instr_source"]}
    except Exception:
        pass
    lde_ms = (phases["intt"][0] + phases["lde"][0]) / steps
    lde_bytes = 8.0 * n * B * (2 + (1 << r) / world)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic", "config": workload_config(args, world),
        "clocks": clocks,
        "e2e": {"value": B * NN / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": B * n * 8,  # whole job: with G ranks each uploads its 1/G of the columns
                "d2h_bytes_per_step": cap_local_words * 8,
                "note": "host (pinned) columns -> gl_commit_create -> cap on host; leaves/digests stay on the "
                        "device behind the handle (fetched on demand by gl_commit_leaves/_open)"},
        "gpu_launches": int(launches),
        "roofline": roof,
        "roofline_issue": issue,
        "phases_ms_per_step": dict({k: v[0] / steps for k, v in phases.items()},
                                   **({"side_stream_nvlink_copy_and_barriers (under the main stream)": side[0] / max(1, side[1])}
                                      if side else {})),
        "roofline_lde": {"kernels": "k_passA + k_passB (iNTT + 2^r coset NTTs, leaf-major stores)", "bound": "hbm",
                         "algorithmic_bytes": lde_bytes, "ms": lde_ms,
                         "achieved": lde_bytes / (lde_ms * 1e-3) / 1e9 if lde_ms else None, "peak": peak,
                         "unit": "GB/s", "frac": lde_bytes / (lde_ms * 1e-3) / 1e9 / peak if lde_ms else None},
        "roofline_ntt": ntt,
        "fri_commit_phase": ({"ms_per_step": sum(a.elapsed_time(b) for a, b in fri_spans[:steps]) / max(1, min(steps, len(fri_spans))),
                              "rounds": len(fri_out[0][0]), "final_poly_len": int(len(fri_out[0][1])),
                              "last_round_cap0": [int(x) for x in fri_out[0][0][-1].hashes[0]],
                              "note": "inside the timed step: alpha/betas from the host transcript, caps to the host"}
                             if fri_out[0] is not None else None),
        "cap0": [int(x) for x in cap_dev[0]],
        "cap_matches_fixture": cap_ok,
        "step_ms_rank0": step_ms,
        "coefficient_transport": (committer.transport + (" (%s)" % committer.transport_note if committer.transport_note else ""))
        if committer is not None else None,
        "input": "splitmix64 counter generator, seed 0x%02x (tests/conftest.py synth; SURVEY 8d)" % args.seed,
    }
    # ---- CPU baseline (bounded sample, rank 0, N=1 only)
    if world == 1 and not args.no_cpu:
        import oracle_lib

        cores = cpu_threads()
        log_n_s = cpu_sample(args, cores)
        run_cpu_once(args, log_n_s, cores, 199)  # first touch of the recycled buffers
        dt, _ = run_cpu_once(args, log_n_s, cores, 200)
        line["cpu_baseline"] = {
            "value": B * (1 << (log_n_s + r)) / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "cpu_model": cpu_model(), "sample_log_n": log_n_s,
            "sample": sample_text(args, log_n_s) + ", one step, %.2f s" % dt}
    if world == 1 and not args.no_extra:
        try:
            line["prove_recursion_shape"] = recursion_shape(local_rank)
        except Exception as e:  # never lose the headline line to the secondary measurement
            line["prove_recursion_shape"] = {"error": repr(e)}
        try:   # in a child process with a timeout: new code, not yet run on a GPU -- it must not be able to take the line down
            env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank)))
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--plonk-circuit-only"], capture_output=True,
                                 text=True, timeout=300, env=env)
            line["prove_plonk_circuit"] = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as e:
            line["prove_plonk_circuit"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# BASELINE configs[3] stand-in: the hot-path call sequence of ONE bench_recursion-sized proof
# (SURVEY section 8d cfg4: the real circuits need the Rust reference; this is the recursion-shaped synthetic)
# ------------------------------------------------------------------------------------------------
def recursion_shape(ctx_device, reps=5):
    """n = 2^14, standard_recursion_config (rate 1/8, cap 4, arity 16 x3, 16-bit PoW, 28 queries):
    per proof = from_values(135 wires) + from_values(20 Z/partial products) + from_coeffs(16 quotient chunks)
    + prove_openings over 4 oracles (84 constants/sigmas committed once at build time), host transcript in
    the loop, HOST buffers in and proof bytes out. Returns GPU and CPU-port milliseconds per proof."""
    import oracle_lib
    import plonky2_b200 as pb
    from conftest import synth

    log_n, r, h = 14, 3, 4
    n = 1 << log_n
    Bs = [84, 135, 20, 16]
    data = [synth(0x40 + i, (B, n)) for i, B in enumerate(Bs)]
    cfg = pb.standard_recursion_fri_config()
    params = cfg.fri_params(log_n, False)
    zeta = (0x123456789ABCDEF % pb.field.ORDER, 0x0FEDCBA987654321 % pb.field.ORDER)
    gz = pb.field.ext_mul(zeta, (pb.field.primitive_root_of_unity(log_n), 0))
    allp = [pb.FriPolynomialInfo(o, i) for o, B in enumerate(Bs) for i in range(B)]
    inst = pb.FriInstanceInfo([pb.FriOracleInfo(B, False) for B in Bs],
                              [pb.FriBatchInfo(zeta, allp), pb.FriBatchInfo(gz, [pb.FriPolynomialInfo(2, 0), pb.FriPolynomialInfo(2, 1)])])
    obatches = [(b.point, [(p.oracle_index, p.polynomial_index) for p in b.polynomials]) for b in inst.batches]
    ctx = pb.default_context(ctx_device)
    const = pb.PolynomialBatch.from_values(data[0], r, False, h, ctx=ctx)

    def gpu_once():
        ch = pb.Challenger()
        ch.observe_cap(const.merkle_tree.cap)
        wires = pb.PolynomialBatch.from_values(data[1], r, False, h, ctx=ctx)
        ch.observe_cap(wires.merkle_tree.cap)
        ch.get_n_challenges(4)
        zs = pb.PolynomialBatch.from_values(data[2], r, False, h, ctx=ctx)
        ch.observe_cap(zs.merkle_tree.cap)
        ch.get_n_challenges(2)
        quot = pb.PolynomialBatch.from_coeffs(data[3], r, False, h, ctx=ctx)
        ch.observe_cap(quot.merkle_tree.cap)
        ch.get_extension_challenge()
        proof = pb.prove_openings(inst, [const, wires, zs, quot], ch, params)
        b = proof.to_bytes()
        for c in (wires, zs, quot):
            c.close()
        return b

    gpu_once()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        proof_bytes = gpu_once()
        ts.append(time.perf_counter() - t0)
    cores = oracle_lib.nproc()
    oconst = oracle_lib.Commit(data[0], r, h, nthreads=cores)

    def cpu_once():
        och = oracle_lib.Challenger()
        och.observe_cap(oconst.cap)
        w = oracle_lib.Commit(data[1], r, h, nthreads=cores)
        och.observe_cap(w.cap)
        och.get_n_challenges(4)
        z = oracle_lib.Commit(data[2], r, h, nthreads=cores)
        och.observe_cap(z.cap)
        och.get_n_challenges(2)
        q = oracle_lib.Commit(data[3], r, h, is_coeffs=True, nthreads=cores)
        och.observe_cap(q.cap)
        och.get_extension_challenge()
        return oracle_lib.prove_openings([oconst, w, z, q], obatches, och, oracle_lib.make_params(r, h, 16, 28, [4, 4, 4]))

    t0 = time.perf_counter()
    oproof = cpu_once()
    cpu_ms = (time.perf_counter() - t0) * 1e3
    # the same sequence through the compiled C++ host layer (include/plonky2_b200.hpp): no Python in the loop
    cpp = None
    try:
        with tempfile.TemporaryDirectory() as tmp:
            exe = os.path.join(tmp, "gl_prove_latency")
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-o", exe,
                                   os.path.join(ROOT, "tools", "prove_latency.cpp"), "-L" + os.path.join(ROOT, "plonky2_b200"),
                                   "-lplonky2_b200", "-Wl,-rpath," + os.path.join(ROOT, "plonky2_b200")])
            cpp = json.loads(subprocess.run([exe, "7"], capture_output=True, text=True, timeout=120).stdout.strip().splitlines()[-1])
    except Exception as e:
        cpp = {"error": repr(e)}
    return {"cpp_host": cpp,"workload": "recursion-shaped synthetic proof, n=2^14, standard_recursion_config "
                        "(3 commitments of 135/20/16 polys + prove_openings over 255 polys, arity 16 x3, PoW 16, 28 queries)",
            "gpu_ms_per_proof_median": float(np.median(ts)) * 1e3, "gpu_ms_per_proof_min": min(ts) * 1e3,
            "cpu_port_ms_per_proof": cpu_ms, "cpu_cores": cores, "proof_bytes": len(proof_bytes),
            "bit_exact_vs_cpu_port": bool(proof_bytes == oproof),
            "note": "host buffers in, proof bytes out, Python host transcript in the loop (includes ctypes/Python overhead)"}


# ------------------------------------------------------------------------------------------------
# BASELINE metric, second half ("prove() ms vs CPU ref") on a plonky2-shaped circuit: the whole prove() --
# commitments, Z / partial products, quotient over every gate type's constraints, openings, FRI -- for a 2^12-row
# circuit in standard_recursion_config, against the same prover assembled from the CPU oracle's pieces
# ------------------------------------------------------------------------------------------------
def plonk_circuit_proof(ctx_device, reps=3):
    """plonk.prove_with_witness (plonk/prover.rs:132-360) for a synthetic circuit of 2^12 rows: 135 wires / 80 routed,
    Arithmetic + Poseidon + every other constraint-carrying gate type, copy constraints, standard FRI parameters
    (rate 1/8, cap 4, arity 16, 16-bit PoW, 28 queries). Host witness in, write_proof_with_public_inputs bytes out."""
    import oracle_lib
    import plonk_circuits as PC
    import plonky2_b200 as pb
    from plonky2_b200 import plonk

    degree_bits = 12
    cfg = plonk.CircuitConfig()
    extra = ("ArithmeticExtensionGate", "MulExtensionGate", "BaseSumGate", "ReducingGate", "ReducingExtensionGate",
             "PoseidonMdsGate", "RandomAccessGate", "ExponentiationGate", "CosetInterpolationGate")
    c = PC.FibonacciCircuit(plonk, cfg, degree_bits, seed=7, poseidon_rows=256, extra=extra, public_inputs=[1, 2, 3])
    fri = pb.standard_recursion_fri_config()
    digest = [0x11, 0x22, 0x33, 0x44]
    ctx = pb.default_context(ctx_device)
    cs = pb.PolynomialBatch.from_values(c.constants_sigmas, cfg.rate_bits, False, cfg.cap_height, ctx=ctx)
    prover_data = plonk.ProverOnlyCircuitData(cs, c.sigmas, digest, fri.fri_params(degree_bits, False))

    def gpu_once():
        return plonk.prove_with_witness(prover_data, c.common, c.wires, c.public_inputs, ctx=ctx).to_bytes()

    proof_bytes = gpu_once()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        proof_bytes = gpu_once()
        ts.append(time.perf_counter() - t0)
    cs.close()
    t0 = time.perf_counter()
    want, parts = PC.oracle_prove(oracle_lib, c, digest, fri, c.public_inputs)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    prog, n_regs = c.common.vanishing_program().compile()
    return {"workload": "plonky2 prove() of a synthetic 2^12-row circuit, standard_recursion_config: %d gate types in %d "
                        "selector groups, quotient program of %d instructions per point" %
                        (len(c.common.gates), c.common.selectors_info.num_selectors(), len(prog)),
            "gpu_ms_per_proof_median": float(np.median(ts)) * 1e3, "gpu_ms_per_proof_min": min(ts) * 1e3,
            "cpu_port_ms_per_proof": cpu_ms, "cpu_cores": oracle_lib.nproc(), "proof_bytes": len(proof_bytes),
            "bit_exact_vs_cpu_port": bool(proof_bytes == want),
            "accepted_by_restated_verifier": PC.oracle_verify(oracle_lib, plonk, c, digest, fri, parts) is None,
            "note": "host witness in, proof bytes out, Python host transcript in the loop; first measurement of this path "
                    "(written after the round's GPU budget was spent)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(PRESETS), help="BASELINE.json preset (default cfg2 shape)")
    ap.add_argument("--cols", type=int, default=234)
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--rate-bits", type=int, default=3)
    ap.add_argument("--cap-height", type=int, default=4)
    ap.add_argument("--seed", type=lambda v: int(v, 0), default=None, help="input generator seed (default: the preset's)")
    ap.add_argument("--ntt-cols", type=int, default=64)
    ap.add_argument("--transport", default="auto", choices=["auto", "multimem", "p2p", "fused", "nccl"],
                    help="N > 1: how the coefficients reach the other ranks (auto = fused NVLink stores, NCCL fallback)")
    ap.add_argument("--fri-commit", action="store_true", default=None,
                    help="include the FRI commit phase of the opening proof in every step (default: on for cfg5)")
    ap.add_argument("--no-fri-commit", dest="fri_commit", action="store_false")
    ap.add_argument("--fri-values", dest="fri_values", action="store_true", default=False,
                    help="N > 1: compose the FRI codeword in the value domain from each rank's own LDE rows (rank-local "
                         "rounds) instead of the replicated coefficient-domain begin. Measured SLOWER for cfg5 on 2 GPUs "
                         "(221 vs 158 ms/step): the openings it needs come from gl_openings, whose one-CTA-per-polynomial "
                         "evaluation is built for many short polynomials, not 64 of length 2^24")
    ap.add_argument("--no-ntt", action="store_true")
    ap.add_argument("--ntt-group", type=int, default=0, help="columns per NTT group (0 = library default)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the recursion-shaped prove() timing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    ap.add_argument("--plonk-circuit-only", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl b200 on one GPU")
    if args.plonk_circuit_only:   # child mode of the secondary measurement `prove_plonk_circuit`
        try:
            print(json.dumps(plonk_circuit_proof(0)), flush=True)
        except Exception as e:
            print(json.dumps({"error": repr(e)}), flush=True)
        return
    if args.config:
        args.cols, args.log_n, args.rate_bits, args.cap_height = PRESETS[args.config][:4]
    if args.seed is None:
        args.seed = preset_of(args)[1]
    if args.fri_commit is None:
        args.fri_commit = preset_of(args)[0] == "cfg5"
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
