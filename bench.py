"""bench.py -- MinHash signatures/sec on the BASELINE.json workload (configs[1]:
1M docs x 256 tokens, num_perm=128 bulk signature build), N GPUs of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's numpy CPU path (oracle port)
    python bench.py --dump-outputs DIR ...    # also write sampled signature rows to DIR/*.npy (see dump_rows)

A "step" is one pass of the hot path over one batch of synthetic token hashes.
  value  : whole-job signatures/s with inputs already resident in HBM (CUDA events on the
           launch stream, max over ranks).  Inputs (1 GB/GPU) are larger than L2.
  e2e    : same metric through the host-buffer C-ABI call (dsk_minhash_bulk_host) with pinned
           HOST buffers: H2D of tokens+offsets and D2H of the signatures inside the timed region.
  roofline: algorithmic bytes (4T+4K per document, SURVEY.md section 8d) / kernel time vs the
           measured HBM copy peak (MEASURED_PEAKS.json).
  cpu_baseline: the oracle port of the reference's numpy path on all host cores, bounded sample.
Scaling is weak (each rank builds its own 1M-document shard; documents shard embarrassingly,
no data-path collective); the optional NCCL all-gather of the signature matrix is timed
separately and reported under "allgather".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# which __global__ function each --kernel choice runs (datasketch_b200/csrc/signature_kernel.cu, minhash_kernels.cu)
KERNEL_NAMES = {"two_phase": "minhash_sig_kernel<two_phase>", "direct": "minhash_bulk_kernel<direct>",
                "exact": "minhash_bulk_kernel<exact>"}
METRIC = "minhash_signatures_per_sec"
UNIT = "signatures/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--docs", type=int, default=1_000_000)
    ap.add_argument("--tokens", type=int, default=256)
    ap.add_argument("--num-perm", type=int, default=128)
    ap.add_argument("--kernel", default="auto", choices=["auto", "two_phase", "direct", "exact"])
    ap.add_argument("--cpu-sample-docs", type=int, default=0, help="0 = auto (about 10-30 s of CPU work)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-dups", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of rows of each timed signature matrix (rank 0) "
                         "to DIR/<name>.npy as float64, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this project's GPU path computed: it needs --impl ours")
    return args


DUMP_BYTES = 63_000_000   # array bytes --dump-outputs writes at most: under 64 MB in all with the .npy headers


def dump_rows(n_docs: int, k: int) -> np.ndarray:
    """Sorted indices of the rows that --dump-outputs writes of each signature matrix (up to three matrices of
    float64): every row when they fit, else a seeded sample that depends on --docs and --num-perm only."""
    m = min(n_docs, DUMP_BYTES // (8 * (3 * k + 1)))
    return np.sort(np.random.default_rng(0).choice(n_docs, size=m, replace=False))


# ---------------------------------------------------------------------------------------------
# synthetic workload
# ---------------------------------------------------------------------------------------------
def make_tokens(n_docs: int, t: int, seed: int, out: np.ndarray) -> None:
    """Uniform 32-bit token hashes (i.i.d.; SURVEY.md section 8d), filled chunk-wise into `out`."""
    rng = np.random.default_rng(seed)
    flat = out.reshape(-1)
    step = 1 << 24
    for i in range(0, flat.size, step):
        j = min(i + step, flat.size)
        flat[i:j] = rng.integers(0, 1 << 32, size=j - i, dtype=np.uint32)


# ---------------------------------------------------------------------------------------------
# CPU baseline: the reference's own MinHash.bulk when oracle/_ref/site holds the reference install
# (oracle/stage_reference.sh, run by build()), else the oracle port of its numpy path; all host cores, pinned workers
# ---------------------------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, "oracle", "_ref", "site")


def reference_kind() -> str:
    return "reference" if os.path.isdir(os.path.join(REF_DIR, "datasketch")) else "port"


def _identity(x):
    return x


_MY = None   # this worker's shard (set in the pool initializer, so that no data is pickled inside the timed region)


def _cpu_init(counter, cpus, per, t, kind):
    """Pool initializer: pin this worker to one core (round-robin over the allowed set) so that repeats and
    boxes compare -- an un-pinned 128-process pool moved 3.5x between two boxes in round 1 -- and build the
    worker's own shard of synthetic tokens."""
    global _MY
    with counter.get_lock():
        i = counter.value
        counter.value += 1
    try:
        os.sched_setaffinity(0, {cpus[i % len(cpus)]})
    except OSError:
        pass
    tok = np.empty((per, t), dtype=np.uint32)
    make_tokens(per, t, 99 + i, tok)
    _MY = tok.tolist() if kind == "reference" else tok   # the reference takes iterables of hashable tokens


def _cpu_worker(args):
    m, t, k, seed, kind = args
    tok = _MY[:m]
    if kind == "reference":          # datasketch.MinHash.bulk itself (datasketch/minhash.py:464-522)
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        from datasketch import MinHash
        mhs = MinHash.bulk(tok, num_perm=k, seed=seed, hashfunc=_identity)
        return int(sum(int(x.hashvalues[0]) for x in mhs) & 0xFFFF)
    from oracle import oracle_np as o
    off = np.arange(tok.shape[0] + 1, dtype=np.int64) * t
    sig = o.bulk_signatures_csr(tok.reshape(-1), off, k, seed)
    return int(sig[:, 0].sum() & 0xFFFF)


def cpu_reference_rate(n_docs: int, t: int, k: int, cores: int, repeats: int = 3):
    """Best-of-`repeats` signatures/s of the reference's CPU path over `cores` pinned processes, each on its own
    equal shard.  Returns (rate, best seconds, kind, all rates)."""
    import multiprocessing as mp
    kind = reference_kind()
    per = max(1, n_docs // cores)
    workers = min(cores, n_docs)
    total = per * workers
    ctx = mp.get_context("fork")
    cpus = sorted(os.sched_getaffinity(0))
    counter = ctx.Value("i", 0)
    rates = []
    with ctx.Pool(workers, initializer=_cpu_init, initargs=(counter, cpus, per, t, kind)) as pool:
        pool.map(_cpu_worker, [(min(per, 8), t, k, 1, kind)] * workers, chunksize=1)  # warm the workers
        for _ in range(repeats):
            t0 = time.perf_counter()
            pool.map(_cpu_worker, [(per, t, k, 1, kind)] * workers, chunksize=1)
            rates.append(total / (time.perf_counter() - t0))
    best = max(rates)
    return best, total / best, kind, rates


def cpu_sample_docs(args, cores: int) -> int:
    return args.cpu_sample_docs or min(args.docs, 2500 * cores)


def workload_config(args, cores: int) -> dict:
    """The `config` object -- identical in both arms (ours and --impl reference)."""
    n, t, k = args.docs, args.tokens, args.num_perm
    return {"workload": "configs[1]: %d docs x %d tokens, num_perm=%d bulk signature build" % (n, t, k),
            "docs_per_gpu": n, "l2": "inputs (%.2f GB/GPU) larger than L2" % (n * t * 4 / 1e9),
            "parallelism": "documents sharded over the GPUs, no data-path collective (weak scaling: %d docs per GPU)" % n,
            "cpu_arm_sample_docs_per_step": cpu_sample_docs(args, cores)}


def cpu_sample_text(sample: int, t: int, cores: int, kind: str, rates) -> str:
    what = ("datasketch.MinHash.bulk (the unmodified reference from oracle/_ref/site, hashfunc=identity on pre-hashed tokens)"
            if kind == "reference" else "oracle port of datasketch's numpy uint64 path")
    return ("%d docs x %d tokens per repeat, best of %d repeats (%s sig/s), %s over %d pinned processes"
            % (sample, t, len(rates), "/".join("%.0f" % r for r in rates), what, cores))


# ---------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self, t0: float, t1: float):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = max(mx, cmax)
            if t0 <= ts <= t1 + 0.15:
                sm.append(clk)
                for nm, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(gpu_index: int):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (what `numactl` would do), so the
    pinned host buffers of the e2e leg are first-touched on the local node.  Best effort; returns a note."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return "numa: unknown"
        if len(bus.split(":")[0]) == 8:          # nvidia-smi prints an 8-digit domain, sysfs uses 4
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return "numa: single node"
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return "numa: node %d (%d cpus)" % (node, len(cpus))
    except Exception as exc:  # noqa: BLE001
        return "numa: not bound (%s)" % type(exc).__name__


# ---------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path -- datasketch.MinHash.bulk from
    oracle/_ref/site when installed (kind "reference"), else its numpy uint64 arithmetic restated in
    oracle/oracle_np.py (kind "port", where no reference was staged) -- on all host cores;
    each step = a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    sample = cpu_sample_docs(args, cores)
    rates, kind = [], "port"
    for i in range(args.warmup + args.steps):
        r, dt, kind, _ = cpu_reference_rate(sample, args.tokens, args.num_perm, cores, repeats=1)
        if i >= args.warmup:
            rates.append((r, dt))
    val = float(max(r for r, _ in rates))           # best step: the least-disturbed one on a shared host
    ms = float(min(dt for _, dt in rates) * 1e3)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, cores),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": cpu_sample_text(sample, args.tokens, cores, kind, [r for r, _ in rates]),
                         "mean": float(np.mean([r for r, _ in rates]))},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import datasketch_b200 as dsk
    from datasketch_b200 import _native as nv
    from datasketch_b200.minhash import _make_permutations

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n, t, k = args.docs, args.tokens, args.num_perm

    # ---- CPU baseline on the same box (rank 0, N=1 only), before CUDA is initialised (fork) --------
    cpu = None
    host_cores = len(os.sched_getaffinity(0))      # before the NUMA binding below narrows the mask
    if rank == 0 and world == 1 and not args.no_cpu:
        sample = cpu_sample_docs(args, host_cores)
        rate, dt, kind, rates = cpu_reference_rate(sample, t, k, host_cores, repeats=3)
        cpu = {"value": rate, "unit": UNIT, "cores": host_cores, "kind": kind,
               "sample": cpu_sample_text(sample, t, host_cores, kind, rates)}

    numa_note = bind_to_gpu_numa_node(local)   # after the CPU baseline (which uses every core)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL_DEBUG keeps whatever level the caller set (the driver reads the communicator lines); its log
        # goes to stderr so that stdout stays the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    perms = _make_permutations(k, 1)

    # ---- synthetic inputs: pinned host copy (for e2e) and resident device copy (for value) ----
    h_tok_t = torch.empty((n, t), dtype=torch.int32, pin_memory=True)
    h_tok = h_tok_t.numpy().view(np.uint32)
    make_tokens(n, t, 1000 + rank, h_tok)
    h_off_t = torch.arange(0, (n + 1) * t, t, dtype=torch.int64).pin_memory()
    h_out_t = torch.empty((n, k), dtype=torch.int32, pin_memory=True)
    d_tok = h_tok_t.to(dev, non_blocking=True)
    d_off = h_off_t.to(dev, non_blocking=True)
    d_out = torch.empty((n, k), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    stream = torch.cuda.current_stream(dev)

    def step_device():
        dsk.engine.bulk_signatures_device(d_tok, d_off, n * t, perms, d_out=d_out, kernel=args.kernel,
                                          stream=stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- value: device-resident, CUDA events ----------------------------------------------------
    BAD = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed_value():
        for _ in range(max(args.warmup, 3)):
            step_device()
        barrier()
        tw0 = time.perf_counter()
        ev0.record(stream)
        for _ in range(args.steps):
            step_device()
        ev1.record(stream)
        barrier()
        tw1 = time.perf_counter()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        return ms, tw0, tw1

    ms_total, t_wall0, t_wall1 = timed_value()
    remeasured = False
    if rank == 0 and world == 1:
        time.sleep(0.05)
        first = sampler.summary(t_wall0, t_wall1)
        if BAD & set(first["reasons"]):      # thermal / hw slowdown seen: re-measure once (timing rules)
            ms_total, t_wall0, t_wall1 = timed_value()
            remeasured = True
    ms_step = ms_total / args.steps
    value = n * world / (ms_step * 1e-3)

    # --dump-outputs: the sampled rows of what each timed leg's last step wrote, taken before the next leg runs
    dump = bool(args.dump_outputs) and rank == 0
    dumped = {}
    if dump:
        rows = dump_rows(n, k)
        d_rows = torch.from_numpy(rows).to(dev)

        def take(name, sig):
            dumped[name] = sig[d_rows].cpu().numpy().view(np.uint32).astype(np.float64)
        take("signatures", d_out)

    # parity spot-check on the benchmark's own output, on EVERY rank (oracle = checker only)
    from oracle import oracle_clib as oc
    idx = np.arange(0, n, max(1, n // 64))[:64]
    got = d_out[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.uint32)
    sub = np.ascontiguousarray(h_tok[idx]).reshape(-1)
    want = oc.minhash_bulk_u32tok(sub, np.arange(len(idx) + 1, dtype=np.int64) * t, perms)
    if not np.array_equal(got, want):
        raise SystemExit("bench: GPU signatures of rank %d differ from the oracle -- number is invalid" % rank)

    # ---- repeated tokens: the same step on documents where 10 % of the positions repeat an earlier token of the same
    # document (multiset input; the reference accepts it, minhash.py:294-297: min is idempotent).  Reported beside the
    # headline so that a regression of the tie handling is visible; parity spot-checked like the headline.
    duplicates = None
    if not args.no_dups:
        d_dup = d_tok.clone()
        v2 = d_dup.view(n, t)
        g = torch.Generator(device=dev).manual_seed(7 + rank)
        pos = torch.arange(t, device=dev)
        for r0 in range(0, n, 65536):
            blk = v2[r0:r0 + 65536]
            rep = (torch.rand(blk.shape, device=dev, generator=g) < 0.1) & (pos > 0)
            src = (torch.rand(blk.shape, device=dev, generator=g) * pos).long()
            blk.copy_(torch.where(rep, torch.gather(blk, 1, src), blk))
        d_out2 = torch.empty_like(d_out)

        def step_dup():
            dsk.engine.bulk_signatures_device(d_dup, d_off, n * t, perms, d_out=d_out2, kernel=args.kernel,
                                              stream=stream.cuda_stream)
        for _ in range(3):
            step_dup()
        barrier()
        ev0.record(stream)
        for _ in range(args.steps):
            step_dup()
        ev1.record(stream)
        barrier()
        ms_d = ev0.elapsed_time(ev1) / args.steps
        if dump:
            take("signatures_repeats", d_out2)
        sub_d = d_dup.view(n, t)[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.uint32).reshape(-1)
        want_d = oc.minhash_bulk_u32tok(np.ascontiguousarray(sub_d), np.arange(len(idx) + 1, dtype=np.int64) * t, perms)
        if not np.array_equal(d_out2[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.uint32), want_d):
            raise SystemExit("bench: signatures of the repeated-token documents differ from the oracle")
        duplicates = {"repeat_share": 0.1, "ms_per_step": ms_d, "value": n / (ms_d * 1e-3), "unit": UNIT + " per GPU",
                      "slowdown_vs_unique": ms_d / ms_step, "rows_verified": True}
        del d_dup, d_out2

    # ---- 64-bit hash values: the same documents with a random high word on every token (minhash.py:294 accepts any hash
    # below 2^64).  The signature kernel's general variant (low-word plane in phase 1, 64-bit form with the conditional
    # subtract only in its exact stage) next to round 1's EXACT kernel, which evaluates the 64-bit form for every
    # (token, permutation); rows spot-checked against the oracle.
    u64_tokens = None
    if not args.no_dups and args.kernel in ("auto", "two_phase"):
        g = torch.Generator(device=dev).manual_seed(11 + rank)
        d_tok64 = torch.randint(0, 1 << 32, (n * t,), device=dev, dtype=torch.int64, generator=g)
        d_tok64.mul_(1 << 32).add_(d_tok.view(-1).to(torch.int64) & 0xFFFFFFFF)   # (hi << 32) | lo, as the bit pattern
        d_out3 = torch.empty_like(d_out)
        res = {}
        for name in ("two_phase", "exact"):
            def step64():
                dsk.engine.bulk_signatures_device(d_tok64, d_off, n * t, perms, d_out=d_out3, kernel=name, stream=stream.cuda_stream)
            for _ in range(2):
                step64()
            barrier()
            ev0.record(stream)
            for _ in range(args.steps):
                step64()
            ev1.record(stream)
            barrier()
            res[name] = ev0.elapsed_time(ev1) / args.steps
            if dump and name == "two_phase":
                take("signatures_u64", d_out3)
            sub64 = d_tok64.view(n, t)[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.uint64).reshape(-1)
            want64 = oc.minhash_bulk_u64tok(np.ascontiguousarray(sub64), np.arange(len(idx) + 1, dtype=np.int64) * t, perms)
            if not np.array_equal(d_out3[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.uint32), want64):
                raise SystemExit("bench: signatures of the 64-bit-token documents (%s) differ from the oracle" % name)
        u64_tokens = {"ms_per_step": res["two_phase"], "value": n / (res["two_phase"] * 1e-3), "unit": UNIT + " per GPU",
                      "slowdown_vs_u32": res["two_phase"] / ms_step, "exact_kernel_ms_per_step": res["exact"],
                      "speedup_vs_exact_kernel": res["exact"] / res["two_phase"], "rows_verified": True,
                      "steps": {"two_phase": args.steps, "exact": args.steps}}
        del d_tok64, d_out3

    # ---- e2e: pinned host buffers through the host C-ABI ------------------------------------------
    e2e = None
    e2e_launches = 0
    if not args.no_e2e:
        h_out = h_out_t.numpy().view(np.uint32)
        h_off = h_off_t.numpy()

        def step_host():
            dsk.engine.bulk_signatures(h_tok.reshape(-1), h_off, perms, kernel=args.kernel, device=local, out=h_out)

        for _ in range(max(2, min(args.warmup, 3))):
            step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        e2e = {"value": n * world * args.steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(h_tok.nbytes + h_off.nbytes) * world,
               "d2h_bytes_per_step": int(h_out.nbytes) * world, "ms_per_step": dt / args.steps * 1e3}
        if not np.array_equal(h_out[idx], want):
            raise SystemExit("bench: host-path signatures of rank %d differ from the oracle -- number is invalid" % rank)
        # the e2e leg's own roofline: the same bytes as bare pinned copies, both directions at once (PCIe duplex)
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        d_scr = torch.empty_like(d_tok)

        def copies():
            with torch.cuda.stream(s_in):
                d_scr.copy_(h_tok_t, non_blocking=True)
            with torch.cuda.stream(s_out):
                h_out_t.copy_(d_out, non_blocking=True)

        keep = h_out[idx].copy()
        copies()
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            copies()
        torch.cuda.synchronize()
        floor_ms = (time.perf_counter() - t0) / 3 * 1e3
        if world > 1:
            tt = torch.tensor([floor_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            floor_ms = float(tt.item())
        e2e["copy_floor_ms"] = floor_ms
        e2e["frac_of_copy_floor"] = floor_ms / e2e["ms_per_step"]
        del d_scr
        assert np.array_equal(h_out[idx], keep)  # d_out holds the same signatures the host path produced
        slices = max(-(-n // (128 << 10)), -(-(n * t) // (16 << 20)))
        e2e_launches = slices * args.steps

    # ---- optional: NCCL all-gather of the signature matrix (assembly for LSH bucketing) -----------
    allgather = None
    if world > 1:
        full = torch.empty((world * n, k), dtype=torch.int32, device=dev)
        for _ in range(2):
            dist.all_gather_into_tensor(full, d_out)
        barrier()
        ev0.record(stream)
        for _ in range(args.steps):
            step_device()
            dist.all_gather_into_tensor(full, d_out)
        ev1.record(stream)
        barrier()
        tt = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_g = float(tt.item()) / args.steps
        allgather = {"value": n * world / (ms_g * 1e-3), "unit": UNIT, "ms_per_step": ms_g,
                     "gathered_bytes_per_gpu": int(full.numel() * 4), "how": "kernel, then NCCL all_gather_into_tensor"}
        # fused variant: the kernel stores every row into all ranks' matrices over NVLink (no NCCL pass)
        try:
            from datasketch_b200.distributed import FusedGather
            del full
            fg = FusedGather(world * n, k, device=local)
            for _ in range(2):
                fg.build(d_tok, d_off, n * t, perms, row_offset=rank * n, kernel=args.kernel)
            barrier()
            ev0.record(stream)
            for _ in range(args.steps):
                fg.build(d_tok, d_off, n * t, perms, row_offset=rank * n, kernel=args.kernel, sync=False)
            ev1.record(stream)
            fg.finish()
            barrier()
            tt = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms_f = float(tt.item()) / args.steps
            ok = bool(torch.equal(fg.buf[rank * n: rank * n + 4096], d_out[:4096]))
            other = (rank + 1) % world
            chk = torch.empty((4096, k), dtype=torch.int32, device=dev)
            src = d_out[:4096].contiguous()
            gl = [torch.empty_like(src) for _ in range(world)]
            dist.all_gather(gl, src)
            ok = ok and bool(torch.equal(fg.buf[other * n: other * n + 4096], gl[other]))
            allgather["fused"] = {"value": n * world / (ms_f * 1e-3), "unit": UNIT, "ms_per_step": ms_f,
                                  "how": "dsk_minhash_bulk_gather: peer stores over NVLink in the kernel epilogue",
                                  "rows_verified": ok}
        except Exception as exc:  # noqa: BLE001  (symmetric memory unavailable on this box)
            allgather["fused"] = {"unavailable": repr(exc)[:200]}

    # ---- strong scaling: the metric's own shape -- args.docs documents IN TOTAL, split over the ranks, timed from
    # tokens-resident to the full [docs, K] signature matrix present on EVERY rank (what LSH bucketing needs) ----
    strong = None
    if world > 1:
        ns = n // world
        d_off_s = d_off[: ns + 1]
        d_out_s = torch.empty((ns, k), dtype=torch.int32, device=dev)

        def timed(fn):
            for _ in range(3):
                fn()
            barrier()
            ev0.record(stream)
            for _ in range(args.steps):
                fn()
            ev1.record(stream)
            barrier()
            tt = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()) / args.steps

        full_s = torch.empty((world * ns, k), dtype=torch.int32, device=dev)

        def step_build():
            dsk.engine.bulk_signatures_device(d_tok, d_off_s, ns * t, perms, d_out=d_out_s, kernel=args.kernel,
                                              stream=stream.cuda_stream)

        def step_nccl():
            step_build()
            dist.all_gather_into_tensor(full_s, d_out_s)

        ms_b = timed(step_build)
        ms_n = timed(step_nccl)
        strong = {"docs_total": ns * world, "unit": UNIT,
                  "build_only": {"value": ns * world / (ms_b * 1e-3), "ms_per_step": ms_b,
                                 "how": "each rank's %d-document shard, signatures stay sharded" % ns},
                  "nccl": {"value": ns * world / (ms_n * 1e-3), "ms_per_step": ms_n,
                           "how": "kernel, then NCCL all_gather_into_tensor"},
                  "gathered_bytes_received_per_gpu": int((world - 1) * ns * k * 4)}
        try:
            from datasketch_b200.distributed import FusedGather
            fgs = FusedGather(world * ns, k, device=local)

            def step_fused():   # build + peer stores, then a device-side cross-rank barrier: the matrix is complete
                fgs.build(d_tok, d_off_s, ns * t, perms, row_offset=rank * ns, kernel=args.kernel, sync=False)
                fgs.hdl.barrier()

            ms_s = timed(step_fused)
            other = (rank + 1) % world
            ok = bool(torch.equal(fgs.buf[rank * ns: rank * ns + 4096], d_out_s[:4096]))
            ok = ok and bool(torch.equal(fgs.buf[other * ns: other * ns + 4096], full_s[other * ns: other * ns + 4096]))
            strong["fused"] = {"value": ns * world / (ms_s * 1e-3), "ms_per_step": ms_s, "rows_verified": ok,
                               "how": "dsk_minhash_bulk_gather (peer stores in the kernel epilogue) + device barrier"}
            del fgs
        except Exception as exc:  # noqa: BLE001
            strong["fused"] = {"unavailable": repr(exc)[:200]}
        best = max((v for v in (strong["nccl"], strong.get("fused", {})) if "value" in v), key=lambda v: v["value"])
        strong["value"], strong["ms_per_step"] = best["value"], best["ms_per_step"]
        # every rank must RECEIVE (world-1)/world of the matrix over NVLink: that, not the integer math, bounds it
        link = 770.0   # GB/s per direction per GPU, measured peer copy (B200_PROFILING.md)
        strong["link_floor_ms"] = strong["gathered_bytes_received_per_gpu"] / (link * 1e9) * 1e3
        strong["limit"] = ("receive side of the gather: %.0f MB per GPU at %.0f GB/s = %.2f ms, vs %.2f ms of kernel"
                           % (strong["gathered_bytes_received_per_gpu"] / 1e6, link, strong["link_floor_ms"], ms_b))
        del full_s, d_out_s
    else:
        strong = {"docs_total": n, "unit": UNIT, "value": value, "ms_per_step": ms_step,
                  "how": "N=1: the device-resident step itself (no exchange)"}

    if rank == 0:
        sampler.stop()
    clocks = sampler.summary(t_wall0, t_wall1) if rank == 0 else None
    if clocks is not None:
        clocks["remeasured"] = remeasured
        if clocks["samples"] < 3:   # the timed region is only tens of ms: add the samples of the whole run under load
            wide = sampler.summary(t_wall0 - 0.2, time.perf_counter())
            clocks["sm_mhz_whole_run"] = wide["sm_mhz"]
            clocks["reasons"] = sorted(set(clocks["reasons"]) | set(wide["reasons"]))
            clocks["samples_whole_run"] = wide["samples"]

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak = float(json.load(open(peaks_path))["hbm_gbs"])
            peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        alg_bytes = (4 * t + 4 * k) * n  # per launch, per GPU
        achieved = alg_bytes / (ms_step * 1e-3) / 1e9
        traffic = None  # DRAM bytes per launch from the committed ncu --set full capture of this kernel/workload
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        h = nv.perm_handle(perms, local)
        kern = args.kernel if args.kernel != "auto" else ("two_phase" if h.n_unsafe == 0 else "exact")
        if os.path.exists(tpath):
            ent = json.load(open(tpath)).get("%s|%dx%dxK%d" % (KERNEL_NAMES[kern], n, t, k))
            if ent:
                traffic = ent["traffic_bytes_per_launch"] / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64 (mod 2^64 wrap, mod 2^61-1) on u32 lanes", "data": "synthetic",
            "config": workload_config(args, host_cores),
            "kernel": KERNEL_NAMES[kern], "host": numa_note,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_unit": "GB per launch (ncu dram read+write; algorithmic %.3f GB)"
                                                             % (alg_bytes / 1e9), "peak_source": peak_src,
                         "note": "binding roof is the integer pipe (T*K evaluations/doc), see DESIGN.md"},
            "e2e": e2e, "clocks": clocks,
            # the two-phase path launches minhash_sig_kernel twice per device-resident step (documents, then the piece
            # table of long documents -- empty here, an idle launch); the host pipeline launches it once per slice
            "gpu_launches": (2 if kern == "two_phase" else 1) * args.steps * (1 if duplicates is None else 2) + e2e_launches
                            + (0 if u64_tokens is None else 3 * args.steps),
        }
        # the roof that actually binds this kernel: one 32-bit IMAD per (token, permutation) evaluation is the floor
        # of any exact scheme, and B200 issues IMAD at 16 lanes/clk/SMSP = 64 lanes/clk/SM (profiles/, DESIGN.md 5)
        sm_count = nv.device_info(local)["sm_count"]
        clk_mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
        evals_per_s = float(n) * t * k / (ms_step * 1e-3)
        imad_peak = sm_count * 64 * clk_mhz * 1e6
        line["int_pipe"] = {"bound": "imad (fmaheavy pipe)", "achieved": evals_per_s, "peak": imad_peak,
                            "unit": "evaluations/s per GPU", "frac": evals_per_s / imad_peak,
                            "note": "peak = SMs x 64 IMAD lanes/clk x SM clock under load; 1 IMAD per evaluation minimum"}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if allgather is not None:
            line["allgather"] = allgather
        line["strong"] = strong
        if duplicates is not None:
            line["duplicates"] = duplicates
        if u64_tokens is not None:
            line["u64_tokens"] = u64_tokens
        print(json.dumps(line), flush=True)
    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
        dumped["rows"] = rows.astype(np.float64)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
