#!/usr/bin/env python
"""bench.py — POST label throughput (labels/s) of the B200 engine, per the driver's contract.

Workload (BASELINE.json configs[1]): 4-SU init, scrypt N = 8192, r = p = 1, single B200, labels
discarded ("/dev/null").  One *step* = one batch of `--batch` consecutive labels of the 2^34-label
index space (default: 72 layers of resident scratchpads ~ 5.5 M labels ~ 3 s, so that the driver's 20 steps sample
~10^8 labels / a minute of steady state per arm; the reference's default ComputeBatchSize is 2^20), exactly what one `initialize(start, end)`
call of the reference's initializer does per ComputeBatchSize batch (activation/post.go:295).

  value      labels/s with the output resident in HBM (b200post_labels_range_dev), device-timed
  e2e        labels/s through the host-buffer C-ABI call (b200post_labels_range): commitment H2D and
             16 B/label D2H inside the timed region
  roofline   the ROMix kernel against the measured HBM copy bandwidth; algorithmic bytes =
             2*128*N + 16 = 2 097 168 B/label (SURVEY.md §8d)
  cpu_baseline  the oracle port on this box's host cores (bounded sample)

N > 1 (torchrun): one process per GPU, contiguous index shards, no data-path collective; the only
exchange is an NCCL all-gather of one 48-byte VRF candidate per rank per step (SURVEY.md §8e).

`--impl reference` times the CPU oracle (the reference's own provider cannot be built here:
DESIGN.md §3) on rank 0 only.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step of each arm returned to its caller
(every 8th of its first 2^21 labels and the VRF nonce candidate) as float .npy files, so that two builds can be
compared output for output on identical inputs.  The sampled label indices are fixed: they depend neither on the
batch (as long as it holds 2^21 labels) nor on --steps, so a wave size that differs with free HBM or occupancy moves none.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_SCRYPT = 8192
BYTES_PER_LABEL = 2 * 128 * N_SCRYPT + 16          # algorithmic HBM bytes per label (SURVEY.md §8d)
NUM_LABELS_4SU = 4 * 2**32
METRIC = "POST labels/sec (scrypt N=8192 init)"
ALU_OPS_PER_BLOCKMIX = 553                         # alu-pipe SASS instructions per BlockMix of the shipped kernel (profiles/)
HBM_FALLBACK_GBS = 6650.0                          # /opt/skills/guides/B200_PROFILING.md fallback
# Each arm's last step starts at a fixed index of the rank's shard and its earlier steps lie contiguously below it, so
# consecutive calls continue one another (the engine pre-fills the first layer of the range that follows a call).  The
# default batch follows the engine's wave size (free HBM, occupancy); anchoring the last step keeps its first labels at
# the same indices whatever the wave.  Each arm stays inside one 2^32-aligned window for ~780 steps of 5.5 M labels.
DEV_LAST_START, E2E_LAST_START = 2**33 - 2**26, 2**34 - 2**26
DUMP_SPAN, DUMP_EVERY = 1 << 21, 8                 # --dump-outputs keeps every 8th label of a step's first 2^21: 2^18 rows


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            try:
                pw.append(float(f[2]))
            except ValueError:
                pass
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort(); pw.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": pw[len(pw) // 2] if pw else None,          # median board power during the timed region
                "samples": len(sm), "reasons": sorted(reasons)}


def best_thread_count(orc, commitment: bytes):
    """The oracle is DRAM-latency bound (1 MiB scratchpad per thread) and the box may cap CPU time below
    its visible core count: use the thread count that gives the highest labels/s on a short probe."""
    avail = orc.default_threads()
    L = orc.lib()
    default_impl = L.oracle_get_impl()
    best = (1, 0.0, default_impl)
    # ROMix implementations: the default (AVX2, two labels per thread) and, where the CPU has it, AVX-512 with four
    # labels per thread, which is faster per thread but needs 4 MiB of cache per thread
    for impl in sorted({default_impl, 3}):
        if L.oracle_set_impl(impl) != 0:
            continue
        t = avail
        while t >= 1:
            probe = max(t * 16, 64)
            rate = probe / orc.c_time_labels(commitment, N_SCRYPT, 0, probe, t)
            if rate > best[1]:
                best = (t, rate, impl)
            if t == 1:
                break
            t = max(t // 2, 1)
    L.oracle_set_impl(best[2])       # stays selected for the timed sample; results are identical (tests/test_oracle.py)
    return best[0], best[1]


def cpu_baseline(orc, seconds_target: float = 10.0) -> dict:
    """Oracle port timed on all host cores on a bounded sample of the same workload."""
    commitment = bytes(range(32))
    cores, rate = best_thread_count(orc, commitment)
    # calibrate on ~2 s (the short probe flatters a box whose visible cores are not all its own), then sample ~seconds_target
    cal = int(max(cores * 8, rate * 2.0))
    rate = cal / orc.c_time_labels(commitment, N_SCRYPT, 1 << 19, cal, cores)
    sample = int(max(cores * 32, min(rate * seconds_target, 1 << 20)))
    t = orc.c_time_labels(commitment, N_SCRYPT, 1 << 20, sample, cores)
    return {"value": sample / t, "unit": "labels/s", "cores": cores, "kind": "port",
            "sample": f"{sample} labels of the N=8192 init (oracle/post_oracle.c, ROMix impl {orc.lib().oracle_get_impl()} "
                      f"[2 = AVX2 x2 labels, 3 = AVX-512 x4], {cores} pthreads, {t:.1f} s)"}


def _valid_proofs(b2, vf, pr, provider: int, n_identities: int, k2: int, labels_per_id: int, k1: int):
    """Real valid proofs at N = 8192: each identity's small POST (labels_per_id labels) is initialised on the GPU and proven
    with the product's scan; the verifier must accept them.  Returns [(Proof, ProofMetadata)]."""
    import numpy as np
    rng = np.random.default_rng(11)
    out = []
    for _ in range(n_identities):
        node_id, atx, ch = (bytes(rng.integers(0, 256, 32, dtype=np.uint8)) for _ in range(3))
        labels, _ = b2.labels_range(b2.commitment(node_id, atx), N_SCRYPT, 0, labels_per_id, provider=provider)
        nonce, packed, pow_, _ = pr.prove_scan(labels, ch, 16, [0], k1, k2, labels_per_id, provider=provider)
        out.append((vf.Proof(nonce, packed, pow_), vf.ProofMetadata(node_id, atx, ch, 1, labels_per_id)))
    return out


def bench_verify(b2, provider: int, orc=None, n_proofs: int = 10000, k2: int = 37) -> dict:
    """BASELINE.json configs[2]: PostVerifier batch, 10 000 proofs x K2 = 37 indices, N = 8192, one B200.
    MIXED batch: half the proofs are VALID (real proofs of small POSTs initialised and proven on this GPU, repeated),
    half have one index bumped (systest/tests/distributed_post_verification_test.go:254-256) and are rejected at a known
    position.  Timed end to end through b200post_verify_batch with host buffers: index unpack + key derivation (host),
    H2D, gather kernels, on-device AES verdict, D2H.  `with_k2pow` adds the RandomX check of every proof (device).
    The CPU side is MEASURED: the oracle recomputes the K2 labels of a sample of the same proofs on all host cores and
    judges them (what verifying.ProofVerifier.Verify does per proof on NumCPU/2 workers, activation/post.go:101-111)."""
    import numpy as np
    vf = importlib.import_module("go-spacemesh_b200.verify")
    pr = importlib.import_module("go-spacemesh_b200.prove")
    labels_per_id, k1 = 4096, 96
    bits = vf.bits_per_index(labels_per_id)
    base = _valid_proofs(b2, vf, pr, provider, 48, k2, labels_per_id, k1)
    params = vf.VerifyParams(k1=k1, k2=k2, scrypt_n=N_SCRYPT)
    proofs, metas, expect_bad = [], [], []
    for i in range(n_proofs):
        p, m = base[i % len(base)]
        if i % 2 == 0:
            proofs.append(p); expect_bad.append(None)
        else:
            idx = vf.unpack_indices(p.indices, bits, k2)
            pos = (i // 2) % k2
            idx[pos] = (idx[pos] + 1) % labels_per_id
            proofs.append(vf.Proof(p.nonce, vf.pack_indices(idx, bits), p.pow)); expect_bad.append(pos)
        metas.append(m)
    batch = vf.PreparedBatch(proofs, metas, params)     # C structs built once: the timed region is the C-ABI call
    warm_walls = []
    for _ in range(2):      # warm-up at full size: grow-only judge buffers sized, any speculative init layer drained
        t0 = time.perf_counter()
        batch.run(provider, "skip")
        warm_walls.append(time.perf_counter() - t0)

    def stage_us():
        out = {}
        for ln in b2.metrics_text().splitlines():
            for key in ("verify_prepare_us_total", "verify_gather_judge_us_total"):
                if ln.startswith("b200post_" + key + " "):
                    out[key] = float(ln.split()[1])
        return out
    launches0 = b2.launch_count()
    s0 = stage_us()
    t0 = time.perf_counter()
    st, bad = batch.run(provider, "skip")
    wall = time.perf_counter() - t0
    s1 = stage_us()
    n_valid = sum(1 for x in st if x == 0)
    # a tampered index may still qualify by chance (probability ~ k1 / labels): only rejected ones must name the position
    positions_ok = all(e is None or s == 0 or b == e for s, b, e in zip(st, bad, expect_bad))
    valid_ok = all(s == 0 for s, e in zip(st, expect_bad) if e is None)
    # with the k2pow (RandomX) check of every proof on the device; pow_difficulty = ff..ff so that verdicts do not change
    batch.run(provider, "builtin")
    t0 = time.perf_counter()
    st_pow, _ = batch.run(provider, "builtin")
    wall_pow = time.perf_counter() - t0
    # latency of small batches (one proof per Verify call is the reference's shape, activation/post_verifier.go:303-350)
    latency = []
    for n in (1, 16, 256):
        small = vf.PreparedBatch(proofs[:n], metas[:n], params)
        small.run(provider, "skip")
        best = min(_timed(lambda: small.run(provider, "skip")) for _ in range(3))
        latency.append({"proofs": n, "ms": 1e3 * best, "gpu_device_ms": b2.last_call_ms(provider)})
    res = {"workload": f"{n_proofs} proofs x K2={k2}, N=8192: 50 % valid (real proofs of {len(base)} small POSTs, repeated), 50 % with one index bumped",
           "proofs": n_proofs, "k2": k2, "labels_recomputed": n_proofs * k2, "seconds": wall,
           "proofs_per_s": n_proofs / wall, "labels_per_s": n_proofs * k2 / wall,
           "valid": n_valid, "invalid": n_proofs - n_valid, "valid_proofs_all_accepted": valid_ok,
           "rejected_at_the_bumped_position": positions_ok,
           "gpu_device_ms": b2.last_call_ms(provider),
           "host_prepare_ms": (s1.get("verify_prepare_us_total", 0) - s0.get("verify_prepare_us_total", 0)) / 1e3,
           "gather_judge_wall_ms": (s1.get("verify_gather_judge_us_total", 0) - s0.get("verify_gather_judge_us_total", 0)) / 1e3,
           "gpu_launches": int(b2.launch_count() - launches0), "warmup_seconds": warm_walls,
           "with_k2pow": {"seconds": wall_pow, "proofs_per_s": n_proofs / wall_pow, "same_verdicts": list(st_pow) == list(st),
                          "note": "one RandomX hash per proof on the device, all proofs of the batch in one k2pow batch"},
           "latency": latency,
           "note": "verdict conventions (AES keys, index packing, K3 subset) unpinned (DESIGN.md §2); label function pinned"}
    if orc is not None:
        # measured CPU verifier: K2 label recomputations of a sample of the SAME proofs on all host cores + the judge
        sample = 256
        comms = np.concatenate([np.tile(np.frombuffer(orc.py_commitment(metas[i].node_id, metas[i].commitment_atx_id), dtype=np.uint8), (k2, 1))
                                for i in range(sample)])
        idxs = np.array([v for i in range(sample) for v in vf.unpack_indices(proofs[i].indices, bits, k2)], dtype=np.uint64)
        threads = orc.default_threads()
        orc.c_labels_gather(comms[:threads], idxs[:threads], N_SCRYPT, threads=threads)        # thread start-up, page faults
        t0 = time.perf_counter()
        labs = orc.c_labels_gather(comms, idxs, N_SCRYPT, threads=threads)
        cpu_wall = time.perf_counter() - t0
        diff = orc.py_proving_difficulty(k1, labels_per_id)
        verdicts = [all(orc.py_label_passes(labs[i * k2 + j].tobytes(), metas[i].challenge, proofs[i].nonce, proofs[i].pow, diff) for j in range(k2))
                    for i in range(sample)]
        res["cpu_baseline"] = {"proofs_per_s": sample / cpu_wall, "cores": threads, "kind": "port", "measured": True,
                               "sample": f"{sample} of the same proofs: their {sample * k2} labels recomputed by oracle/post_oracle.c on {threads} threads "
                                         f"({cpu_wall:.2f} s); the per-label AES judge (< 0.1 % of a CPU verifier's work) is checked, not timed",
                               "verdicts_equal_gpu": verdicts == [s == 0 for s in st[:sample]]}
    return res


def _timed(fn) -> float:
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def dump_outputs(out_dir: str, arm: str, labels, index, vrf) -> None:
    """DIR/<arm>_*.npy: sampled labels (uint8[rows, 16] as float32), their label indices and the VRF nonce candidate
    (index, or -1 when there is none, and its 32-byte label, zeros when there is none) as float64 / float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"labels": labels.astype(np.float32), "label_index": index.astype(np.float64),
              "vrf_index": np.array([vrf[0] if vrf else -1], dtype=np.float64),
              "vrf_label32": np.frombuffer(vrf[1] if vrf else bytes(32), dtype=np.uint8).astype(np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{arm}_{name}.npy"), a)


def bench_k2pow(b2, provider: int, with_cpu: bool) -> dict:
    """BASELINE.json configs[4] on one GPU: k2pow (RandomX) nonce search over one challenge, difficulty 0 so that nothing
    stops it early; hashes/s over whole device batches (device time from the engine's CUDA events), dataset resident.
    CPU side: the oracle port (interpreter, fast mode, all host threads) on a bounded sample."""
    import numpy as np
    k2 = importlib.import_module("go-spacemesh_b200.k2pow")
    rng = np.random.default_rng(5)
    ch, node = bytes(rng.integers(0, 256, 8, dtype=np.uint8)), bytes(rng.integers(0, 256, 32, dtype=np.uint8))
    t0 = time.perf_counter()
    k2.prepare(provider=provider)
    dataset_s = time.perf_counter() - t0
    n = k2.batch_size(provider)
    k2.search(0, ch, node, b"\x00" * 32, 0, n, provider=provider)          # warm-up batch
    launches0 = b2.launch_count()
    found, done = k2.search(0, ch, node, b"\x00" * 32, n, 2 * n, provider=provider)
    tm = k2.last_timing(provider)
    sample = k2.hashes(0, ch, node, 3 * n, 32, provider=provider)
    res = {"workload": "k2pow nonce search, one challenge, difficulty 0 (no early exit), RandomX fast mode (2080 MiB dataset in HBM)",
           "hashes": done, "hashes_per_s": done / (tm["total_ms"] / 1e3), "device_ms": tm["total_ms"], "vm_kernel_ms": tm["vm_kernel_ms"],
           "vm_kernel_share": tm["vm_kernel_ms"] / tm["total_ms"], "batch": n, "batch_latency_ms": tm["total_ms"] / max(1, done // n),
           "scratchpad_gib": n * 2 / 1024, "dataset_build_s": dataset_s, "gpu_launches": int(b2.launch_count() - launches0),
           "vm_mode": b2.get_option("rx_vm_mode"),
           "parity": "RandomX pinned on its official vectors through this engine (tests/test_gpu_k2pow.py); k2pow input layout unpinned"}
    if with_cpu:
        from oracle import pyrandomx as orx
        c = orx.Cache(orx.K2POW_CACHE_KEY)
        try:
            threads = orx.default_threads()
            t0 = time.perf_counter(); c.init_dataset(threads); ds = time.perf_counter() - t0
            probe, _, secs = c.k2pow_scan(0, ch, node, 3 * n, 32, threads=min(32, threads))
            res["sample_equals_oracle"] = bool((probe == sample).all())
            _, _, secs = c.k2pow_scan(0, ch, node, 0, 4 * threads, threads=threads, want_hashes=False)       # calibration
            count = int(max(threads * 4, min(4 * threads / secs * 8.0, 1 << 16)))
            _, _, secs = c.k2pow_scan(0, ch, node, 4 * threads, count, threads=threads, want_hashes=False)
            res["cpu_baseline"] = {"hashes_per_s": count / secs, "cores": threads, "kind": "port",
                                   "sample": f"{count} hashes, oracle/randomx_oracle.c (interpreter, AES-NI, fast mode; dataset built in {ds:.1f} s), {secs:.1f} s"}
        finally:
            c.close()
    return res


def run_reference(args, rank: int, world: int) -> None:
    """--impl reference: the CPU oracle (port) on rank 0; other ranks exit 0 without work."""
    if rank != 0:
        return
    from oracle import pyoracle as orc
    orc.build()
    commitment = bytes(range(32))
    cores, rate = best_thread_count(orc, commitment)
    # bounded sample per step: ~2 s of work at the probed rate, a whole number of 4-label groups per thread
    per_step = max(cores * 64, int(rate * 2.0) // (4 * cores) * (4 * cores), 256)
    for w in range(args.warmup):
        orc.c_time_labels(commitment, N_SCRYPT, w * per_step, min(per_step, cores * 8), cores)
    t_total = 0.0
    for s in range(args.steps):
        t_total += orc.c_time_labels(commitment, N_SCRYPT, (1 << 24) + s * per_step, per_step, cores)
    value = per_step * args.steps / t_total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "labels/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "4-SU POST init (2^34 labels), scrypt-jane (ChaCha20/8 + Keccak-512) N=8192 r=1 p=1, labels discarded",
                       "step": f"bounded sample: {per_step} labels per step on {cores} host threads"},
            "cpu_baseline": {"value": value, "unit": "labels/s", "cores": cores, "kind": "port",
                             "sample": f"{per_step} labels/step x {args.steps} steps, oracle/post_oracle.c, ROMix impl "
                                       f"{orc.lib().oracle_get_impl()} [2 = AVX2 x2 labels, 3 = AVX-512 x4]"},
            "e2e": {"value": value, "unit": "labels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="labels per step per GPU (0 = 72 layers of resident scratchpads ~ 5.5 M labels ~ 3 s: 20 steps sample ~ 10^8 labels / 60 s of steady state, SURVEY.md §8d cfg2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the configs[2] verify-batch measurement")
    ap.add_argument("--no-k2pow", action="store_true", help="skip the configs[4] k2pow (RandomX) measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs of each arm to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        print("bench.py: --dump-outputs ignored: the reference arm times the oracle, which returns no labels",
              file=sys.stderr)
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    b2 = importlib.import_module("go-spacemesh_b200")
    if not b2.LIB_PATH.exists():
        raise SystemExit("libb200post.so missing: run __graft_entry__.build() (no fallback path exists)")
    if not torch.cuda.is_available() or not b2.providers():
        raise SystemExit("bench.py needs a CUDA device: the label engine has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # the contract is ONE JSON line on stdout: libraries that print there (NCCL announces its version on stdout when
    # NCCL_DEBUG is set in the environment) are sent to stderr for the duration of the run
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    prov = b2.providers()[local_rank]
    commitment = b2.commitment(bytes(range(32)), bytes(range(32, 64)))
    diff = b2.vrf_difficulty(NUM_LABELS_4SU * world)

    wave = b2.wave_slots(N_SCRYPT, provider=local_rank)                    # resident scratchpads per wave
    tpb = b2.get_option("tpb")
    batch = args.batch or 72 * wave
    d_out = torch.empty((batch, 16), dtype=torch.uint8, device=dev)        # labels stay in HBM for `value`
    h_out = np.empty((batch, 16), dtype=np.uint8)                          # host sink for `e2e`

    # steps: the device-resident arm's warm-up and timed steps, two e2e warm-up steps that continue them, a gap, then
    # the e2e timed steps
    dev_last = args.warmup + args.steps - 1
    e2e_first = 2 * args.warmup + args.steps + 2
    e2e_last = e2e_first + args.steps - 1

    def shard_start(step: int) -> int:
        # weak scaling: every rank initialises its own contiguous slice of a (4*world)-SU space
        last, last_start = (dev_last, DEV_LAST_START) if step < e2e_first else (e2e_last, E2E_LAST_START)
        return rank * NUM_LABELS_4SU + last_start + (step - last) * batch

    sharding = importlib.import_module("go-spacemesh_b200.sharding")

    def exchange(vrf):
        """The path's only exchange step: min-reduction of the VRF nonce candidate over ranks
        (one 48-byte record per rank, NCCL all_gather + local lexicographic min)."""
        return sharding.allgather_vrf(vrf, device=dev) if world > 1 else vrf

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps: int, first_step: int):
        """EXACTLY K steps bracketed by barrier + synchronize on both sides.  Returns, max over ranks:
        (wall seconds, ms between two CUDA events recorded on the engine's launching stream around the K
        steps — gaps between calls included, ms summed over the calls alone)."""
        barrier()
        b2.timer_mark(0, local_rank)
        t0 = time.perf_counter()
        calls_ms = 0.0
        for s in range(steps):
            fn(first_step + s)
            calls_ms += b2.last_call_ms(local_rank)
        b2.timer_mark(1, local_rank)
        barrier()
        el = time.perf_counter() - t0
        bracket_ms = b2.timer_elapsed_ms(local_rank)
        if world > 1:
            t = torch.tensor([el, bracket_ms, calls_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            el, bracket_ms, calls_ms = float(t[0]), float(t[1]), float(t[2])
        return el, bracket_ms, calls_ms

    debug = bool(os.environ.get("B200POST_BENCH_DEBUG"))
    last_vrf = {}                                                          # arm -> the VRF candidate of its latest step

    def step_dev(s: int):
        t_a = time.perf_counter()
        vrf = b2.labels_range_dev(commitment, N_SCRYPT, shard_start(s), batch, d_out.data_ptr(), provider=local_rank,
                                  vrf_difficulty_=diff)
        t_b = time.perf_counter()
        last_vrf["dev"] = exchange(vrf)
        if debug:
            print(f"[rank {rank}] step {s}: call {1e3 * (t_b - t_a):.1f} ms (device {b2.last_call_ms(local_rank):.1f}), "
                  f"exchange {1e3 * (time.perf_counter() - t_b):.1f} ms", file=sys.stderr, flush=True)

    def step_e2e(s: int):
        nonce = b2.VrfNonce()
        import ctypes
        rc = b2.lib().b200post_labels_range(local_rank, commitment, N_SCRYPT, shard_start(s), batch, h_out.ctypes.data,
                                            ctypes.cast(ctypes.c_char_p(diff), ctypes.c_void_p), ctypes.byref(nonce), None)
        if rc:
            raise RuntimeError(b2.lib().b200post_last_error().decode())
        last_vrf["e2e"] = exchange((int(nonce.index), bytes(nonce.label32)) if nonce.found else None)

    # ---- device-resident arm (value)
    for w in range(args.warmup):
        step_dev(w)
    b2.romix_time(provider=local_rank, reset=True)
    launches0 = b2.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    wall, dev_ms, calls_ms = timed(step_dev, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    launches = b2.launch_count() - launches0
    romix_ms, romix_k, romix_labels = b2.romix_time(provider=local_rank, reset=True)
    dump = bool(args.dump_outputs) and rank == 0
    if dump:            # the same rows of both arms' last steps; they do not depend on the batch once it is >= DUMP_SPAN
        rows = np.arange(0, min(batch, DUMP_SPAN), DUMP_EVERY)
        dump_outputs(args.dump_outputs, "dev", d_out[torch.from_numpy(rows).to(dev)].cpu().numpy(),
                     shard_start(dev_last) + rows, last_vrf["dev"])

    # ---- end-to-end arm (host buffers through the reference-facing C-ABI call)
    for w in range(2):
        step_e2e(args.warmup + args.steps + w)
    wall_e2e, dev_ms_e2e, _ = timed(step_e2e, args.steps, e2e_first)
    if dump:
        dump_outputs(args.dump_outputs, "e2e", h_out[rows], shard_start(e2e_last) + rows, last_vrf["e2e"])

    total_labels = batch * args.steps * world
    # device-event time is the clock for `value` (max over ranks); wall clock is the cross-check
    value = total_labels / (dev_ms / 1e3) if dev_ms > 0 else total_labels / wall
    value_wall = total_labels / wall
    e2e_value = total_labels / wall_e2e

    peak, peak_src = measured_peaks()
    labels_per_launch = romix_labels / max(romix_k, 1)     # label-equivalents per ROMix launch (engine-counted)
    romix_avg_ms = romix_ms / max(romix_k, 1)
    achieved = labels_per_launch * BYTES_PER_LABEL / (romix_avg_ms / 1e3) / 1e9 if romix_avg_ms > 0 else 0.0
    # dram__bytes of one launch comes from an `ncu --set full` capture (a number measured under ncu is never a bench value,
    # so it cannot be taken live here); the file records which build it was captured on
    traffic, traffic_src = None, None
    tfile = ROOT / "profiles" / "romix_dram_bytes_per_launch.json"
    if tfile.exists():
        try:
            tj = json.loads(tfile.read_text())
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("captured_on", "build not recorded in the file")
        except Exception:  # noqa: BLE001
            traffic = None

    verify_extra = None
    k2pow_extra = None
    if world == 1 and not args.no_k2pow:          # before verify: its builtin pow check would otherwise have built the dataset already
        k2pow_extra = bench_k2pow(b2, local_rank, with_cpu=not args.no_cpu_baseline)
    if world == 1 and not args.no_verify:
        orc_mod = None
        if not args.no_cpu_baseline:
            from oracle import pyoracle as orc_mod
            orc_mod.build()
        verify_extra = bench_verify(b2, local_rank, orc_mod)

    # ALU ceiling probe (N = 1 only): the same ROMix arithmetic with no scratchpad traffic ("nomem" variant; its
    # outputs are not labels).  The label kernel is integer-issue-bound, so this — not the HBM peak — is the
    # ceiling its instruction stream can reach on this device at this clock (DESIGN.md §4).
    alu_probe = None
    if world == 1:
        keep = {k: b2.get_option(k) for k in ("romix_variant", "tpb")}
        try:
            b2.set_option("romix_variant", 3); b2.set_option("tpb", 128)
            slots = b2.wave_slots(N_SCRYPT, provider=local_rank)
            b2.labels_range(commitment, N_SCRYPT, 0, slots, provider=local_rank, discard=True)
            b2.romix_time(provider=local_rank, reset=True)
            b2.labels_range(commitment, N_SCRYPT, slots, 3 * slots, provider=local_rank, discard=True)
            ms, k, lab = b2.romix_time(provider=local_rank, reset=True)
            alu_probe = lab / (ms / 1e3)
        finally:
            for k_, v_ in keep.items():
                b2.set_option(k_, v_)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "labels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "4-SU POST init (2^34 labels/GPU), scrypt-jane (ChaCha20/8 + Keccak-512) N=8192 r=1 p=1, labels discarded (/dev/null sink)",
                       "labels_per_step_per_gpu": batch, "wave_slots": wave, "provider": prov["model"],
                       "romix_variant": b2.get_option("romix_variant"), "rotate_mask": b2.get_option("rotate_mask"),
                       "tpb": tpb, "l2": "working set = wave_slots x 1 MiB scratch >> 126 MB L2; every step uses fresh indices",
                       "parallelism": f"index-range shards x{world}, NCCL all-gather of one 48-B VRF record per step" if world > 1 else "single GPU",
                       "timer": "two CUDA events on the engine's launching stream bracketing the K steps (barrier + synchronize on both sides), max over ranks",
                       "value_from_call_times_only": total_labels / (calls_ms / 1e3) if calls_ms > 0 else None,
                       "value_wall_clock": value_wall},
            "e2e": {"value": e2e_value, "unit": "labels/s", "h2d_bytes_per_step": 32 + 32, "d2h_bytes_per_step": batch * 16 + 48},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "romix_pipe_kernel" if b2.get_option("romix_variant") == 4 else "romix_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         # integer roofline of the label function: 2N BlockMix x 553 alu-pipe instructions (512 XOR/rotate
                         # of two ChaCha20/8 cores + 41 XOR/address, counted in the SASS) = 9.06 M per label, at the
                         # measured 64 ops/clk/SM (profiles/r01_alubench.log) and the maximum SM clock
                         "int_roofline_labels_per_s": prov["sm_count"] * 64 * (clocks["sm_mhz"] * 1e6 if clocks and clocks.get("sm_mhz") else 1.965e9) / (16384 * ALU_OPS_PER_BLOCKMIX),
                         "int_roofline_at_max_clock_labels_per_s": prov["sm_count"] * 64 * (clocks["sm_max_mhz"] * 1e6 if clocks and clocks.get("sm_max_mhz") else 1.965e9) / (16384 * ALU_OPS_PER_BLOCKMIX),
                         "int_roofline_clock": "median SM clock sampled during the timed region" if clocks and clocks.get("sm_mhz") else "nominal 1.965 GHz (no nvidia-smi sample)",
                         "alu_ceiling_labels_per_s": alu_probe,
                         "frac_of_alu_ceiling": (labels_per_launch / (romix_avg_ms / 1e3) / alu_probe) if alu_probe and romix_avg_ms > 0 else None,
                         "bytes_per_label": BYTES_PER_LABEL, "labels_per_launch": labels_per_launch,
                         "avg_launch_ms": romix_avg_ms, "launches_timed": int(romix_k),
                         "kernel_share_of_step": (romix_ms / calls_ms) if calls_ms else None},
            "clocks": clocks,
        }
        if clocks and clocks.get("power_w"):      # rank 0's board power x ranks: every rank runs the same kernel on the same part
            line["labels_per_joule"] = value / (clocks["power_w"] * world)
        if verify_extra:
            line["verify"] = verify_extra
        if k2pow_extra:
            line["k2pow"] = k2pow_extra
        if not args.no_cpu_baseline and world == 1:      # the CPU baseline is an N = 1 measurement
            from oracle import pyoracle as orc
            orc.build()
            line["cpu_baseline"] = cpu_baseline(orc)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
