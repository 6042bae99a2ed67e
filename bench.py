#!/usr/bin/env python
"""bench.py — the driver-facing benchmark of the B200 state-root engine.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py ... --dump-outputs DIR       (also write what the last timed step computed as DIR/<name>.npy)

Headline workload (BASELINE.json configs[1], "C2"): batch keccak256 of 10M 32-byte keys per GPU — the
AccountHashing / StorageHashing inner loop.  One step = one pass over the batch.
  value : digests/s, inputs resident in HBM, CUDA events on the launching stream, max over ranks
  e2e   : same metric through the C-ABI with HOST (page-locked) buffers, H2D + hash + D2H inside the region
Objects in the same JSON line (each with its own `roofline`: HBM fraction from the algorithmic bytes of SURVEY.md §8d,
`alu_frac` against the measured ALU-pipe ceiling, `traffic` from the committed ncu sums in profiles/roofline_traffic.json):
  state_root    C3 (configs[2]): StateRoot over 1M accounts x 16 slots per GPU, leaves/s; at N>1 the accounts are sharded by
                top key nibble and the 16-entry frontier is all-gathered inside b200_state_root_sharded_dev (NCCL behind the
                C ABI) — the only collective of the path; e2e through b200_state_root_full with host buffers
  mainnet_shape C4 (configs[3]; on by default at N>1): 31.25M-leaf mainnet-shaped shard per GPU = 250M leaves on 8 GPUs
  hash_partition (N>1): AccountHashing at N>1 — keccak + all-to-all of (digest, row) by owner rank + sort
  incremental   C5 (configs[4]): 10k dirty accounts against a resident 100M-leaf trie, latency; the incremental root is
                checked against a from-scratch device build of the updated state inside the run
  dynamic       the in-place block-update path (b200_dtrie_apply at 100M leaves, mixed blocks; b200_dstate_apply on the C3
                state) and the f2/f3/f4 legs (hash+sort, ordered roots, table rows), each in its own process and each
                checking itself (per-block roots against the static path / a twin, and an undo block back to the seed root)
  cpu_baseline  the oracle's keccak on the host cores, bounded sample; clocks; gpu_launches; parity_spot_check.

--impl reference times the CPU restatement of reth's algorithm (oracle/, all host threads) on the SAME 10M keys and config:
reth itself cannot be built in this image (no Rust toolchain; its keccak/HashBuilder live in external crates), see DESIGN.md.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2_KEYS = 10_000_000
C3_ACCOUNTS = 1_000_000
C3_SLOTS = 16
METRIC = "keccak256_digests_per_sec"
UNIT = "digests/s"
DUMP_SEED = 20240917
DUMP_ROWS = 131_072        # sampled digest rows: 131072 x 32 float32 = 16 MB
DUMP_MAX_BYTES = 64 << 20


def effective_cpus() -> int:
    """Host threads this process can really run: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


OUT_FD = [None]  # the real stdout when fd 1 is parked on stderr (multi-rank runs)


def emit(line: dict) -> None:
    """The one JSON line of the run, on the real stdout."""
    txt = json.dumps(line) + "\n"
    if OUT_FD[0] is None:
        sys.stdout.write(txt)
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(OUT_FD[0], txt.encode())


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def c2_config(n_keys: int, world: int) -> dict:
    """`config` of the headline line: the same dict on both arms (the driver compares them)."""
    return {"workload": "C2: batch keccak256 of 10M 32-byte keys per GPU (AccountHashing/StorageHashing inner loop)",
            "keys_per_gpu": n_keys, "msg_len": 32, "parallelism": f"keys sharded over {world} GPU(s), no collective",
            "l2": "input 320 MB + output 320 MB per step exceed the 126 MB L2; no flush needed"}


# ------------------------------------------------------------------------------------------------ --dump-outputs
def dump_rows(n: int) -> np.ndarray:
    """Ascending digest rows --dump-outputs writes: all of them up to DUMP_ROWS, else a fixed sample seeded by DUMP_SEED,
    so that two builds run with the same arguments write the same rows."""
    if n <= DUMP_ROWS:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))


def keccak_dump(digests: np.ndarray, rows: np.ndarray) -> dict:
    """digests: uint8 [len(rows), 32], the digests of `rows` of the batch."""
    return {"keccak_digests": digests.astype(np.float32), "keccak_digest_rows": rows.astype(np.float64)}


def root_dump(root_hex: str) -> np.ndarray:
    return np.frombuffer(bytes.fromhex(root_hex), np.uint8).astype(np.float32)


def write_dumps(out_dir: str, arrays: dict) -> None:
    """Writes every array as out_dir/<name>.npy: bytes as float32, row indices as float64 (exact below 2^53)."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ synthetic data
def splitmix64_torch(seed: int, n: int, device):
    """n 64-bit words of the splitmix64 stream (SURVEY.md §8d: C2 = seed 2, C3 = seed 3) as int64."""
    import torch
    M = (1 << 64) - 1

    def s64(x):  # python int -> wrapped signed 64
        x &= M
        return x - (1 << 64) if x >= (1 << 63) else x

    idx = torch.arange(1, n + 1, dtype=torch.int64, device=device)
    z = idx * s64(0x9E3779B97F4A7C15) + s64(seed)

    def lsr(v, k):
        return (v >> k) & ((1 << (64 - k)) - 1)

    z = (z ^ lsr(z, 30)) * s64(0xBF58476D1CE4E5B9)
    z = (z ^ lsr(z, 27)) * s64(0x94D049BB133111EB)
    return z ^ lsr(z, 31)


def random_keys_torch(seed: int, n: int, device):
    return splitmix64_torch(seed, 4 * n, device).view(n, 4)


def be_sort_key(words):
    """int64 [n] whose signed order equals the bytewise order of the first 8 bytes of each 32-byte row."""
    import torch
    b = words[:, 0].contiguous().view(torch.uint8).view(-1, 8).to(torch.int64)
    k = torch.zeros(b.shape[0], dtype=torch.int64, device=words.device)
    for i in range(8):
        k = (k << 8) | b[:, i]
    return k ^ (-(1 << 63))


def make_c3_shard(seed: int, n_accounts: int, slots: int, nibble_lo: int, nibble_hi: int, device):
    """C3-shaped shard resident on `device`: uniform random account keys inside top nibbles
    [nibble_lo, nibble_hi), `slots` random slots each, everything sorted as the C ABI requires."""
    import torch
    akeys = random_keys_torch(seed, n_accounts, device)
    ab = akeys.view(torch.uint8).view(n_accounts, 32)
    span = nibble_hi - nibble_lo
    top = (ab[:, 0] >> 4).to(torch.int64) % span + nibble_lo
    ab[:, 0] = (top.to(torch.uint8) << 4) | (ab[:, 0] & 0x0F)
    order = torch.sort(be_sort_key(akeys), stable=True).indices
    akeys = akeys[order].contiguous()
    w = splitmix64_torch(seed ^ 0xACC0, 8 * n_accounts, device).view(n_accounts, 8)
    accts = torch.zeros((n_accounts, 72), dtype=torch.uint8, device=device)
    accts[:, 0:2] = (w[:, 0] & 0xFFFF).contiguous().view(torch.uint8).view(n_accounts, 8)[:, 0:2]  # nonce < 2^16
    accts[:, 8 + 22:8 + 32] = w[:, 1:3].contiguous().view(torch.uint8).view(n_accounts, 16)[:, :10]  # balance < 2^80
    accts[:, 40:72] = w[:, 4:8].contiguous().view(torch.uint8).view(n_accounts, 32)  # code hash (contracts)
    m = n_accounts * slots
    skeys = random_keys_torch(seed ^ 0x5107, m, device)
    seg = torch.arange(m, dtype=torch.int64, device=device) // slots
    o1 = torch.sort(be_sort_key(skeys), stable=True).indices
    o2 = torch.sort(seg[o1], stable=True).indices
    skeys = skeys[o1[o2]].contiguous()
    vals = torch.zeros((m, 32), dtype=torch.uint8, device=device)
    v = splitmix64_torch(seed ^ 0x7A1, m, device) | 1  # uniform in [1, 2^64): RLP 1..9 bytes
    vals[:, 24:32] = v.view(torch.uint8).view(m, 8).flip(1)  # big-endian
    offs = torch.arange(0, n_accounts + 1, dtype=torch.int64, device=device) * slots
    return dict(akeys=akeys.view(torch.uint8).view(-1), accts=accts.view(-1), skeys=skeys.view(torch.uint8).view(-1),
                svals=vals.view(-1), offs=offs, n_accounts=n_accounts, n_slots=m)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU during the timed region (pynvml)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------ roofline
ALU_INSTR_PER_KECCAK_F = 4220.0  # ALU-pipe instructions per digest of keccak256_fixed32_kernel counted from its SASS
                                 # (tools/sass_count.py -> profiles/r02_keccak_sass_count.txt: 132 + 22 x 183 + 62; ncu
                                 # counts 4286 instructions of all kinds per digest, profiles/r02_keccak32.md)
ALU_LANES_PER_CLK_PER_SM = 64.0  # measured: profiles/r01_pipe_microbench.txt


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return json.load(open(peaks_path))["hbm_gbs"], "of measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "of fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_of(key):
    prof = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(prof):
        return json.load(open(prof)).get(key)
    return None


def make_roofline(algo_bytes: float, seconds: float, keccak_f: float, sm_mhz, traffic_key: str, kernel: str, n_sms: int = 148):
    """roofline object of one leg: `achieved` = algorithmic bytes (SURVEY.md §8d) / device time against the HBM peak (the
    contract figure), `alu_frac` = Keccak-f executed / device time against the measured ALU-pipe ceiling (the binding one)."""
    peak, src = hbm_peak()
    achieved = algo_bytes / seconds / 1e9
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
         "traffic": traffic_of(traffic_key), "kernel": kernel, "peak_source": src,
         "algorithmic_bytes_per_launch": algo_bytes, "keccak_f_per_launch": keccak_f, "alu_frac": None,
         "note": "Keccak-f is ALU-bound (~4220 ALU-pipe instructions per permutation on the 64-lane/clk/SM ALU pipe): alu_frac is the binding roofline"}
    if sm_mhz:
        alu_peak = n_sms * ALU_LANES_PER_CLK_PER_SM * sm_mhz * 1e6 / ALU_INSTR_PER_KECCAK_F
        r["alu_peak_keccak_f_per_s"] = alu_peak
        r["alu_frac"] = (keccak_f / seconds) / alu_peak
    return r


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_keccak_baseline(target_seconds: float = 12.0):
    """oracle keccak over 32-byte keys on all host cores; bounded sample of the C2 workload."""
    import oracle
    cores = effective_cpus()
    n = 2_000_000
    from tests.util import random_keys
    keys = random_keys(2, n)
    oracle.keccak256_fixed(keys[:100_000], threads=cores)  # warm
    t0 = time.perf_counter()
    reps = 0
    while True:
        oracle.keccak256_fixed(keys, threads=cores)
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= target_seconds or reps >= 64:
            break
    res = {"value": n * reps / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"{reps} x {n} of the 10M 32-byte keys (splitmix64 seed 2), scalar C keccak, {cores} threads, chunks of 100"}
    # best-effort SIMD figure (BASELINE.md §2): 8 sponges per AVX-512 register.  reth hashes one key at a time with
    # scalar assembly, so `value` stays the scalar port; this is reported beside it.
    if oracle.keccak256_fixed_simd(keys[:1024], threads=1) is not None:
        t0 = time.perf_counter()
        r2 = 0
        while r2 < 4 or time.perf_counter() - t0 < 3.0:
            oracle.keccak256_fixed_simd(keys, threads=cores)
            r2 += 1
        res["simd_value"] = n * r2 / (time.perf_counter() - t0)
        res["simd_note"] = "8-way AVX-512 multi-buffer Keccak (oracle/keccak_avx512.c), same threads; not what reth executes"
    return res


def cpu_state_root_baseline(n_accounts: int = 40_000, slots: int = 16):
    """oracle ParallelStateRoot-shaped build on all host cores over a C3-shaped sample."""
    import oracle
    from tests.util import synth_accounts, synth_storage
    cores = effective_cpus()
    akeys, accs = synth_accounts(3, n_accounts)
    skeys, svals, offs = synth_storage(3, np.full(n_accounts, slots))
    leaves = n_accounts * (slots + 1)
    t0 = time.perf_counter()
    oracle.state_root_full(akeys, accs, skeys, svals, offs, threads=cores)
    dt = time.perf_counter() - t0
    t1 = time.perf_counter()
    oracle.state_root_full(akeys, accs, skeys, svals, offs, threads=1)
    dt1 = time.perf_counter() - t1
    return {"value": leaves / dt, "unit": "leaves/s", "cores": cores, "kind": "port",
            "single_thread_value": leaves / dt1,
            "sample": f"{n_accounts} accounts x {slots} slots ({leaves} leaves): storage tries on {cores} threads, "
                      "account trie serial (ParallelStateRoot shape); single_thread_value = StateRoot shape"}


def run_reference(args, rank, world):
    """--impl reference: the CPU restatement timed on the host cores, same metric/config, bounded sample."""
    if rank != 0:
        return
    import oracle
    from tests.util import random_keys
    cores = effective_cpus()
    n = args.keys  # the same batch as the GPU arm: one step = one pass over all 10M keys
    keys = random_keys(2, n)
    for _ in range(args.warmup):
        oracle.keccak256_fixed(keys, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = oracle.keccak256_fixed(keys, threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        rows = dump_rows(n)
        write_dumps(args.dump_outputs, keccak_dump(out[rows], rows))
    val = n * args.steps / dt
    sample = f"each step hashes all {n} 32-byte keys on {cores} host threads (scalar C keccak, chunks of 100)"
    simd_val = None
    if oracle.keccak256_fixed_simd(keys[:1024], threads=1) is not None:
        t1 = time.perf_counter()
        reps = max(1, min(args.steps, 5))
        for _ in range(reps):
            oracle.keccak256_fixed_simd(keys, threads=cores)
        simd_val = n * reps / (time.perf_counter() - t1)
    sr = cpu_state_root_baseline()
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": c2_config(n, args.gpus),
        "reference": "CPU restatement of reth's algorithm (oracle/); reth cannot be built here (no Rust toolchain)",
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "simd_value": simd_val,
                         "simd_note": "8-way AVX-512 multi-buffer Keccak, best-effort figure; reth hashes one key at a time "
                                      "with scalar assembly, which is what `value` restates"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "state_root": {"value": sr["value"], "unit": "leaves/s", "cores": cores, "sample": sr["sample"],
                       "single_thread_value": sr["single_thread_value"]},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ main arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--keys", type=int, default=C2_KEYS, help="keys per GPU for the keccak workload")
    ap.add_argument("--accounts", type=int, default=C3_ACCOUNTS, help="accounts per GPU for the state-root workload")
    ap.add_argument("--skip-state-root", action="store_true")
    ap.add_argument("--base-accounts", type=int, default=100_000_000, help="resident base trie of the incremental (C5) leg")
    ap.add_argument("--dirty", type=int, default=10_000, help="dirty accounts per incremental update")
    ap.add_argument("--skip-incremental", action="store_true")
    ap.add_argument("--c4", action="store_true", help="also run the mainnet-shape leg (BASELINE config 4): per GPU "
                    "--c4-leaves leaves, 80%% EOAs, Zipf(1.2) storage sizes (on by default at N>1: 250M leaves over 8 GPUs)")
    ap.add_argument("--skip-c4", action="store_true")
    ap.add_argument("--c4-leaves", type=int, default=31_250_000, help="leaves per GPU (250M over 8 GPUs)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-dynamic", action="store_true", help="skip the in-place block-update legs (dynamic resident trie / "
                    "state: tools/dtrie_bench.py, tools/dstate_bench.py, each in its own process) and the f2/f3/f4 throughput legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed as "
                    "DIR/<name>.npy (float32/float64, rank 0): a seeded sample of the keccak digests with its row indices, "
                    "and the roots of the state-root legs that ran")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from reth_b200 import Engine

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # one process per GPU: this rank's CPUs and its page-locked staging buffers on the GPU's own socket (SCALE_r01: GPUs 0-3
    # hang off NUMA node 0, 4-7 off node 1; the e2e leg moves 640 MB per step and GPU through host memory)
    from reth_b200 import numa_bind_thread
    numa_node = numa_bind_thread(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the caller set it (the driver reads the communicator's rank count from that log).
        # stdout carries exactly one JSON line, and NCCL logs to fd 1 directly (at init, at the first use of a
        # collective, at destroy): fd 1 stays parked on stderr for the whole run, the line goes to the saved fd.
        sys.stdout.flush()
        OUT_FD[0] = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
        warm = torch.zeros(1, device=dev)
        dist.all_reduce(warm)
        torch.cuda.synchronize()
    eng = Engine(local_rank)
    comm = None
    if world > 1:
        # the library's own communicator (b200_comm_*): the frontier all-gather runs inside b200_state_root_sharded_dev on the
        # engine's stream; torch.distributed only carries the 128-byte NCCL id and the max-over-ranks of the timings
        from reth_b200 import Comm
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(Comm.unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        comm = Comm(eng, bytes(uid.cpu().numpy()), world, rank)
    # a dedicated (non-default) stream: torch events, NCCL and the engine's kernels are all ordered on it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng.use_torch_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------------------------------------------------------- C2: keccak, inputs resident in HBM
    n = args.keys
    d_keys = random_keys_torch(2 + 1000 * rank, n, dev).view(torch.uint8).view(-1)
    d_out = torch.empty(n * 32, dtype=torch.uint8, device=dev)
    for _ in range(args.warmup):
        eng.keccak256_fixed_dev(d_keys, 32, 32, n, d_out)
    barrier()
    launches0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        e0.record()
        for _ in range(args.steps):
            eng.keccak256_fixed_dev(d_keys, 32, 32, n, d_out)
        e1.record()
        barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    gpu_launches = eng.launch_count() - launches0
    ms_per_step = ms_total / args.steps
    value = world * n * args.steps / (ms_total * 1e-3)

    # spot-check the timed output against the oracle (checker only)
    import oracle
    idx = torch.randint(0, n, (64,), device=dev)
    got = d_out.view(n, 32)[idx].cpu().numpy()
    exp = oracle.keccak256_fixed(d_keys.view(n, 32)[idx].cpu().numpy())
    parity_ok = bool((got == exp).all())
    dumps = {}
    if args.dump_outputs and rank == 0:
        rows = dump_rows(n)
        dumps.update(keccak_dump(d_out.view(n, 32)[torch.from_numpy(rows).to(dev)].cpu().numpy(), rows))

    # ---------------------------------------------------------------- C2 e2e: host buffers through the C ABI
    h_in = eng.pinned_empty((n, 32))
    h_out = eng.pinned_empty((n, 32))
    h_in[:] = d_keys.view(n, 32).cpu().numpy()
    eng.set_stream(None)
    for _ in range(2):
        eng.keccak256_fixed(h_in, 32, out=h_out)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.keccak256_fixed(h_in, 32, out=h_out)
    dt = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e = {"value": world * n * e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": n * 32,
           "d2h_bytes_per_step": n * 32, "steps": e2e_steps, "numa_node_bound": numa_node,
           "api": "b200_keccak256_fixed (host pointers, page-locked, chunked double-buffered H2D/kernel/D2H)"}
    eng.use_torch_stream()

    # ---------------------------------------------------------------- roofline of the dominant kernel
    # 32 B key read + 32 B digest written per digest (SURVEY.md §8d); one Keccak-f per digest
    roofline = make_roofline(64.0 * n, ms_per_step * 1e-3, float(n), clk.summary()["sm_mhz"],
                             "keccak256_fixed32_kernel_dram_bytes_per_launch", "keccak256_fixed32_kernel")
    sm_mhz = clk.summary()["sm_mhz"]

    # ---------------------------------------------------------------- C3: state root
    state_root = None
    if not args.skip_state_root:
        state_root = bench_state_root(args, eng, dev, rank, world, barrier, max_over_ranks, sm_mhz, comm)

    c4 = None
    if (args.c4 or world > 1) and not args.skip_c4:
        c4 = bench_c4(args, eng, dev, rank, world, barrier, max_over_ranks, comm)

    hash_part = None
    if comm is not None and not args.skip_state_root:
        hash_part = bench_hash_partition(args, eng, comm, dev, rank, world, barrier, max_over_ranks)

    incremental = None
    if not args.skip_incremental and world == 1:
        incremental = bench_incremental(args, eng, dev, sm_mhz, skip_cpu=args.skip_cpu)

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        cpu = cpu_keccak_baseline()
        if state_root is not None:
            state_root["cpu_baseline"] = cpu_state_root_baseline()

    dynamic = None
    if not args.skip_dynamic and rank == 0 and world == 1:
        dynamic = bench_dynamic(args)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": c2_config(n, world),
            "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(gpu_launches), "roofline": roofline,
            "cpu_baseline": cpu, "state_root": state_root, "mainnet_shape": c4, "hash_partition": hash_part,
            "incremental": incremental,
            "parity_spot_check": parity_ok,
        }
        if dynamic is not None:
            line["dynamic"] = dynamic
        if args.dump_outputs:
            for name, leg, key in (("state_root", state_root, "root"), ("mainnet_shape_root", c4, "root"),
                                   ("incremental_root", incremental, "root_after")):
                if leg and leg.get(key):
                    dumps[name] = root_dump(leg[key])
            write_dumps(args.dump_outputs, dumps)
        emit(line)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def bench_state_root(args, eng, dev, rank, world, barrier, max_over_ranks, sm_mhz=None, comm=None):
    import torch
    import torch.distributed as dist
    n_acc = args.accounts
    lo, hi = rank * 16 // world, (rank + 1) * 16 // world
    if world > 16:
        raise SystemExit("top-nibble sharding supports at most 16 ranks")
    sh = make_c3_shard(3 + 1000 * rank, n_acc, C3_SLOTS, lo, hi, dev)
    leaves = n_acc * (C3_SLOTS + 1)
    d_root = torch.zeros(32, dtype=torch.uint8, device=dev)
    d_front = torch.zeros(16 * 68, dtype=torch.uint8, device=dev)
    gathered = [torch.zeros(16 * 68, dtype=torch.uint8, device=dev) for _ in range(world)] if world > 1 else None

    def step():
        if world == 1:
            eng.state_root_full_dev(sh["akeys"], sh["accts"], n_acc, sh["skeys"], sh["svals"], sh["offs"],
                                    sh["n_slots"], d_root)
        else:
            # frontier -> ncclAllGather (16 x 68 B per rank: the one collective of the path) -> root, one C call
            comm.state_root_sharded_dev(sh["akeys"], sh["accts"], n_acc, sh["skeys"], sh["svals"], sh["offs"], sh["n_slots"], d_root)

    for _ in range(max(2, args.warmup - 1)):
        step()
    barrier()
    eng.dev_status()
    steps = max(3, min(args.steps, 10))
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    eng.dev_status()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    stats = eng.last_stats()
    res = {"metric": "state_root_leaves_per_sec", "value": world * leaves / (ms * 1e-3), "unit": "leaves/s",
           "ms_per_step": ms, "steps": steps, "gpu_launches": int(eng.launch_count() - l0),
           "config": {"workload": f"C3: StateRoot over {n_acc} accounts x {C3_SLOTS} storage slots per GPU, "
                                  "level-by-level node-hash frontier", "leaves_per_gpu": leaves,
                      "parallelism": "single GPU" if world == 1 else
                      f"accounts sharded by top key nibble over {world} GPUs, one ncclAllGather of 16 frontier entries inside "
                      "b200_state_root_sharded_dev"},
           "root": bytes(d_root.cpu().numpy()).hex(),
           "node_digests_per_sec": world * stats["hashed_nodes"] / (ms * 1e-3) if world == 1 else None,
           "stats": stats,
           "algorithmic_gb_per_s": world * (n_acc * C3_SLOTS * 64 + n_acc * 104) / (ms * 1e-3) / 1e9}
    # per GPU: 64 B per storage leaf + 104 B per account leaf (SURVEY.md §8d); Keccak-f = rate blocks absorbed, counted on
    # the device (stats.keccak_f)
    kf = float(stats.get("keccak_f") or 0) or 1.494 * leaves
    res["roofline"] = make_roofline(float(n_acc * C3_SLOTS * 64 + n_acc * 104), ms * 1e-3, kf, sm_mhz,
                                    "state_root_c3_dram_bytes_per_step", "state_root_full (leaf + branch kernels of one build)")
    if world == 1:
        # e2e: host (page-locked) buffers through b200_state_root_full
        h = {k: eng.pinned_empty(tuple(v.shape), np.uint8 if v.dtype == torch.uint8 else np.int64)
             for k, v in sh.items() if hasattr(v, "shape")}
        for k in h:
            h[k][...] = sh[k].cpu().numpy()
        eng.set_stream(None)
        accts = h["accts"].view(eng_account_dtype())
        for _ in range(2):
            root = eng.state_root_full(h["akeys"], accts, h["skeys"], h["svals"], h["offs"].view(np.uint64))
        t0 = time.perf_counter()
        e2e_steps = 3
        for _ in range(e2e_steps):
            root = eng.state_root_full(h["akeys"], accts, h["skeys"], h["svals"], h["offs"].view(np.uint64))
        dt = time.perf_counter() - t0
        eng.use_torch_stream()
        res["e2e"] = {"value": leaves * e2e_steps / dt, "unit": "leaves/s",
                      "h2d_bytes_per_step": int(sum(v.nbytes for v in h.values())), "d2h_bytes_per_step": 32,
                      "root_matches_device_run": root.hex() == res["root"],
                      "api": "b200_state_root_full (host pointers, page-locked)"}
    return res


def bench_hash_partition(args, eng, comm, dev, rank, world, barrier, max_over_ranks):
    """AccountHashing at N > 1 (SURVEY.md §8e): every rank holds an arbitrary slice of the plain table (20-byte addresses with a
    72-byte account row each); b200_hash_partition_dev hashes, all-to-alls (digest, row) by owner rank over NVLink and sorts."""
    import torch
    n = args.keys // 2
    t_in = random_keys_torch(11 + 1000 * rank, n, dev).view(torch.uint8).view(n, 32)[:, :20].contiguous().view(-1)
    t_val = splitmix64_torch(13 + 1000 * rank, 9 * n, dev).view(torch.uint8).view(-1)
    cap = n + n // 2 + 1024
    t_k = torch.empty(cap * 32, dtype=torch.uint8, device=dev)
    t_v = torch.empty(cap * 72, dtype=torch.uint8, device=dev)
    got = 0
    for _ in range(2):
        got = comm.hash_partition_dev(t_in, 20, 20, n, t_val, 72, cap, t_k, t_v)
    barrier()
    steps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        got = comm.hash_partition_dev(t_in, 20, 20, n, t_val, 72, cap, t_k, t_v)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    k = t_k.view(cap, 32)[:got]
    pre = be_sort_key(k.contiguous().view(torch.int64).view(got, 4))
    ok = bool((pre[1:] >= pre[:-1]).all().item()) and bool(((k[:, 0] >> 4).to(torch.int64) * world // 16 == rank).all().item())
    return {"metric": "hash_partition_keys_per_sec", "value": world * n / (ms * 1e-3), "unit": "keys/s", "ms_per_step": ms,
            "keys_per_gpu": n, "row_bytes": 72, "rows_received_rank0": got, "sorted_and_owned_rank0": ok,
            "exchange_bytes_per_gpu": int(n * (world - 1) / world * (32 + 72)),
            "config": {"workload": f"{n} addresses + 72-byte rows per GPU: keccak, all-to-all by top nibble over {world} GPUs, sort"}}


def make_c4_shard(seed: int, leaves: int, nibble_lo: int, nibble_hi: int, device):
    """Mainnet-shaped shard (SURVEY.md §8d C4): 20% of the leaves are accounts, 80% of the accounts are EOAs without
    storage, the contracts' slot counts follow Zipf(s=1.2) (a few huge tries, a long tail of tiny ones)."""
    import torch
    n_acc = leaves // 5
    n_slots = leaves - n_acc
    n_contracts = n_acc // 5
    ranks = np.arange(1, n_contracts + 1, dtype=np.float64) ** -1.2
    lo, hi = 1.0, float(n_slots)
    for _ in range(60):  # scale so that the sizes sum to n_slots
        c = 0.5 * (lo + hi)
        tot = np.maximum(1, np.floor(c * ranks)).sum()
        lo, hi = (c, hi) if tot < n_slots else (lo, c)
    sizes = np.maximum(1, np.floor(lo * ranks)).astype(np.int64)
    sizes[0] += n_slots - int(sizes.sum())
    rng = np.random.default_rng(seed)
    counts = np.zeros(n_acc, np.int64)
    counts[rng.choice(n_acc, n_contracts, replace=False)] = sizes  # contracts scattered over the key space
    akeys = random_keys_torch(seed, n_acc, device)
    ab = akeys.view(torch.uint8).view(n_acc, 32)
    span = nibble_hi - nibble_lo
    top = (ab[:, 0] >> 4).to(torch.int64) % span + nibble_lo
    ab[:, 0] = (top.to(torch.uint8) << 4) | (ab[:, 0] & 0x0F)
    akeys = akeys[torch.sort(be_sort_key(akeys), stable=True).indices].contiguous()
    w = splitmix64_torch(seed ^ 0xACC0, 8 * n_acc, device).view(n_acc, 8)
    accts = torch.zeros((n_acc, 72), dtype=torch.uint8, device=device)
    accts[:, 0:2] = (w[:, 0] & 0xFFFF).contiguous().view(torch.uint8).view(n_acc, 8)[:, 0:2]
    accts[:, 8 + 22:8 + 32] = w[:, 1:3].contiguous().view(torch.uint8).view(n_acc, 16)[:, :10]
    accts[:, 40:72] = w[:, 4:8].contiguous().view(torch.uint8).view(n_acc, 32)
    t_counts = torch.from_numpy(counts).to(device)
    offs = torch.zeros(n_acc + 1, dtype=torch.int64, device=device)
    offs[1:] = torch.cumsum(t_counts, 0)
    m = int(offs[-1].item())
    seg = torch.repeat_interleave(torch.arange(n_acc, dtype=torch.int64, device=device), t_counts)
    skeys = random_keys_torch(seed ^ 0x5107, m, device)
    o1 = torch.sort(be_sort_key(skeys), stable=True).indices
    o2 = torch.sort(seg[o1], stable=True).indices
    skeys = skeys[o1[o2]].contiguous()
    del o1, o2, seg
    vals = torch.zeros((m, 32), dtype=torch.uint8, device=device)
    v = splitmix64_torch(seed ^ 0x7A1, m, device) | 1
    vals[:, 24:32] = v.view(torch.uint8).view(m, 8).flip(1)
    return dict(akeys=akeys.view(torch.uint8).view(-1), accts=accts.view(-1), skeys=skeys.view(torch.uint8).view(-1),
                svals=vals.view(-1), offs=offs, n_accounts=n_acc, n_slots=m, max_trie=int(sizes[0]),
                contracts=n_contracts)


def bench_c4(args, eng, dev, rank, world, barrier, max_over_ranks, comm=None):
    """BASELINE config 4: MerkleExecute-style full build of a mainnet-shaped state, subtries sharded over the GPUs."""
    import torch
    import torch.distributed as dist
    lo, hi = rank * 16 // world, (rank + 1) * 16 // world
    sh = make_c4_shard(4 + 1000 * rank, args.c4_leaves, lo, hi, dev)
    n_acc, leaves = sh["n_accounts"], sh["n_accounts"] + sh["n_slots"]
    d_root = torch.zeros(32, dtype=torch.uint8, device=dev)
    d_front = torch.zeros(16 * 68, dtype=torch.uint8, device=dev)
    gathered = [torch.zeros(16 * 68, dtype=torch.uint8, device=dev) for _ in range(world)] if world > 1 else None

    def step():
        if world == 1:
            eng.state_root_full_dev(sh["akeys"], sh["accts"], n_acc, sh["skeys"], sh["svals"], sh["offs"], sh["n_slots"], d_root)
        else:
            comm.state_root_sharded_dev(sh["akeys"], sh["accts"], n_acc, sh["skeys"], sh["svals"], sh["offs"], sh["n_slots"], d_root)

    for _ in range(2):
        step()
    barrier()
    eng.dev_status()
    steps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    eng.dev_status()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    stats = eng.last_stats()
    res = {"metric": "state_root_leaves_per_sec", "value": world * leaves / (ms * 1e-3), "unit": "leaves/s", "ms_per_step": ms,
           "steps": steps, "root": bytes(d_root.cpu().numpy()).hex(),
           "config": {"workload": f"C4: mainnet-shape full build, {leaves} leaves per GPU ({world * leaves} total): "
                                  f"{n_acc} accounts (80% EOAs), {sh['contracts']} contracts with Zipf(1.2) storage sizes, "
                                  f"largest trie {sh['max_trie']} slots",
                      "parallelism": "single GPU" if world == 1 else
                      f"accounts sharded by top key nibble over {world} GPUs, one NCCL all-gather of 16 frontier entries"},
           "stats_rank0": stats}
    del sh
    torch.cuda.empty_cache()
    return res


def bench_incremental(args, eng, dev, sm_mhz=None, skip_cpu=False):
    """BASELINE config 5: a resident base trie of --base-accounts accounts (no storage), then updates of --dirty random
    existing accounts (new balance + nonce).  Reports the root latency of one update (device-resident dirty set) and
    the same through the host-pointer C ABI."""
    import torch
    from reth_b200 import ResidentTrie
    n, m = args.base_accounts, args.dirty
    try:
        keys = random_keys_torch(5, n, dev)
        order = torch.sort(be_sort_key(keys), stable=True).indices
        keys = keys[order].contiguous()
        del order
        accts = torch.zeros((n, 72), dtype=torch.uint8, device=dev)
        w = splitmix64_torch(5 ^ 0xACC0, n, dev)
        accts[:, 8 + 24:8 + 32] = w.view(torch.uint8).view(n, 8)  # balance < 2^64
        accts[:, 40:72] = torch.frombuffer(bytearray(bytes.fromhex(
            "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470")), dtype=torch.uint8).to(dev)
        del w
        d_root = torch.zeros(32, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        trie = ResidentTrie.create_dev(eng, keys.view(torch.uint8).view(-1), accts.view(-1), None, n, d_root)
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
    except (RuntimeError, Exception) as e:  # noqa: BLE001 - out of memory on a smaller part: report, do not die
        return {"error": f"{type(e).__name__}: {e}"[:300], "base_leaves": n}
    base_root = bytes(d_root.cpu().numpy()).hex()
    g = torch.Generator(device=dev)
    g.manual_seed(55)
    lat = []
    d_new_root = torch.zeros(32, dtype=torch.uint8, device=dev)
    accts_now = accts  # updated in place as the updates are committed (the base tensor is not needed afterwards)
    reps = 12
    for it in range(reps):
        idx = torch.randperm(n, generator=g, device=dev)[:m] if n < 50_000_000 else \
            torch.unique(torch.randint(0, n, (m + m // 8,), generator=g, device=dev))[:m]
        mm = int(idx.numel())
        dk = keys[idx].contiguous().view(torch.uint8).view(-1)
        da = accts[idx].clone()
        da[:, 0] = it + 1                       # nonce
        da[:, 8 + 24:8 + 32] = torch.randint(0, 255, (mm, 8), generator=g, device=dev, dtype=torch.uint8)
        da = da.view(-1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        trie.update_dev(dk, da, None, mm, d_new_root)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        accts_now[idx] = da.view(mm, 72)
        if it >= 2:
            lat.append((e0.elapsed_time(e1) * 1e3, wall * 1e6))
    stats = eng.last_stats()
    dev_us = float(np.median([a for a, _ in lat]))
    wall_us = float(np.median([b for _, b in lat]))
    # host-pointer path (H2D of the dirty set + D2H of the root inside the call)
    hk = dk.view(mm, 32).cpu().numpy()
    ha = da.view(mm, 72).cpu().numpy().view(eng_account_dtype()).reshape(-1)
    eng.set_stream(None)
    trie.update(hk, ha)
    t0 = time.perf_counter()
    for _ in range(5):
        root = trie.update(hk, ha)
    e2e_us = (time.perf_counter() - t0) / 5 * 1e6
    eng.use_torch_stream()
    # in-bench parity: the incremental root must equal a from-scratch device build of the updated state (the from-scratch
    # path is the one the tests pin against the oracle and reth's golden roots); `accts_now` tracks what was committed
    root_inc = bytes(trie.root())
    d_chk = torch.zeros(32, dtype=torch.uint8, device=dev)
    eng.state_root_dev(keys.view(torch.uint8).view(-1), accts_now.view(-1), None, n, d_chk)
    torch.cuda.synchronize()
    eng.dev_status()
    root_scratch = bytes(d_chk.cpu().numpy())
    if root_inc != root_scratch or root_inc != root:
        raise SystemExit(f"C5 parity: incremental root {root_inc.hex()} / {root.hex()} != from-scratch root {root_scratch.hex()}")
    # Keccak-f of one update: dirty leaves (account leaf RLP 104..148 B -> 1 or 2 rate blocks; these are ~112 B = 1) +
    # re-hashed branch nodes (1..4 blocks by child count); counted on the device when the library reports it
    kf = float(stats.get("keccak_f") or 0) or float(mm + 2.6 * stats["branches_added"])
    # algorithmic bytes: the dirty set in (32 B key + 72 B account) + per re-hashed node its <=16 child refs read and its ref written
    algo = mm * 104.0 + stats["branches_added"] * (16 * 33 + 33)
    res = {"metric": "incremental_root_latency_us", "value": wall_us, "unit": "us", "device_us": dev_us,
           "e2e_us": e2e_us, "base_leaves": n, "dirty_accounts": mm, "dirty_leaves_per_sec": mm / (wall_us * 1e-6),
           "base_build_ms": build_s * 1e3, "base_root": base_root, "root_after": root.hex(),
           "root_check": "incremental root == from-scratch device build of the updated 100M-leaf state: ok",
           "rehashed_branch_nodes": stats["branches_added"], "levels": stats["levels"],
           "resident_bytes": trie.device_bytes(),
           "roofline": make_roofline(algo, dev_us * 1e-6, kf, sm_mhz, "incremental_c5_dram_bytes_per_step",
                                     "b200_trie_update (locate + mark + wavefront)"),
           "config": {"workload": f"C5: {mm}-account dirty set against a resident {n}-leaf base trie, "
                                  "value changes of existing accounts, root path re-hash only"}}
    res["roofline"]["note"] = ("latency-bound: the critical path is ~27 dependent Keccak-f (7 levels x <=4 blocks); "
                               "frac / alu_frac are reported for completeness")
    if not skip_cpu:
        # the CPU restatement has no incremental walk (reth's needs its database); its figure is the from-scratch
        # account-trie fold (StateRoot shape, serial like reth's) on a bounded sample, scaled to the base size
        import oracle
        from tests.util import synth_accounts
        ns = 1_000_000
        ak, ac = synth_accounts(5, ns)
        t0 = time.perf_counter()
        oracle.state_root(ak, ac)
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": ns / dt, "unit": "leaves/s", "cores": 1, "kind": "port",
                               "sample": f"from-scratch account-trie fold over {ns} accounts, single thread (the fold is serial in reth); "
                                         "no incremental CPU path exists outside reth's database walker",
                               "equivalent_full_rebuild_s": n / (ns / dt),
                               "note": "an incremental update on the CPU would touch the same ~46k nodes: at the oracle's "
                                       "~0.55 us per Keccak-f that is ~60 ms single-threaded"}
    trie.close()
    del keys, accts
    torch.cuda.empty_cache()
    return res


def bench_dynamic(args):
    """The in-place block-update path (SURVEY.md §8 f1 / a10: the role reth's sparse trie plays on the live path) and the
    f2/f3/f4 throughput legs, each in its own process (its own CUDA context and a timeout) so that whatever happens there
    cannot touch the numbers above.  Every leg checks itself: the dynamic legs compare every block's root with the static
    merge + from-scratch rebuild path (dtrie) / a device-resident twin (dstate) and finally undo all blocks in one block,
    which must restore the root of the from-scratch build the state was created from."""
    import subprocess
    root = os.path.dirname(os.path.abspath(__file__))
    out = {}
    runs = {
        "dtrie_apply_mixed_block": ["tools/dtrie_bench.py", "--base", str(args.base_accounts), "--dirty", str(args.dirty),
                                    "--mix", "80,10,10", "--compare", "--cpu-sample", "1000000"],
        "dstate_apply_c3_shape": ["tools/dstate_bench.py", "--accounts", "1000000", "--slots", "16", "--touch", "2000",
                                  "--slot-writes", "10", "--device-resident", "--cpu-sample", "40000"],
        "hash_sort_keys": ["tools/hash_sort_bench.py", "--keys", "10000000"],
        "hash_sort_storage": ["tools/hash_sort_storage_bench.py", "--slots", "10000000", "--accounts", "200000"],
        "ordered_roots_receipts": ["tools/ordered_bench.py", "--blocks", "2000", "--items", "200", "--shape", "receipts"],
        "table_rows_c3_shape": ["tools/rows_bench.py", "--accounts", "1000000", "--slots", "16"],
    }
    for name, cmd in runs.items():
        if not os.path.exists(os.path.join(root, cmd[0])):
            continue
        try:
            r = subprocess.run([sys.executable] + cmd, cwd=root, capture_output=True, text=True, timeout=600)
            last = [l for l in r.stdout.splitlines() if l.startswith("{")]
            out[name] = json.loads(last[-1]) if r.returncode == 0 and last else {"error": (r.stderr or r.stdout)[-300:]}
        except Exception as e:  # noqa: BLE001
            out[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
    d = out.get("dtrie_apply_mixed_block", {})
    if d.get("merge_rebuild_wall_us_median") and d.get("apply_wall_us_median"):
        d["speedup_over_merge_rebuild"] = d["merge_rebuild_wall_us_median"] / d["apply_wall_us_median"]
    return out


def eng_account_dtype():
    from reth_b200 import ACCOUNT_DTYPE
    return ACCOUNT_DTYPE


if __name__ == "__main__":
    main()
