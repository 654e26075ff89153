#!/usr/bin/env python3
"""bench.py -- EdDSA-Poseidon verify_batch (and B8 fixed-base / variable-base / compressed-pipeline
secondaries) on N B200s of one node.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # CPU arm: C++ restatement of the reference algorithm
    python bench.py ... --dump-outputs DIR    # also save what the last timed step returned, to compare two builds

The inputs are made from fixed seeds, so two runs with the same arguments time the same signatures.

One "step" = one verify_batch pass over this rank's shard (2^21 signatures per GPU, i.e. BASELINE
config 4's 2^24 signatures over 8 GPUs; 10 % corrupted).  The batch shards with no exchange between
lanes, so there is no data-path collective: torch.distributed is used for the barrier and the
max-over-ranks time only ("scaling": "weak").

Besides the headline line the same JSON object carries (BASELINE.json names two metrics and five configs):
  second_metric   B8 scalar-mults/s: public_batch over 2^20 keys PER GPU on every rank (device-resident and end to
                  end), next to the CPU port of PrivateKey::public
  configs         config 3 (2^22 variable-base pairs) and config 5 (2^24 compressed signatures) at their stated
                  TOTAL size, sharded over the ranks (strong scaling), device-resident, max over ranks
  single_caller   config 4 as written: ONE host batch of 2^24 signatures verified across all N devices by the
                  library's multi-device layer (bjj_multi_*: one context + one host thread per device, no NCCL),
                  from pinned, pageable and page-locked-per-call host memory; run by rank 0 while the other ranks idle
  secondary       the remaining rows of the hot-path table on one GPU, each against its own roofline

Prints ONE JSON line (rank 0).  Keys follow the driver contract; `roofline` is quoted against the
integer-multiply (IMAD) issue rate, the pipe this path is bound by (SURVEY.md section 8d), with HBM as
a secondary counter.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

Q = 21888242871839275222246405745257275088548364400416034343698204186575808495617
SUBORDER = 21888242871839275222246405745257275088614511777268538073601725287587578984328 >> 3
METRIC = "eddsa_poseidon_verifies_per_sec"
UNIT = "verifies/s"

# Algorithmic work per unit, in limb-MACs (one 32x32->64 multiply-accumulate = one IMAD.WIDE.U32 on sm_100a).
# fmul = 128 (8x8 products + 8x8 Montgomery reduction), fsqr = 100 (36 products of the squaring triangle + the same
# reduction), a Montgomery dot product of N terms = 64 N + 64.  Counts are for the algorithms actually built, as
# (multiplications, squarings); derivations in DESIGN.md section 6.
FMUL = 128
FSQR = 100


def mac(mul, sqr=0):
    return mul * FMUL + sqr * FSQR


FERMAT = (56, 253)                                     # fr_inv: a^(Q-2), sliding window of 4 bits (fr_pow_sched): 56 M + 253 S
SQRT_POW = (49, 224)                                   # a^((T-1)/2) of the square root, same method: 49 M + 224 S
ALGO_OPS = {
    # k_verify_hash besides Poseidon: two on-curve gates (2 squarings + 3 multiplications each) + 6 Montgomery conversions
    "verify_hash_extra": (6 + 6, 4),
    # k_verify_ec_vm (half-size scalars, 33 radix-16 windows over the tables of 8A and R8): conversions 4 + map 4
    # + 8A = 3 doublings (4S + 3M, 4S + 4M for the last) + two 9-entry tables 2 x 64 + 32 x 4 doublings
    # + 33 x (8 + 7) table additions + 1 + 17 B8 additions (16 x 7 + 6)
    "verify_ec": (4 + 4 + 10 + 128 + 32 * 13 + 33 * 15 + 1 + 16 * 7 + 6, 12 + 32 * 16),
    # 16-bit comb (17 mixed additions) + map + batched inversion: 5 per lane + one Fermat inversion per 32 lanes
    "fixed_base": (17 * 7 + 1 + 5 + 2 + FERMAT[0] / 32, FERMAT[1] / 32),
    # gate (2S + 3M), conversions, 9-entry table, 64 windows x (4 doublings + 1 addition), batched inversion share
    "mul_scalar": (3 + 4 + 2 + 64 + 7 + 64 * (13 + 7) + 5 + FERMAT[0] / 32, 2 + 64 * 16 + FERMAT[1] / 32),
    # decompress_point: y^2, d y^2; batched inversion (3 + Fermat / 32); x^2 = u / v; a^((T-1)/2) over a 225-bit
    # exponent; x0, b; Pohlig-Hellman 21 + 14 + 7 squarings and 8 multiplications; x0^2; 3 conversions
    "decompress": (1 + 3 + FERMAT[0] / 32 + 1 + SQRT_POW[0] + 2 + 8 + 3, 1 + FERMAT[1] / 32 + SQRT_POW[1] + 42 + 1),
    # PointProjective::add, literal add-2008-bbjlp as src/lib.rs:88-131 sequences it (12 multiplications + 1 squaring) + 9 conversions
    "proj_add": (12 + 9, 1),
}


def poseidon_mac(t, rounds_p, n_inputs):
    """the schedule of csrc/poseidon.cuh: 7 full rounds x (t S-boxes x^5 = 2S + 1M, t dot products of t terms) + the
    last full round (t S-boxes, ONE dot product); partial rounds: t <= 4 one S-box, one dot product, t - 1
    multiplications per round; t >= 5 in groups of three rounds (dot products of t, t + 1, t + 2 terms, then t - 1 dot
    products of 3 terms); + the Montgomery conversions of the inputs and the output"""
    sbox = mac(1, 2)

    def dot(n):
        return n * 64 + 64
    full = 7 * (t * sbox + t * dot(t)) + t * sbox + dot(t)
    if t >= 5:
        groups, rem = divmod(rounds_p, 3)
        partial = groups * (3 * sbox + dot(t) + dot(t + 1) + dot(t + 2) + (t - 1) * dot(3))
        if rem == 2:
            partial += 2 * sbox + dot(t) + dot(t + 1) + (t - 1) * dot(2)
        elif rem == 1:
            partial += sbox + dot(t) + mac(t - 1)
    else:
        partial = rounds_p * (sbox + dot(t) + mac(t - 1))
    return full + partial + mac(n_inputs + 1)


POSEIDON6_MAC = poseidon_mac(6, 60, 0)
# k_verify_split: ~75 Euclid steps x (8 + 8) wide multiplies + two Montgomery products mod l
SPLIT_MAC = 75 * 16 + 2 * FMUL
ALGO_MAC = {k: mac(*v) for k, v in ALGO_OPS.items()}
ALGO_MAC["verify"] = ALGO_MAC["verify_hash_extra"] + ALGO_MAC["verify_ec"] + POSEIDON6_MAC + SPLIT_MAC
# the same counts per KERNEL launch and lane (tools/ncu_summarize.py divides the executed IMAD.WIDE of a capture by these)
KERNEL_MAC = {
    "k_verify_ec_vm": ALGO_MAC["verify_ec"],
    "k_verify_hash": ALGO_MAC["verify_hash_extra"] + POSEIDON6_MAC,
    "k_poseidon<6>": poseidon_mac(6, 60, 5),
    "k_fixed_base": mac(17 * 7 + 3),
    "k_public": mac(17 * 7 + 3),
    "k_mul_scalar(": mac(3 + 4 + 2 + 64 + 7 + 64 * 20 + 2, 2 + 64 * 16),
    "k_decompress_finish": mac(1 + 1 + SQRT_POW[0] + 2 + 8 + 2, SQRT_POW[1] + 42 + 1),
}
# Measured on B200 (profiles/r1_pipe_probe.jsonl): IMAD.WIDE.U32 issues at 32 lanes/clk/SM -- half the 32-bit IMAD
# rate that SURVEY.md section 8d's model (64 lanes/clk/SM) assumes.
WIDE_MAC_LANES_PER_CLK_SM = 32
MODEL_LANES_PER_CLK_SM = 64


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler(threading.Thread):
    """samples SM clocks / throttle reasons of one GPU while the timed region runs: NVML in-process (a sample
    every 20 ms, cheap enough for 8 ranks at once), `nvidia-smi -lms` as the fallback when pynvml is missing"""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device = device
        self.rows = []          # (sm_mhz, sm_max_mhz, [reason names])
        self.stop_flag = threading.Event()
        self.proc = None
        self.source = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.device < len(ids) and ids[self.device].isdigit():
                return int(ids[self.device])
        return self.device

    def _run_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
        smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        self.source = "nvml"
        while not self.stop_flag.is_set():
            sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
            mask = int(get_reasons(h))
            self.rows.append((sm, smax, [nm for nm, bit in self.NVML_REASONS if mask & bit]))
            time.sleep(0.02)

    def _run_smi(self):
        self.source = "nvidia-smi"
        self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + self.FIELDS,
                                      "--format=csv,noheader,nounits", "-lms", "100"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                self.rows.append((float(r[1]), float(r[2]), [nm for nm, v in zip(names, r[5:9]) if v.lower().startswith("active")]))
            except Exception:
                pass
            if self.stop_flag.is_set():
                break

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            try:
                self._run_smi()
            except Exception:
                pass

    def finish(self):
        self.stop_flag.set()
        if self.proc:
            try:
                self.proc.terminate()        # exact PID we started
            except Exception:
                pass
        self.join(timeout=2)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [r[0] for r in self.rows]
        reasons = sorted({nm for r in self.rows for nm in r[2]})
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(r[1] for r in self.rows), "reasons": reasons,
                "samples": len(sm), "source": self.source}


# ---------------------------------------------------------------------------------------------------
# synthetic signatures (SURVEY.md section 8d, config 4): valid signatures made ON THE DEVICE by the
# library's own sign kernel from random keys / messages, then 10 % corrupted on the host by class.
# ---------------------------------------------------------------------------------------------------
CORRUPTIONS = ["flip_S", "flip_msg", "swap_R8", "swap_A", "S_plus_SUBORDER", "msg_gt_Q", "off_curve", "special_point"]


def _to_int(row):
    return int.from_bytes(row.tobytes(), "little")


def _from_int(v):
    return np.frombuffer(int(v).to_bytes(32, "little"), dtype=np.uint8)


def corrupt(cols, seed, denom=10):
    """cols = [r8x, r8y, s, ax, ay, msg] numpy (n,32) arrays, modified in place.  Returns (expected_ok, class_id)
    where class_id = -1 for untouched lanes."""
    n = len(cols[0])
    rng = np.random.default_rng(seed)
    h = rng.integers(0, max(denom, 1), size=n)
    cls = np.where((h == 0) & (denom > 0), rng.integers(0, len(CORRUPTIONS), size=n), -1)
    expected = np.ones(n, dtype=np.uint8)
    r8x, r8y, s, ax, ay, msg = cols
    orig = [c.copy() for c in (r8x, r8y, ax, ay)]
    idx = np.nonzero(cls == 0)[0]
    s[idx, rng.integers(0, 31, size=len(idx))] ^= (1 << rng.integers(0, 8, size=len(idx))).astype(np.uint8)
    expected[idx] = 0
    idx = np.nonzero(cls == 1)[0]
    msg[idx, rng.integers(0, 31, size=len(idx))] ^= (1 << rng.integers(0, 8, size=len(idx))).astype(np.uint8)
    expected[idx] = 0
    idx = np.nonzero(cls == 2)[0]
    r8x[idx], r8y[idx] = orig[0][(idx + 1) % n], orig[1][(idx + 1) % n]
    expected[idx] = 0
    idx = np.nonzero(cls == 3)[0]
    ax[idx], ay[idx] = orig[2][(idx + 1) % n], orig[3][(idx + 1) % n]
    expected[idx] = 0
    for i in np.nonzero(cls == 4)[0]:                      # stays VALID: verify never range-checks S
        s[i] = _from_int(_to_int(s[i]) + SUBORDER)
    idx = np.nonzero(cls == 5)[0]
    msg[idx] = 0xFF
    expected[idx] = 0
    for i in np.nonzero(cls == 6)[0]:                      # x + 1: off the curve -> exact lane
        tgt = r8x if (i & 1) else ax
        tgt[i] = _from_int((_to_int(tgt[i]) + 1) % Q)
    expected[cls == 6] = 0
    specials = [(0, 0), (0, 1), (0, Q - 1)]
    for i in np.nonzero(cls == 7)[0]:
        x, y = specials[int(i) % 3]
        if i & 4:
            r8x[i], r8y[i] = _from_int(x), _from_int(y)
        else:
            ax[i], ay[i] = _from_int(x), _from_int(y)
    expected[cls == 7] = 0
    return expected, cls


DUMP_BUDGET = 64 << 20                                     # bytes over all ranks' --dump-outputs files


def dump_outputs(out_dir, name, arr, rank, world):
    """writes arr as float32 to out_dir/<name>[_rank<r>].npy; when the ranks' files together would exceed DUMP_BUDGET, a
    sample of lanes drawn with a fixed seed (sorted, the same for every run with the same lane count) stands in for all"""
    cap = (DUMP_BUDGET // world - 4096) // 4
    if len(arr) > cap:
        arr = arr[np.sort(np.random.default_rng(0).choice(len(arr), size=cap, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    fname = "%s_rank%d.npy" % (name, rank) if world > 1 else name + ".npy"
    np.save(os.path.join(out_dir, fname), np.asarray(arr, dtype=np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-lanes", type=int, default=21, help="signatures per GPU (2^21 x 8 GPUs = config 4's 2^24)")
    ap.add_argument("--no-secondary", action="store_true", help="headline line only (profiling runs)")
    ap.add_argument("--corrupt-denominator", type=int, default=10,
                    help="1 lane in this many is corrupted (default 10 = the 10 %% of config 4; 0 = none, for diagnosis)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget for the cpu_baseline leg")
    ap.add_argument("--log2-total", type=int, default=24, help="config 4 / 5 total batch of the single-caller and config legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the accept bits of the last timed verify_batch step to DIR/verify_ok[_rank<r>].npy (float32; a fixed "
                         "sample of the lanes when all ranks together would exceed %d MiB)" % (DUMP_BUDGET >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU arm computed; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return
    run_ours(args, rank, local_rank, world)


# ---------------------------------------------------------------------------------------------------
# CPU arm: the C++ restatement of the reference algorithm (oracle/bjj_ref.cpp), one std::thread per core
# ---------------------------------------------------------------------------------------------------
def _cpu_fixture(ora, n_sample, seed=1):
    rng = np.random.default_rng(seed)
    keys = rng.integers(0, 256, size=(n_sample, 32), dtype=np.uint8)
    msgs = rng.integers(0, 256, size=(n_sample, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x1F
    rx, ry, s, _ = ora.sign(keys, msgs)
    ax, ay = ora.public(keys)
    return keys, msgs, [rx, ry, s, ax, ay, msgs]


def cpu_verify_rate(n_sample, steps, warmup, seed=1):
    """times the C++ restatement of the reference algorithm (oracle port) over n_sample signatures"""
    import common
    ora = common.OracleC(threads=os.cpu_count() or 1)
    _, _, cols = _cpu_fixture(ora, n_sample, seed)
    expected, _ = corrupt(cols, seed)
    for _ in range(warmup):
        ora.verify(*cols)
    t0 = time.perf_counter()
    for _ in range(steps):
        ok = ora.verify(*cols)
    dt = time.perf_counter() - t0
    assert np.array_equal(ok, expected), "oracle disagrees with the constructed expectations"
    return n_sample * steps / dt, dt / steps, ora.threads


def cpu_public_rate(n_sample):
    """PrivateKey::public (src/lib.rs:304-306) through the CPU port: B8 * scalar_key(key) by double-and-add"""
    import common
    ora = common.OracleC(threads=os.cpu_count() or 1)
    keys = np.random.default_rng(3).integers(0, 256, size=(n_sample, 32), dtype=np.uint8)
    t0 = time.perf_counter()
    ora.public(keys)
    return n_sample / (time.perf_counter() - t0), ora.threads


def cpu_config1(n=1024):
    """BASELINE config 1 = the reference's criterion workloads (benches/bench_babyjubjub.rs:30-53: add, mul_scalar,
    compress, decompress, sign, verify) on a 1,024-element batch, through the CPU port: all host threads (the rayon
    par_iter stand-in) and one thread (what criterion's per-call times correspond to)."""
    import common
    out = {}
    for label, threads in (("all_threads", os.cpu_count() or 1), ("one_thread", 1)):
        ora = common.OracleC(threads=threads)
        keys, msgs, cols = _cpu_fixture(ora, n, 11)
        rx, ry, s, ax, ay, _ = cols
        one = np.zeros((n, 32), dtype=np.uint8)
        one[:, 0] = 1
        comp = ora.compress(ax, ay)
        ops = {
            "add": lambda: ora.add(ax, ay, one, rx, ry, one),
            "mul_scalar": lambda: ora.mul_scalar(ax, ay, s),
            "compress": lambda: ora.compress(ax, ay),
            "decompress": lambda: ora.decompress(comp),
            "sign": lambda: ora.sign(keys, msgs),
            "verify": lambda: ora.verify(*cols),
            "public": lambda: ora.public(keys),
        }
        res = {}
        for name, fn in ops.items():
            fn()
            reps, t0 = 0, time.perf_counter()
            while True:
                fn()
                reps += 1
                dt = time.perf_counter() - t0
                if dt > 0.25 or reps >= 50:
                    break
            res[name] = {"ops_per_s": n * reps / dt, "us_per_op": dt / (n * reps) * 1e6 * (threads if label == "all_threads" else 1)}
        out[label] = {"threads": threads, "ops": res}
    return out


def run_reference(args):
    """reference arm: the reference's own CPU algorithm (C++ restatement; the Rust crate cannot be built
    in this image) on all host threads, on a bounded sample of the same workload"""
    cores = os.cpu_count() or 1
    n_sample = 512 * cores
    rate, sec_per_step, threads = cpu_verify_rate(n_sample, args.steps, args.warmup)
    pub_rate, _ = cpu_public_rate(256 * cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 (4x64-bit Montgomery)", "data": "synthetic",
        "config": {"workload": "verify (EdDSA-Poseidon), 10% corrupted; bounded sample of config 4", "sample_signatures": n_sample},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d signatures per step, std::thread per core" % n_sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "second_metric": {"metric": "b8_scalar_mults_per_sec", "value": pub_rate, "unit": "mults/s", "cores": threads,
                          "sample": "%d keys, PrivateKey::public through the CPU port" % (256 * cores)},
        "config1_cpu": cpu_config1(1024),
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
def kernel_metrics():
    """per-kernel counters extracted from the committed ncu captures (tools/ncu_summarize.py -> profiles/)"""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_kernel_metrics.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def run_ours(args, rank, local_rank, world):
    import torch
    import babyjubjub_rs_b200 as bjj
    import common
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    cpu_group = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # CPU-side group: ranks that wait for rank 0's single-caller legs must not spin a kernel on their GPU
        cpu_group = dist.new_group(backend="gloo")
    dev = torch.device("cuda", local_rank)
    eng = bjj.Engine(local_rank)
    lib, ctx = eng.lib, eng.ctx
    # a dedicated non-default stream: the kernels are launched on it (passed to the _dev entry points) and the
    # CUDA events that time them are recorded on the same stream
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    assert stream.cuda_stream != 0
    n = 1 << args.log2_lanes

    def dptr(t):
        return ctypes.c_void_p(t.data_ptr())

    def hptr(t):
        return ctypes.c_void_p(t.data_ptr())

    def check(rc, what):
        if rc not in (0,):
            raise RuntimeError("%s failed: %d (%s)" % (what, rc, lib.bjj_error_string(rc).decode()))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return bjj.max_over_ranks(x, dist, dev)

    def timed_dev(fn, steps, warmup=3):
        """K back-to-back calls on `stream`, CUDA events on the same stream, barrier + synchronize on both sides,
        max over ranks -> ms per step"""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    def timed_host(fn, steps, warmup=2):
        for _ in range(warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        barrier()
        return max_over_ranks(time.perf_counter() - t0) / steps * 1e3

    # ---- data: keys / msgs random on the device; signatures by the library's sign kernel -------------
    def make_signatures(count, seed):
        g = torch.Generator(device=dev)
        g.manual_seed(seed)
        keys = torch.randint(0, 256, (count, 32), dtype=torch.uint8, device=dev, generator=g)
        msgs = torch.randint(0, 256, (count, 32), dtype=torch.uint8, device=dev, generator=g)
        msgs[:, 31] &= 0x1F                                   # < 2^253 < Q
        r8x, r8y, s, ax, ay = (torch.empty((count, 32), dtype=torch.uint8, device=dev) for _ in range(5))
        st = torch.empty(count, dtype=torch.uint8, device=dev)
        for off in range(0, count, 1 << 21):
            m = min(1 << 21, count - off)
            sl = slice(off, off + m)
            check(lib.bjj_sign_batch_dev(ctx, m, dptr(keys[sl]), dptr(msgs[sl]), dptr(r8x[sl]), dptr(r8y[sl]), dptr(s[sl]),
                                         dptr(st[sl]), sp), "sign")
            check(lib.bjj_public_batch_dev(ctx, m, dptr(keys[sl]), dptr(ax[sl]), dptr(ay[sl]), sp), "public")
        torch.cuda.synchronize()
        assert int(st.max().item()) == 0
        return keys, msgs, r8x, r8y, s, ax, ay

    keys, msgs, r8x, r8y, s, ax, ay = make_signatures(n, 0xB200 + rank)
    cols_h = [t.cpu().numpy() for t in (r8x, r8y, s, ax, ay, msgs)]
    expected, cls = corrupt(cols_h, 0xC0DE + rank, args.corrupt_denominator)
    pinned = [torch.from_numpy(c).pin_memory() for c in cols_h]
    cols_d = [p.to(dev, non_blocking=True) for p in pinned]
    ok_d = torch.zeros(n, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def step_dev():
        check(lib.bjj_verify_batch_dev(ctx, n, *[dptr(c) for c in cols_d], dptr(ok_d), sp), "verify_batch_dev")

    # ---- headline: device-resident timing --------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step_dev()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_dev()
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = eng.kernel_launches - launches0
    clocks = sampler.finish()
    check(lib.bjj_sync(ctx), "sync")
    ok_h = ok_d.cpu().numpy()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "verify_ok", ok_h, rank, world)
    mism = int((ok_h != expected).sum())
    dev_ms = max_over_ranks(dev_ms)
    value = world * n * args.steps / (dev_ms * 1e-3)

    # ---- end to end: host (pinned) buffers through the C ABI, H2D + D2H inside the timed region -------------
    ok_pin = torch.zeros(n, dtype=torch.uint8).pin_memory()

    def step_e2e():
        check(lib.bjj_verify_batch(ctx, n, *[hptr(p) for p in pinned], hptr(ok_pin)), "verify_batch")

    e2e_ms = timed_host(step_e2e, args.steps)
    e2e_value = world * n / (e2e_ms * 1e-3)
    mism += int((ok_pin.numpy() != expected).sum())

    # ---- oracle spot check (outside every timed region): random lanes + every corruption class ---------------
    checked = 0
    if rank == 0:
        ora = common.OracleC(threads=os.cpu_count() or 1)
        rng = np.random.default_rng(5)
        pick = [rng.choice(n, size=2048, replace=False)]
        for c in range(len(CORRUPTIONS)):
            idx = np.nonzero(cls == c)[0]
            pick.append(idx[:256])
        pick = np.unique(np.concatenate(pick))
        ok_ref = ora.verify(*[c[pick] for c in cols_h])
        mism += int((ok_ref != ok_h[pick]).sum())
        checked = len(pick)
    if mism:
        raise SystemExit("PARITY FAILURE: %d lanes differ from the oracle / constructed expectations" % mism)

    peaks, peak_kind = measured_peaks()
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    props = torch.cuda.get_device_properties(local_rank)
    sms = props.multi_processor_count
    mac_peak = sms * WIDE_MAC_LANES_PER_CLK_SM * sm_max * 1e6 / 1e12      # T limb-MAC/s, measured IMAD.WIDE rate
    imad_peak = mac_peak * 1e12

    second = None
    configs = []
    if not args.no_secondary:
        # ---- second headline metric: B8 scalar-mults/s = PrivateKey::public over 2^20 keys PER GPU (config 2) -----
        nk = 1 << 20
        gk = torch.Generator(device=dev)
        gk.manual_seed(77 + rank)
        pkeys = torch.randint(0, 256, (nk, 32), dtype=torch.uint8, device=dev, generator=gk)
        prx, pry = (torch.empty((nk, 32), dtype=torch.uint8, device=dev) for _ in range(2))
        ms = timed_dev(lambda: check(lib.bjj_public_batch_dev(ctx, nk, dptr(pkeys), dptr(prx), dptr(pry), sp), "public_dev"), args.steps)
        pk_pin = pkeys.cpu().pin_memory()
        ox_pin, oy_pin = (torch.empty((nk, 32), dtype=torch.uint8).pin_memory() for _ in range(2))
        ms_e2e = timed_host(lambda: check(lib.bjj_public_batch(ctx, nk, hptr(pk_pin), hptr(ox_pin), hptr(oy_pin)), "public"), args.steps)
        assert np.array_equal(ox_pin.numpy(), prx.cpu().numpy()) and np.array_equal(oy_pin.numpy(), pry.cpu().numpy())
        if rank == 0:
            idx = torch.randperm(nk, device=dev)[:1024]
            ex, ey = common.OracleC(threads=os.cpu_count() or 1).public(pkeys[idx].cpu().numpy())
            assert np.array_equal(prx[idx].cpu().numpy(), ex) and np.array_equal(pry[idx].cpu().numpy(), ey), "public_batch parity"
        rate = world * nk / (ms * 1e-3)
        second = {"metric": "b8_scalar_mults_per_sec", "workload": "public_batch: 2^20 random keys per GPU (config 2), weak scaling",
                  "value": rate, "unit": "mults/s", "n_gpus": world, "ms_per_step": ms,
                  "roofline_frac_imad": rate / world * ALGO_MAC["fixed_base"] / imad_peak,
                  "e2e": {"value": world * nk / (ms_e2e * 1e-3), "unit": "mults/s", "h2d_bytes_per_step": nk * 32, "d2h_bytes_per_step": nk * 64,
                          "path": "bjj_public_batch (C ABI, pinned host buffers); 96 B per key cross PCIe"},
                  "oracle_checked_lanes": 1024}
        del pkeys, prx, pry

        # ---- configs 3 and 5 at their stated TOTAL size, sharded over the ranks (strong scaling) ----------------------
        n3 = (1 << 22) // world
        g3 = torch.Generator(device=dev)
        g3.manual_seed(303 + rank)
        k3 = torch.randint(0, 256, (n3, 32), dtype=torch.uint8, device=dev, generator=g3)
        k3[:, 31] &= 0x3F
        reps = (n3 + n - 1) // n
        px3 = ax.repeat(reps, 1)[:n3].contiguous()
        py3 = ay.repeat(reps, 1)[:n3].contiguous()
        ox3, oy3 = (torch.empty((n3, 32), dtype=torch.uint8, device=dev) for _ in range(2))
        ms = timed_dev(lambda: check(lib.bjj_mul_scalar_batch_dev(ctx, n3, dptr(px3), dptr(py3), dptr(k3), dptr(ox3), dptr(oy3), sp), "mul_scalar"),
                       max(2, args.steps // 2), warmup=1)
        if rank == 0:
            idx = torch.randperm(n3, device=dev)[:512]
            ex, ey = common.OracleC(threads=os.cpu_count() or 1).mul_scalar(px3[idx].cpu().numpy(), py3[idx].cpu().numpy(), k3[idx].cpu().numpy())
            assert np.array_equal(ox3[idx].cpu().numpy(), ex) and np.array_equal(oy3[idx].cpu().numpy(), ey), "mul_scalar_batch parity"
        rate = world * n3 / (ms * 1e-3)
        configs.append({"config": 3, "metric": "variable_base_scalar_mults_per_sec",
                        "workload": "mul_scalar_batch: 2^22 (point, 254-bit scalar) pairs in all, 2^22/%d per GPU" % world,
                        "value": rate, "unit": "mults/s", "n_gpus": world, "scaling": "strong", "ms_per_step": ms,
                        "roofline_frac_imad": rate / world * ALGO_MAC["mul_scalar"] / imad_peak, "oracle_checked_lanes": 512})
        del k3, px3, py3, ox3, oy3

        n5 = (1 << args.log2_total) // world
        k5, m5, r5x, r5y, s5, a5x, a5y = make_signatures(n5, 0x5005 + rank)
        comp_r, comp_a = (torch.empty((n5, 32), dtype=torch.uint8, device=dev) for _ in range(2))
        check(lib.bjj_compress_batch_dev(ctx, n5, dptr(r5x), dptr(r5y), dptr(comp_r), sp), "compress")
        check(lib.bjj_compress_batch_dev(ctx, n5, dptr(a5x), dptr(a5y), dptr(comp_a), sp), "compress")
        torch.cuda.synchronize()
        sig64 = torch.cat([comp_r, s5], dim=1).contiguous()
        del k5, r5x, r5y, s5, a5x, a5y, comp_r
        m5[::10, 0] ^= 1                                       # 10 % wrong message
        sig64[5::97, :32] = 0xFF                               # undecodable R8 (y >= Q)
        ok5, st5 = (torch.empty(n5, dtype=torch.uint8, device=dev) for _ in range(2))
        ms = timed_dev(lambda: check(lib.bjj_verify_compressed_batch_dev(ctx, n5, dptr(sig64), dptr(comp_a), dptr(m5), dptr(ok5), dptr(st5), sp),
                                     "verify_compressed"), 2, warmup=1)
        if rank == 0:
            eok, est = common.OracleC(threads=os.cpu_count() or 1).verify_compressed(sig64[:2048].cpu().numpy(), comp_a[:2048].cpu().numpy(),
                                                                                    m5[:2048].cpu().numpy())
            assert np.array_equal(ok5[:2048].cpu().numpy(), eok) and np.array_equal(st5[:2048].cpu().numpy(), est), "verify_compressed parity"
        frac_ok = float(ok5.float().mean().item())
        assert 0.85 < frac_ok < 0.92, frac_ok                   # 10 % wrong messages + 1 % undecodable R8
        rate = world * n5 / (ms * 1e-3)
        configs.append({"config": 5, "metric": "compressed_pipeline_verifies_per_sec",
                        "workload": "verify_compressed_batch: 2^%d x (64 B sig + 32 B pk + 32 B msg) in all, 2^%d/%d per GPU; decompress R8 and A -> "
                                    "Poseidon -> Straus" % (args.log2_total, args.log2_total, world),
                        "value": rate, "unit": "verifies/s", "n_gpus": world, "scaling": "strong", "ms_per_step": ms,
                        "roofline_frac_imad": rate / world * (ALGO_MAC["verify"] + 2 * ALGO_MAC["decompress"]) / imad_peak, "oracle_checked_lanes": 2048})
        del sig64, comp_a, m5, ok5, st5
        torch.cuda.empty_cache()

    if rank != 0:
        if dist is not None:
            # rank 0 now drives every device from ONE process (single_caller) and runs the one-GPU legs: wait on the CPU
            torch.cuda.synchronize()
            dist.barrier(group=cpu_group)
            dist.destroy_process_group()
        return

    model_peak = sms * MODEL_LANES_PER_CLK_SM * sm_max * 1e6 / 1e12        # SURVEY model (32-bit IMAD rate)
    per_gpu = value / world
    achieved = per_gpu * ALGO_MAC["verify"] / 1e12
    km = kernel_metrics()
    ec = km.get("k_verify_ec_vm", {})
    roofline = {
        "bound": "imad", "achieved": achieved, "peak": mac_peak, "unit": "T limb-MAC/s", "frac": achieved / mac_peak,
        "peak_kind": "measured: %d SMs x %d IMAD.WIDE lanes/clk x %.0f MHz (profiles/r1_pipe_probe.jsonl, profiles/r2_ncu_probe_summary.txt)"
                     % (sms, WIDE_MAC_LANES_PER_CLK_SM, sm_max),
        "frac_of_survey_model": achieved / model_peak,
        "survey_model_peak": model_peak,
        "algorithmic_mac_per_verify": ALGO_MAC["verify"],
        "frac_at_observed_clock": (achieved / (sms * WIDE_MAC_LANES_PER_CLK_SM * clocks["sm_mhz"] * 1e6 / 1e12)) if clocks.get("sm_mhz") else None,
        # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch, from the committed ncu --set full
        # capture (profiles/r2_kernel_metrics.json), scaled from the captured lane count to this launch
        "traffic": int(ec["dram_bytes_per_lane"] * n) if ec.get("dram_bytes_per_lane") else None,
        "traffic_note": "per-thread window tables (2 x 9 x 128 B written, 66 x 128 B read per lane) dominate; algorithmic 225 B per lane; "
                        "HBM is a secondary counter for this kernel",
        "dominant_kernel": "k_verify_ec_vm (Straus pass over half-size scalars on shared-memory slots)",
        "kernels": {k: {kk: v[kk] for kk in ("ms_per_2p20_lanes", "fmaheavy_pct", "issue_active_pct", "no_instruction_per_issue",
                                              "executed_wide_over_algorithmic", "fma_pipe_passenger_frac", "dram_bytes_per_lane") if kk in v}
                    for k, v in km.items()},
        "hbm": {"achieved_gbs": per_gpu * 193 / 1e9, "peak_gbs": peaks.get("hbm_gbs"), "peak_kind": peak_kind,
                "note": "193 B per verify (6 x 32 B in, 1 B out); secondary counter, this path is not HBM-bound"},
    }

    single = None
    secondary = []
    if not args.no_secondary:
        single = run_single_caller(args, bjj, torch, world, cols_h, expected, lib)
        secondary = run_secondaries(args, eng, torch, dev, stream, common, (keys, msgs, r8x, r8y, s, ax, ay))

    cores = os.cpu_count() or 1
    probe_rate, _, threads = cpu_verify_rate(64 * cores, 1, 0)
    n_sample = int(min(1 << 18, max(256 * cores, probe_rate * args.cpu_seconds)))
    rate, _, threads = cpu_verify_rate(n_sample, 1, 0)
    cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": "%d signatures (10%% corrupted), C++ restatement of the reference algorithm, one std::thread per core" % n_sample}
    if second is not None:
        pub_rate, pub_threads = cpu_public_rate(int(min(1 << 16, max(64 * cores, 0.15 * probe_rate * args.cpu_seconds))))
        second["cpu_baseline"] = {"value": pub_rate, "unit": "mults/s", "cores": pub_threads, "kind": "port",
                                  "sample": "PrivateKey::public through the CPU port (LSB-first double-and-add, src/lib.rs:149-164)"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": "verify_batch: 2^%d EdDSA-Poseidon signatures per GPU (config 4: 2^24 over 8 GPUs), 10%% corrupted in 8 classes"
                               % args.log2_lanes,
                   "signatures_per_gpu": n, "l2": "inputs larger than L2 (%.0f MB per step)" % (n * 192 / 1e6),
                   "sharding": "contiguous slices per rank, no collective"},
        "roofline": roofline,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 192, "d2h_bytes_per_step": n,
                "path": "bjj_verify_batch (C ABI, pinned host buffers, chunked double-buffered copies), one call per rank"},
        "gpu_launches": launches,
        "clocks": clocks,
        "gpu": {"name": props.name, "uuid": str(getattr(props, "uuid", "")), "sms": sms},
        "parity": {"lanes_checked_vs_oracle": checked, "lanes_checked_vs_construction": 2 * n, "mismatches": 0},
        "second_metric": second,
        "configs": configs,
        "single_caller": single,
        "secondary": secondary,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(group=cpu_group)
        dist.destroy_process_group()


def run_single_caller(args, bjj, torch, world, cols_h, expected, lib):
    """config 4 as written: ONE caller, ONE host batch of 2^24 signatures, all `world` devices, through bjj_multi_*
    (one context + one host thread per device inside the library, no NCCL).  Strong scaling: the total is fixed."""
    total = 1 << args.log2_total
    n = len(expected)
    reps = (total + n - 1) // n
    exp_all = np.tile(expected, reps)[:total]
    me = bjj.MultiEngine(devices=list(range(world)))
    out = {"workload": "verify_batch: ONE host batch of 2^%d signatures (10%% corrupted) over %d device(s), bjj_multi_verify_batch"
                       % (args.log2_total, world),
           "n_gpus": world, "scaling": "strong", "devices_used": me.devices, "unit": UNIT,
           "h2d_bytes_per_step": total * 192, "d2h_bytes_per_step": total}
    pageable = [np.ascontiguousarray(np.tile(c, (reps, 1))[:total]) for c in cols_h]
    ok = np.empty(total, dtype=np.uint8)
    launches0 = me.kernel_launches

    def run(cols, okbuf, register):
        me.set_host_register(register)
        me.verify_batch(*cols, out=okbuf)           # warm-up (arenas, tables)
        t0 = time.perf_counter()
        steps = 2
        for _ in range(steps):
            me.verify_batch(*cols, out=okbuf)
        dt = (time.perf_counter() - t0) / steps
        assert np.array_equal(np.asarray(okbuf), exp_all), "single-caller parity"
        return total / dt, dt * 1e3

    v, ms = run(pageable, ok, False)
    out["pageable"] = {"value": v, "ms_per_step": ms, "note": "plain malloc'd arrays, what the INTEGRATION.md binding passes"}
    v, ms = run(pageable, ok, True)
    out["pageable_registered_per_call"] = {"value": v, "ms_per_step": ms, "note": "cudaHostRegister + Unregister inside every call"}
    pinned = [torch.from_numpy(c).pin_memory() for c in pageable]
    del pageable
    ok_pin = torch.empty(total, dtype=torch.uint8).pin_memory()
    v, ms = run([p.numpy() for p in pinned], ok_pin.numpy(), False)
    out["pinned"] = {"value": v, "ms_per_step": ms, "note": "bjj_host_alloc / cudaHostAlloc'd arrays"}
    out["value"] = out["pinned"]["value"]
    out["gpu_launches"] = me.kernel_launches - launches0
    me.close()
    return out


def run_secondaries(args, eng, torch, dev, stream, common, sig):
    """the remaining rows of the hot-path table on one GPU (rank 0), each checked against the oracle on a sample"""
    lib, ctx = eng.lib, eng.ctx
    sp = ctypes.c_void_p(stream.cuda_stream)
    out = []
    ora = common.OracleC(threads=os.cpu_count() or 1)
    keys, msgs, r8x, r8y, s, ax, ay = sig
    g = torch.Generator(device=dev)
    g.manual_seed(79)

    def dptr(t):
        return ctypes.c_void_p(t.data_ptr())

    def timed(fn, steps, warmup=2):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    peaks, _ = measured_peaks()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    imad_peak = sms * WIDE_MAC_LANES_PER_CLK_SM * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    n = 1 << 20
    comp_a, comp_r = (torch.empty((n, 32), dtype=torch.uint8, device=dev) for _ in range(2))
    lib.bjj_compress_batch_dev(ctx, n, dptr(ax[:n]), dptr(ay[:n]), dptr(comp_a), sp)
    lib.bjj_compress_batch_dev(ctx, n, dptr(r8x[:n]), dptr(r8y[:n]), dptr(comp_r), sp)

    # decompress_point (row a7): 2^20 compressed points, ~125 multiplications + ~275 squarings each -> IMAD-bound
    st2 = torch.empty(n, dtype=torch.uint8, device=dev)
    dx, dy = (torch.empty((n, 32), dtype=torch.uint8, device=dev) for _ in range(2))
    ms = timed(lambda: lib.bjj_decompress_batch_dev(ctx, n, dptr(comp_r), dptr(dx), dptr(dy), dptr(st2), sp), args.steps)
    ex, ey, est = ora.decompress(comp_r[:1024].cpu().numpy())
    assert np.array_equal(dx[:1024].cpu().numpy(), ex) and np.array_equal(st2[:1024].cpu().numpy(), est), "decompress_batch parity"
    rate = n / (ms * 1e-3)
    out.append({"metric": "decompress_points_per_sec", "workload": "decompress_batch: 2^20 compressed points", "value": rate,
                "unit": "points/s", "ms_per_step": ms, "roofline_frac_imad": rate * ALGO_MAC["decompress"] / imad_peak, "oracle_checked_lanes": 1024})

    # POSEIDON.hash, every width poseidon-rs accepts (row a8 + next row f-2): t = n_inputs + 1
    rounds_p = [56, 57, 56, 60, 60, 63]                  # poseidon-rs / circomlib R_P for t = 2..7 (R_F = 8)
    ins_all = [ax[:n], ay[:n], r8x[:n], r8y[:n], msgs[:n], dx]
    ho = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    for nin in range(1, 7):
        ins = [t.contiguous() for t in ins_all[:nin]]
        arr = (ctypes.c_void_p * nin)(*[t.data_ptr() for t in ins])
        ms = timed(lambda: lib.bjj_poseidon_batch_dev(ctx, nin, n, arr, dptr(ho), sp), max(2, args.steps // 2), warmup=1)
        eh = ora.poseidon([t[:128].cpu().numpy() for t in ins])
        assert np.array_equal(ho[:128].cpu().numpy(), eh), "poseidon_batch parity (t = %d)" % (nin + 1)
        t = nin + 1
        rp = rounds_p[t - 2]
        pmac = poseidon_mac(t, rp, nin)
        rate = n / (ms * 1e-3)
        out.append({"metric": "poseidon%d_hashes_per_sec" % nin, "workload": "poseidon_batch: 2^20 x %d inputs (t = %d)" % (nin, t),
                    "value": rate, "unit": "hashes/s", "ms_per_step": ms,
                    "roofline_frac_imad": rate * pmac / imad_peak, "oracle_checked_lanes": 128})

    # PrivateKey::sign (next row f-3) as a pipeline of kernels: BLAKE-512 x2 -> two fixed-base multiplications with
    # batched inversions -> Poseidon t = 6 -> S
    ns = 1 << 19
    o = [torch.empty((ns, 32), dtype=torch.uint8, device=dev) for _ in range(3)]
    sst = torch.empty(ns, dtype=torch.uint8, device=dev)
    ms = timed(lambda: lib.bjj_sign_batch_dev(ctx, ns, dptr(keys[:ns]), dptr(msgs[:ns]), dptr(o[0]), dptr(o[1]), dptr(o[2]), dptr(sst), sp),
               max(2, args.steps // 2), warmup=1)
    er = ora.sign(keys[:256].cpu().numpy(), msgs[:256].cpu().numpy())
    assert all(np.array_equal(o[k][:256].cpu().numpy(), er[k]) for k in range(3)), "sign_batch parity"
    rate = ns / (ms * 1e-3)
    out.append({"metric": "signatures_per_sec", "workload": "sign_batch: 2^19 (key, msg) pairs", "value": rate, "unit": "signatures/s",
                "ms_per_step": ms, "roofline_frac_imad": rate * (2 * ALGO_MAC["fixed_base"] + poseidon_mac(6, 60, 5)) / imad_peak,
                "oracle_checked_lanes": 256})

    # verify_schnorr (next row f-4): the verify pipeline with full-width scalars (64-65 windows)
    # Schnorr fixture from the EdDSA one: any (pk, r, s, msg) works for timing; parity against the oracle on a sample
    okb, stb = (torch.empty(ns, dtype=torch.uint8, device=dev) for _ in range(2))
    ms = timed(lambda: lib.bjj_verify_schnorr_batch_dev(ctx, ns, dptr(ax[:ns]), dptr(ay[:ns]), dptr(msgs[:ns]), dptr(r8x[:ns]), dptr(r8y[:ns]),
                                                        dptr(s[:ns]), dptr(okb), dptr(stb), sp), max(2, args.steps // 2), warmup=1)
    eok, est = ora.verify_schnorr(*[t[:256].cpu().numpy() for t in (ax, ay, msgs, r8x, r8y, s)])
    assert np.array_equal(okb[:256].cpu().numpy(), eok) and np.array_equal(stb[:256].cpu().numpy(), est), "verify_schnorr parity"
    out.append({"metric": "schnorr_verifies_per_sec", "workload": "verify_schnorr_batch: 2^19 (pk, r, s, msg)", "value": ns / (ms * 1e-3),
                "unit": "verifies/s", "ms_per_step": ms, "oracle_checked_lanes": 256})

    # adversarial batch: every A off the curve -> every lane on the literal (exact) ladder
    na = 1 << 17
    bad_ax = ax[:na].clone()
    bad_ax[:, 0] ^= 1                                       # x xor 1: off the curve with overwhelming probability
    oka = torch.empty(na, dtype=torch.uint8, device=dev)
    ms = timed(lambda: lib.bjj_verify_batch_dev(ctx, na, dptr(r8x[:na]), dptr(r8y[:na]), dptr(s[:na]), dptr(bad_ax), dptr(ay[:na]), dptr(msgs[:na]),
                                                dptr(oka), sp), 2, warmup=1)
    eok = ora.verify(*[t[:256].cpu().numpy() for t in (r8x, r8y, s, bad_ax, ay, msgs)])
    assert np.array_equal(oka[:256].cpu().numpy(), eok), "adversarial verify parity"
    out.append({"metric": "adversarial_verifies_per_sec", "workload": "verify_batch: 2^17 signatures, 100% off-curve A (every lane replays "
                "the reference's LSB-first double-and-add literally)", "value": na / (ms * 1e-3), "unit": "verifies/s", "ms_per_step": ms,
                "roofline_frac_imad": na / (ms * 1e-3) * (mac(257 * 24 + 17 * 7 + 20 + FERMAT[0], 257 * 2 + FERMAT[1]) + POSEIDON6_MAC) / imad_peak, "oracle_checked_lanes": 256})

    # Point::compress (row a6): pure data movement, 64 B in + 32 B out per point -> HBM-bound
    n = 1 << 22
    bx = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=g)
    by = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=g)
    bx[:, 31] &= 0x0F
    by[:, 31] &= 0x0F
    bo = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    ms = timed(lambda: lib.bjj_compress_batch_dev(ctx, n, dptr(bx), dptr(by), dptr(bo), sp), args.steps * 4)
    assert np.array_equal(bo[:4096].cpu().numpy(), ora.compress(bx[:4096].cpu().numpy(), by[:4096].cpu().numpy())), "compress parity"
    gbs = n * 96 / (ms * 1e-3) / 1e9
    out.append({"metric": "compress_points_per_sec", "workload": "compress_batch: 2^22 points (403 MB per step, larger than L2)",
                "value": n / (ms * 1e-3), "unit": "points/s", "ms_per_step": ms,
                "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak},
                "oracle_checked_lanes": 4096})
    # PointProjective::add (row a2): 6 x 32 B in, 3 x 32 B out, 13 fmul (+9 Montgomery conversions)
    n = 1 << 21
    one = torch.zeros((n, 32), dtype=torch.uint8, device=dev)
    one[:, 0] = 1
    px2, py2 = bx[:n].contiguous(), by[:n].contiguous()
    qx2, qy2 = bx[n:2 * n].contiguous(), by[n:2 * n].contiguous()
    o3 = [torch.empty((n, 32), dtype=torch.uint8, device=dev) for _ in range(3)]
    ms = timed(lambda: lib.bjj_add_batch_dev(ctx, n, dptr(px2), dptr(py2), dptr(one), dptr(qx2), dptr(qy2), dptr(one),
                                             dptr(o3[0]), dptr(o3[1]), dptr(o3[2]), sp), args.steps * 2)
    ea = ora.add(*[t[:1024].cpu().numpy() for t in (px2, py2, one, qx2, qy2, one)])
    assert all(np.array_equal(o3[k][:1024].cpu().numpy(), ea[k]) for k in range(3)), "add_batch parity"
    rate = n / (ms * 1e-3)
    out.append({"metric": "projective_adds_per_sec", "workload": "add_batch: 2^21 projective pairs (literal add-2008-bbjlp)",
                "value": rate, "unit": "adds/s", "ms_per_step": ms, "roofline_frac_imad": rate * ALGO_MAC["proj_add"] / imad_peak,
                "hbm_frac": rate * 288 / 1e9 / hbm_peak, "oracle_checked_lanes": 1024})
    return out


if __name__ == "__main__":
    main()
