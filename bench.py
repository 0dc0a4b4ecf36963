#!/usr/bin/env python
"""bench.py -- driver contract: `python bench.py --gpus N --steps K --warmup W [--impl reference]` prints ONE JSON line.

Workloads (BASELINE.json configs; `--workload`):
  shot  batched Shot proofs, k=11 (DEFAULT; config 3: independent proofs per GPU)  metric proofs_per_sec
  board Board proofs, k=12 (config 2)                                               metric proofs_per_sec
  commit  column commitments of one large proof, sharded per GPU     (config 5)   metric commit_points_per_sec
  msm   raw MSM over Vesta/Pallas, 2^LOG points resident in HBM       (config 4)   metric msm_points_per_sec
  ntt   Fp NTT / coset extension, 2^LOG elements                      (config 4)   metric ntt_gbytes_per_sec

A "step" = one pass of the hot path over one batch of synthetic input.  `value` = device-resident throughput,
`e2e` = same metric through the reference-facing C-ABI call with HOST buffers (H2D/D2H inside the timed
region).  `roofline` = dominant kernel, timed live with CUDA events on the launching stream (library profile
scopes).  `cpu_baseline` = the oracle (C restatement of halo2_proofs' rayon algorithms) on this box's host cores
over a bounded sample.  `--impl reference` times that CPU restatement alone (the Rust reference cannot be built
or run here: no cargo, crates not vendored -- DESIGN.md).  `--dump-outputs DIR` writes what the last device-resident
step computed (proof bytes, MSM point, NTT output or commitments) for output-for-output comparison of two builds.
"""
import argparse, json, os, subprocess, sys, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import numpy as np


def box_gpus(args):
    """GPUs this process can see on the box (no CUDA context is created): torch's device count, else CUDA_VISIBLE_DEVICES /
    /dev/nvidia<N>, else the launch size."""
    try:
        import torch
        n = torch.cuda.device_count()
        if n > 0:
            return n
    except Exception:      # noqa: BLE001
        pass
    import glob
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis is not None and vis.strip():
        return max(1, len([v for v in vis.split(",") if v.strip()]))
    n = len(glob.glob("/dev/nvidia[0-9]*"))
    return max(1, n or int(os.environ.get("LOCAL_WORLD_SIZE", args.gpus)))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("BZ_WORKLOAD", "shot"))
    ap.add_argument("--batch", type=int, default=int(os.environ.get("BZ_BATCH", "64")), help="proofs per step per GPU (shot / board)")
    ap.add_argument("--inflight", type=int, default=int(os.environ.get("BZ_INFLIGHT", "0")),
                    help="concurrent prover lanes per GPU (own host thread + CUDA stream each; shot / board); "
                         "0 = auto: one per host core available to this GPU, between 2 and 6")
    ap.add_argument("--log2n", dest="log", type=int, default=22, help="log2 of the problem size (msm / ntt workloads)")
    ap.add_argument("--k", type=int, default=16, help="rows = 2^k of the board_scaled workload (BASELINE config 5 asks k=20)")
    ap.add_argument("--curve", type=int, default=1, help="0 Vesta, 1 Pallas (msm workload)")
    ap.add_argument("--scalars", default="uniform", choices=["uniform", "witness"],
                    help="msm workload: uniform scalars, or SURVEY config 4 (W): 70 %% zero, 20 %% one, 5 %% in [2, 2^10), 5 %% uniform")
    ap.add_argument("--columns", type=int, default=32, help="independent column commitments per step (commit workload)")
    ap.add_argument("--cpu-sample-log", type=int, default=18)
    ap.add_argument("--no-extras", dest="extras", action="store_false",
                    help="default (shot) run only: skip the compact Board / MSM / NTT sub-benchmarks reported under `extras`")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last device-resident step computed as DIR/<name>.npy "
                         "(bytes as float32, at most 64 MB in all); inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.inflight <= 0:          # measured on 1xB200 / 16 cores: 4 lanes 3 153, 6 lanes 3 254, 8 lanes 3 286 Shot proofs/s
        try:
            cores = len(os.sched_getaffinity(0))
        except AttributeError:
            cores = os.cpu_count() or 4
        # the share of the box's cores one GPU gets -- from the GPUs the BOX has, not from --gpus, so that every N of a
        # scaling run on one box uses the same lanes x batch per GPU (weak scaling: per-GPU work fixed)
        args.inflight = max(2, min(6, cores // box_gpus(args)))
    return args


# ------------------------------------------------------------------------------------------------------
# fma-heavy pipe cost of one field multiplication in the shipped SASS, in IMAD-equivalents (issue slots of the pipe):
# 71 IMAD.WIDE.U32(.X) at HALF rate (measured: bz_imad_wide_peak = 0.455 x bz_imad_peak) = 142, plus 25 IMAD.HI + 11 IMAD +
# 18 IMAD.X at full rate = 54  ->  196  (cuobjdump -sass of fe_mul_raw; DESIGN.md §3)
FMA_PER_MUL = 196
def ncu_dram_bytes_per_add():
    """DRAM bytes fb_accumulate_kernel moves per mixed addition, from the newest committed `ncu --set full` capture:
    profiles/traffic.json is written by profiles/traffic.py out of profiles/*_ncu_full_summary.csv (dram__bytes_read.sum +
    dram__bytes_write.sum of the kernel / the additions of that launch).  None when no capture is committed."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return float(d["fb_accumulate_kernel"]["dram_bytes_per_add"]), d["fb_accumulate_kernel"]["source"]
    except Exception:      # noqa: BLE001
        return None, None


def set_sync_policy(args, local_rank):
    """Host threads that wait for a stream spin by default (CUDA's choice when cores outnumber contexts).  Measured on 1xB200
    with the process pinned to 4 cores (what an 8-GPU box leaves per GPU): 4 lanes spinning 3 212 proofs/s, 6 lanes spinning
    3 230, 6 lanes with blocking waits 3 160 (and 16 ms instead of 6.5 ms single-proof latency) -- so spinning stays, even
    oversubscribed.  BZ_BLOCKING_SYNC=1 switches the primary context to blocking waits BEFORE it is created (A/B)."""
    if os.environ.get("BZ_BLOCKING_SYNC") == "1":
        import ctypes
        cu = ctypes.CDLL("libcuda.so.1")
        dev = ctypes.c_int(0)
        ok = cu.cuInit(0) == 0 and cu.cuDeviceGet(ctypes.byref(dev), local_rank) == 0 and cu.cuDevicePrimaryCtxSetFlags_v2(dev, 4) == 0   # CU_CTX_SCHED_BLOCKING_SYNC
        return "blocking" if ok else "spin (could not set blocking)"
    return "spin"


def config_for(wl, sched="spin"):
    """The `config` object of the JSON line -- built the same way by the GPU arm and by --impl reference, so the two lines carry
    identical dicts."""
    if isinstance(wl, ProofWorkload):
        l2 = "per-step working set (window tables + batch work areas) far larger than L2; no flush needed"
    elif getattr(wl, "n", 0) * 96 > 126e6:
        l2 = "inputs larger than L2 (no flush needed)"
    else:
        l2 = "inputs < L2; not flushed"
    cfg = {"workload": wl.name, "l2": l2, "host_wait": sched}
    if isinstance(wl, ProofWorkload):
        cfg["lanes"] = "every lane proves its K batches back to back inside the timed region (independent proofs: no barrier between the steps of different lanes)"
    return cfg


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        if os.environ.get("BZ_NO_CLOCK_SAMPLER"):
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_LIMIT = 64 << 20


def dump_outputs(outputs, out_dir):
    """outputs: {name: array whose first axis indexes items}.  Every item is written as its bytes in float32 (exact); if
    that exceeds DUMP_LIMIT in all, every output keeps the same seeded random sample of a share of its items."""
    os.makedirs(out_dir, exist_ok=True)
    rows = {k: np.ascontiguousarray(v).view(np.uint8).reshape(len(v), -1) for k, v in outputs.items()}
    total = sum(4 * r.size for r in rows.values())
    budget = DUMP_LIMIT - 4096 * len(rows)                       # room for the .npy headers
    for name, r in rows.items():
        if total > budget:
            keep = max(1, len(r) * budget // total)
            r = r[np.sort(np.random.default_rng(0).choice(len(r), keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), r.astype(np.float32))


def rand_field(rng, n):
    """n x 4 uint64 limbs < 2^253: valid Montgomery residues of either field (synthetic data)."""
    a = rng.integers(0, 2**63, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 61) - 1)
    return a


def make_bases(co, curve, n):
    """n valid, pairwise distinct-looking curve points without n hash-to-curves: take 256 hash-derived points
    P_j and build B_i = P_{i mod 256} + [i div 256] Q' by repeated addition in the C oracle (setup only)."""
    import ctypes
    C = co.CURVES[curve][0]
    h = C.hash_to_curve("Halo2-Parameters")
    m = min(n, 256)
    seed = co.points_to_mont(curve, [h(b"\x00" + i.to_bytes(4, "little")) for i in range(m)])
    step = co.points_to_mont(curve, [h(b"\x01")])
    out = np.empty((n, 8), dtype=np.uint64)
    out[:m] = seed
    cur = seed.copy()
    tmp = np.empty(8, dtype=np.uint64)
    done = m
    while done < n:
        for j in range(m):
            co.lib().orc_point_add(curve, co._p(cur[j]), co._p(step), co._p(tmp))
            cur[j] = tmp
        take = min(m, n - done)
        out[done:done + take] = cur[:take]
        done += take
    return out


# ------------------------------------------------------------------------------------------------------
class MsmWorkload:
    dtype = "u32x8 (255-bit Montgomery, integer pipe)"

    def __init__(self, args):
        self.log, self.curve = args.log, args.curve
        self.n = 1 << self.log
        self.metric, self.unit = "msm_points_per_sec", "points/s"
        self.scalar_kind = getattr(args, "scalars", "uniform")
        kind = "uniform scalars" if self.scalar_kind == "uniform" else "witness-like scalars (70 % zero, 20 % one, 5 % below 2^10, 5 % uniform)"
        self.name = f"raw {'Pallas' if self.curve else 'Vesta'} MSM 2^{self.log} points, {kind} (BASELINE config 4)"

    def host_inputs(self, rank):
        from oracle import c_oracle as co            # setup only: valid curve points for the synthetic bases
        rng = np.random.default_rng(1234 + rank)
        t = time.time()
        # 2^16 distinct points tiled: the MSM cost does not depend on distinctness, setup time does
        m = min(self.n, 1 << 14)
        pts = make_bases(co, self.curve, m)
        bases = np.tile(pts, (self.n // m, 1))
        scalars = rand_field(rng, self.n)
        if self.scalar_kind == "witness":
            # Montgomery images of 0 .. 1023 as a table; the scalar field of curve id c is field id c (Vesta: Fp, Pallas: Fq)
            p = co.FIELDS[self.curve].p
            small = np.array([[((v << 256) % p >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)] for v in range(1024)], dtype=np.uint64)
            u = rng.random(self.n)
            pick = np.where(u < 0.70, 0, np.where(u < 0.90, 1, rng.integers(2, 1024, size=self.n)))
            scalars = np.where((u < 0.95)[:, None], small[pick], scalars)
        return scalars, bases

    def setup(self, ctx, rank):
        self.ctx = ctx
        world = int(os.environ.get("WORLD_SIZE", "1"))
        self.world = world
        if world > 1:
            # SURVEY §8e: ONE large MSM split by point range; every rank reduces its range, partials are all-gathered
            from battlezips_halo2_b200.sharding import shard_range
            sc, ba = self.host_inputs(0)                      # same global input on every rank
            lo, hi = shard_range(self.n, rank, world)
            self.n_total, self.n = self.n, hi - lo
            self.full = (sc, ba) if rank == 0 else None
            self.scalars, self.bases = np.ascontiguousarray(sc[lo:hi]), np.ascontiguousarray(ba[lo:hi])
            self.scaling = "strong"
        else:
            self.scalars, self.bases = self.host_inputs(rank)
        import torch
        self.h_scalars = torch.from_numpy(self.scalars.view(np.int64)).pin_memory()
        self.h_bases = torch.from_numpy(self.bases.view(np.int64)).pin_memory()
        self.d_scalars = ctx.to_device(self.scalars)
        self.d_bases = ctx.to_device(self.bases)
        self.d_out = ctx.alloc(96)
        if world > 1:
            self.t_jac = torch.zeros(12, dtype=torch.int64, device="cuda")
            self.t_all = torch.zeros((world, 12), dtype=torch.int64, device="cuda")
            self.t_sum = torch.zeros(8, dtype=torch.int64, device="cuda")
        self.h2d, self.d2h = self.n * 96, 96

    def _combine(self):
        """all-gather the 96 B Jacobian partials over NCCL and add them on the device (bz_point_sum_dev); no host round trip"""
        from battlezips_halo2_b200.sharding import allgather_point_sum_dev
        allgather_point_sum_dev(self.ctx, self.curve, self.t_jac, self.t_all, self.t_sum)

    def result_affine(self):
        return self.t_sum.cpu().numpy().view(np.uint64)

    def check(self):
        """N > 1: the all-gathered, summed result equals the un-split MSM of the whole input computed on rank 0's GPU"""
        if self.world == 1 or self.full is None:
            return None
        c = self.ctx
        sc, ba = self.full
        d_s, d_b, d_j, d_a = c.to_device(sc), c.to_device(ba), c.alloc(96), c.alloc(64)
        c._check(c.lib.bz_msm_dev(c.h, self.curve, d_s.ptr, d_b.ptr, self.n_total, d_j.ptr, 0))
        c._check(c.lib.bz_batch_normalize_dev(c.h, self.curve, d_j.ptr, d_a.ptr, 1))
        exp = d_a.download((8,))
        for d in (d_s, d_b, d_j, d_a):
            d.free()
        return bool(np.array_equal(exp, self.result_affine()))

    def step_device(self):
        import ctypes
        c = self.ctx
        if self.world > 1:
            c._check(c.lib.bz_msm_dev(c.h, self.curve, self.d_scalars.ptr, self.d_bases.ptr, self.n, ctypes.c_void_p(self.t_jac.data_ptr()), 0))
            self._combine()
            return self.n_total / self.world       # bench multiplies by world: total points once per step
        c._check(c.lib.bz_msm_dev(c.h, self.curve, self.d_scalars.ptr, self.d_bases.ptr, self.n, self.d_out.ptr, 0))
        return self.n

    def step_e2e(self):
        import ctypes
        c = self.ctx
        out = np.empty(12, dtype=np.uint64)
        c._check(c.lib.bz_best_multiexp(c.h, self.curve, ctypes.c_void_p(self.h_scalars.data_ptr()),
                                        ctypes.c_void_p(self.h_bases.data_ptr()), self.n, out.ctypes.data_as(ctypes.c_void_p)))
        if self.world > 1:
            import torch
            self.t_jac.copy_(torch.from_numpy(out.view(np.int64)))
            self._combine()
            return self.n_total / self.world
        return self.n

    def outputs(self):
        """the MSM result of the last device step as an affine point (Jacobian coordinates are not unique)"""
        if self.world > 1:
            return {"msm": self.result_affine()[None]}
        c = self.ctx
        d_a = c.alloc(64)
        c._check(c.lib.bz_batch_normalize_dev(c.h, self.curve, self.d_out.ptr, d_a.ptr, 1))
        out = d_a.download((1, 8))
        d_a.free()
        return {"msm": out}

    def dominant(self):
        # MSM algorithmic bytes: 32 B scalar + 64 B base per point (SURVEY §8d: 96*N); dominant kernel = bucket accumulation
        return "msm_bucket", 96.0 * self.n

    def close(self):
        for d in (self.d_scalars, self.d_bases, self.d_out):
            d.free()
        self.h_scalars = self.h_bases = None

    def cpu(self, sample_log, steps=1):
        from oracle import c_oracle as co
        m = 1 << min(sample_log, self.log)
        s, b = self.scalars[:m].copy(), self.bases[:m].copy()
        co.best_multiexp(self.curve, s[:1024], b[:1024])
        t = time.perf_counter()
        for _ in range(steps):
            co.best_multiexp(self.curve, s, b)
        dt = (time.perf_counter() - t) / steps
        return m / dt, f"best_multiexp restated (C, {co.get_threads()} threads) on the first 2^{min(sample_log, self.log)} points of the same input", co.get_threads(), dt


class NttWorkload:
    dtype = "u32x8 (255-bit Montgomery, integer pipe)"

    def __init__(self, args):
        self.log = args.log
        self.n = 1 << self.log
        self.metric, self.unit = "ntt_gbytes_per_sec", "GB/s"
        self.name = f"Fp forward NTT 2^{self.log} (64*N algorithmic bytes) (BASELINE config 4)"

    def setup(self, ctx, rank):
        import torch
        self.ctx = ctx
        rng = np.random.default_rng(99 + rank)
        self.a = rand_field(rng, self.n)
        self.h_a = torch.from_numpy(self.a.view(np.int64)).pin_memory()
        self.d_a = ctx.to_device(self.a)
        self.d_b = ctx.alloc(self.n * 32)
        self.h2d = self.d2h = self.n * 32
        F = ctx  # omega for the host-API call
        p = 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001
        root = 0x2bce74deac30ebda362120830561f81aea322bf2b7bb7584bdad6fabd87ea32f
        om = pow(root, 1 << (32 - self.log), p)
        self.omega = np.frombuffer(((om << 256) % p).to_bytes(32, "little"), dtype=np.uint64).copy()

    def step_device(self):
        c = self.ctx
        c._check(c.lib.bz_ntt_dev(c.h, 0, self.d_a.ptr, self.d_b.ptr, self.log, 0, 1))
        return 64.0 * self.n / 1e9

    def step_e2e(self):
        import ctypes
        c = self.ctx
        c._check(c.lib.bz_best_fft(c.h, 0, ctypes.c_void_p(self.h_a.data_ptr()), self.omega.ctypes.data_as(ctypes.c_void_p), self.log))
        return 64.0 * self.n / 1e9

    def outputs(self):
        return {"ntt": self.d_b.download((self.n, 4))}

    def dominant(self):
        npass = 1 if self.log <= 12 else (2 if self.log <= 20 else 3)
        return "ntt_pass", 64.0 * self.n / npass      # per launch: each pass reads+writes the array once

    def field_muls(self):
        return (self.n // 2) * self.log               # butterflies of one transform (SURVEY §8d)

    def close(self):
        self.d_a.free(); self.d_b.free()
        self.h_a = None

    def cpu(self, sample_log, steps=1):
        from oracle import c_oracle as co
        lg = min(sample_log + 2, self.log)
        a = self.a[: 1 << lg].copy()
        p = 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001
        root = 0x2bce74deac30ebda362120830561f81aea322bf2b7bb7584bdad6fabd87ea32f
        om = co.to_mont(0, [pow(root, 1 << (32 - lg), p)])
        t = time.perf_counter()
        for _ in range(steps):
            co.best_fft(0, a, om, lg)
        dt = (time.perf_counter() - t) / steps
        return 64.0 * (1 << lg) / 1e9 / dt, f"best_fft restated (C, {co.get_threads()} threads) at 2^{lg}", co.get_threads(), dt


class CommitWorkload:
    """Params::commit of `columns` independent polynomials of 2^k uniform scalars (the large-column commit of BASELINE config 5),
    column-sharded across the GPUs of the job; the commitments are all-gathered (64 B each)."""
    dtype = "u32x8 (255-bit Montgomery, integer pipe)"

    def __init__(self, args):
        self.k, self.M = args.k, args.columns
        self.n = 1 << self.k
        self.metric, self.unit = "commit_points_per_sec", "points/s"
        self.scaling = "strong"
        self.name = (f"Params::commit of {self.M} independent columns of 2^{self.k} uniform scalars, device URS from Params::new, "
                     f"columns sharded per GPU + all-gather of the commitments (BASELINE config 5 / north-star column sharding)")

    def setup(self, ctx, rank):
        import torch
        from battlezips_halo2_b200 import arithmetic as ar
        from battlezips_halo2_b200.plonk import prover as PR
        from battlezips_halo2_b200.sharding import shard_range
        self.ctx, self.rank = ctx, rank
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.urs = ar.params_new(ctx, self.k, curve=0)
        self.params = PR.Params(ctx, self.k, self.urs["g"], self.urs["g_lagrange"], self.urs["w"], self.urs["u"])
        self.lo, self.hi = shard_range(self.M, rank, self.world)
        self.per = (self.M + self.world - 1) // self.world
        cnt = self.hi - self.lo
        rng = np.random.default_rng(777)                      # every rank draws the same global columns, keeps its range
        cols = []
        for j in range(self.M):
            c = rand_field(rng, self.n)
            if self.lo <= j < self.hi or (rank == 0 and j in (0, self.M - 1)):
                cols.append((j, c))
        mine = [c for j, c in cols if self.lo <= j < self.hi]
        self.sample = {j: c for j, c in cols if j in (0, self.M - 1)} if rank == 0 else {}
        self.blinds_np = rand_field(np.random.default_rng(778), self.M)
        host = np.stack(mine) if mine else np.zeros((1, self.n, 4), np.uint64)
        self.h_polys = torch.from_numpy(host.view(np.int64)).pin_memory()
        self.d_polys = torch.empty_like(self.h_polys, device="cuda")
        self.d_polys.copy_(self.h_polys)
        self.d_blinds = torch.from_numpy(np.ascontiguousarray(self.blinds_np[self.lo:self.hi] if cnt else self.blinds_np[:1]).view(np.int64)).cuda()
        self.d_local = torch.zeros((self.per, 8), dtype=torch.int64, device="cuda")
        self.cnt = cnt
        self.h2d, self.d2h = int(cnt * self.n * 32), int(self.M * 64)
        torch.cuda.synchronize()

    def _commit(self):
        from battlezips_halo2_b200.sharding import allgather_commitments
        if self.cnt:
            self.params.commit_batch_dev(self.d_polys.data_ptr(), self.d_blinds.data_ptr(), self.cnt, self.d_local.data_ptr())
        self.result = allgather_commitments(self.d_local, self.M, self.rank, self.world)
        return self.M * self.n / self.world       # bench multiplies by world: all columns once per step

    def step_device(self):
        return self._commit()

    def step_e2e(self):
        self.d_polys.copy_(self.h_polys, non_blocking=True)
        units = self._commit()
        self.h_result = self.result.cpu()
        return units

    def outputs(self):
        return {"commitments": self.result.cpu().numpy()}

    def dominant(self):
        tag = "fixed_msm" if self.k <= 19 else "msm_bucket"
        return tag, 96.0 * self.n

    def check(self):
        """rank 0: the gathered commitments of the first and last column equal the single-call Params::commit"""
        if self.rank != 0:
            return None
        res = self.result.cpu().numpy().view(np.uint64)
        for j, col in self.sample.items():
            exp = self.params.commit(col, self.blinds_np[j])
            if not np.array_equal(res[j], exp):
                return False
        return True

    def cpu(self, sample_log, steps=1):
        from oracle import c_oracle as co
        m = 1 << min(sample_log, self.k)
        col = next(iter(self.sample.values())) if self.sample else rand_field(np.random.default_rng(1), m)
        s, b = np.ascontiguousarray(col[:m]), np.ascontiguousarray(self.urs["g"][:m])
        t = time.perf_counter()
        for _ in range(steps):
            co.best_multiexp(0, s, b)
        dt = (time.perf_counter() - t) / steps
        return m / dt, f"best_multiexp restated (C, {co.get_threads()} threads) on the first 2^{min(sample_log, self.k)} terms of one column", co.get_threads(), dt

    def close(self):
        self.params.close()
        self.d_polys = self.h_polys = None


class ProofWorkload:
    """create_proof for a batch of independent proofs of the Shot (k=11) or Board (k=12) circuit mirror.
    unit = proofs; every proof has its own RNG stream; witnesses cycle over 8 distinct synthetic jobs."""
    dtype = "u32x8 (255-bit Montgomery, integer pipe)"
    metric, unit = "proofs_per_sec", "proofs/s"
    DISTINCT = int(os.environ.get("BZ_DISTINCT", "32"))      # distinct synthetic witnesses the batch cycles over (config 3: pattern x shot cell)

    def __init__(self, args, which):
        self.which, self.B, self.T = which, args.batch, max(1, args.inflight)
        self.k = 11 if which == "shot" else 12
        if which == "board_scaled":          # BASELINE config 5: Board replicated down a 2^k-row table
            self.k, self.B, self.T, self.DISTINCT = args.k, 1, 1, 1
        if which == "board_scaled":
            self.world = int(os.environ.get("WORLD_SIZE", "1"))
            self.scaling = "strong" if self.world > 1 else "weak"
            self.name = (f"Board circuit replicated to k={self.k} (many boards per proof), ONE proof"
                         + (f" across {self.world} GPUs: commitment MSMs dealt out by column / split by point range, NCCL all-gather of the 96 B results"
                            if self.world > 1 else "") + ", URS from Params::new on the device (BASELINE config 5)")
            return
        self.name = (f"batched {'Shot' if which == 'shot' else 'Board'} proofs (k={self.k}, IPA/Pasta), {self.T} lanes x {self.B} independent "
                     f"proofs per GPU per step, synthetic witnesses (BASELINE config {'3' if which == 'shot' else '2'})")

    def _jobs(self, rank):
        from battlezips_halo2_b200.circuits import shot_circuit, board_circuit
        from battlezips_halo2_b200.plonk import prover as PR
        make = shot_circuit if self.which == "shot" else board_circuit
        if self.which == "board_scaled":
            from battlezips_halo2_b200.circuits import board_circuit_scaled
            jobs = [board_circuit_scaled(self.k, seed=0)]          # every rank proves the SAME circuit when the proof is sharded
        else:
            jobs = [make(rank * 1000 + i) for i in range(self.DISTINCT)]
        cs, _, asg0 = jobs[0]
        self.ir = cs.to_ir()
        self.asg0 = asg0
        n = 1 << self.k
        adv = np.stack([np.stack([PR.mont(col) for col in asg.advice]) for _, _, asg in jobs])        # (D, G, n, 4)
        self.instances_d = [asg.instance for _, _, asg in jobs]
        return adv

    def _num_random(self):
        ir, n = self.ir, 1 << self.k
        bf, G, L = ir["blinding_factors"], ir["num_advice"], len(ir["lookups"])
        chunk = ir["degree"] - 2
        nsets = (len(ir["permutation"]) + chunk - 1) // chunk
        return G * (bf + 1) + G + L * (2 * (bf + 1) + 2) + nsets * (bf + 1) + L * (bf + 1) + n + 1 + (ir["degree"] - 1) + 1 + n + 1 + 2 * self.k

    def _wide(self, rank, count):
        """count x R x 8 uint64 RNG words (SplitMix64 streams; every proof its own seed)."""
        R = self._num_random()
        out = np.empty((count, R, 8), dtype=np.uint64)
        for i in range(count):
            idx = np.arange(1, 8 * R + 1, dtype=np.uint64)
            with np.errstate(over="ignore"):
                z = np.uint64(0xB200B200B200B200 + rank * 1000003 + i) + idx * np.uint64(0x9E3779B97F4A7C15)
                z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
                z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
                z = z ^ (z >> np.uint64(31))
            out[i] = z.reshape(R, 8)
        return out

    def setup(self, ctx, rank):
        import torch, ctypes
        import battlezips_halo2_b200 as bz
        from battlezips_halo2_b200.plonk import prover as PR
        from concurrent.futures import ThreadPoolExecutor
        self.ctx, self.PR = ctx, PR
        adv_d = self._jobs(rank)
        fxp = os.path.join(ROOT, "tests", "golden", f"params_vesta_k{self.k}.npz")
        if os.path.exists(fxp):
            fx = np.load(fxp)
        else:
            fx = self._synthetic_urs(ctx)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(ctx.device)[0]
        t0 = time.perf_counter()
        self.params = PR.Params(ctx, self.k, fx["g"], fx["g_lagrange"], fx["w"], fx["u"])     # window tables: shared by all lanes
        ctx.sync()
        self.setup_info = {"params_table_build_s": round(time.perf_counter() - t0, 3), "params_hbm_bytes": int(free0 - torch.cuda.mem_get_info(ctx.device)[0]),
                           "note": "one-off per Params (outside the timed steps): window tables of g || w || u and g_lagrange || w"}
        self.fx = fx
        B, T = self.B, self.T
        ni = self.ir["num_instance"]
        self.lens = np.array([len(self.instances_d[0][i]) for i in range(ni)], dtype=np.uint32)
        self.stride = int(self.lens.max())
        mapping = self.asg0.permutation_mapping()
        self.lanes = []
        sharded = self.which == "board_scaled" and getattr(self, "world", 1) > 1
        wide_all = self._wide(0 if sharded else rank, B * T)
        self.sharded = sharded
        if sharded:
            # exchange buffers: the MSM partial sums are tiny; the point-range split of h(X) moves (8n + 4n + 2n) x 32 B per proof
            ctx.set_sharding(rank, self.world, capacity=14 * (1 << self.k) * 32 // self.world + (1 << 16))
        for t in range(T):
            lane = {}
            lane["stream"] = torch.cuda.current_stream() if t == 0 else torch.cuda.Stream()
            lane["ctx"] = ctx if t == 0 else bz.Context(ctx.device, stream=lane["stream"].cuda_stream)
            lane["pk"] = PR.ProvingKey(lane["ctx"], self.params, self.ir, self.asg0.fixed, mapping, 0x1234567890ABCDEF1234567890ABCDEF)
            sel = [(t * B + i) % self.DISTINCT for i in range(B)]
            lane["sel"] = sel
            advice = np.ascontiguousarray(adv_d[sel])                        # (B, G, n, 4)
            wide = np.ascontiguousarray(wide_all[t * B:(t + 1) * B])
            inst = np.zeros((B, ni, self.stride, 4), dtype=np.uint64)
            for b in range(B):
                for i in range(ni):
                    inst[b, i, :self.lens[i]] = PR.mont(self.instances_d[sel[b]][i])
            lane["proofs"] = np.zeros((B, lane["pk"].proof_size), dtype=np.uint8)
            ones = np.tile(PR.mont([1])[0], (advice.shape[0], advice.shape[1], advice.shape[2], 1))       # Assigned::Trivial: denominator one
            lane["h"] = [torch.from_numpy(x.view(np.int64)).pin_memory() for x in (inst, advice, wide, ones)]
            lane["d"] = [h.to(f"cuda:{ctx.device}") for h in lane["h"][:3]]
            lane["d_den"] = torch.empty_like(lane["h"][3], device=f"cuda:{ctx.device}")
            lane["d_adv_e2e"] = torch.empty_like(lane["h"][1], device=f"cuda:{ctx.device}")
            lane["step"] = 0
            lane["bytes"] = advice.nbytes + wide.nbytes + inst.nbytes + ones.nbytes
            self.lanes.append(lane)
        self.advice, self.wide = np.ascontiguousarray(adv_d[:1]), wide_all[:2]
        self.pk = self.lanes[0]["pk"]
        self.setup_info["work_hbm_bytes"] = int(free0 - torch.cuda.mem_get_info(ctx.device)[0]) - self.setup_info["params_hbm_bytes"]
        self.setup_info["distinct_witnesses"] = self.DISTINCT
        self.h2d = sum(l["bytes"] for l in self.lanes)
        self.d2h = sum(l["proofs"].nbytes for l in self.lanes)
        self.pool = ThreadPoolExecutor(T)

    def _synthetic_urs(self, ctx):
        """k > 13: no committed URS fixture; Params::new(k) runs on the device (hash-to-curve x 2^k + group inverse FFT), so
        these proofs are real and verified on the device; the (slow) oracle cross-check is skipped at these sizes."""
        from battlezips_halo2_b200 import arithmetic as ar
        self.device_urs = True
        return ar.params_new(ctx, self.k, curve=0)

    STEP_INC = 0x9E3779B97F4A7C15 - (1 << 64)        # odd: every RNG word of every proof changes every step (fresh randomness per proof)

    def _lane_run(self, lane, device):
        """One create_proof call of a lane.  The RNG words are advanced first, so no two calls prove with the same randomness.
        device = True: inputs resident in HBM.  device = False (e2e): what the reference-facing host does per call -- the
        `Assigned` advice (numerators + denominators, host memory) goes through poly::batch_invert_assigned on the device,
        instances and RNG words are read from host memory by the call, proofs come back to host memory."""
        import ctypes, torch
        c = lane["ctx"]
        vp = ctypes.c_void_p
        lane["step"] += 1
        with torch.cuda.stream(lane["stream"]):
            if device:
                lane["d"][2].add_(self.STEP_INC)
                ptrs = [vp(d.data_ptr()) for d in lane["d"]]
            else:
                hw = lane["h"][2].numpy()
                np.add(hw, np.int64(self.STEP_INC), out=hw)
                lane["d_adv_e2e"].copy_(lane["h"][1], non_blocking=True)
                lane["d_den"].copy_(lane["h"][3], non_blocking=True)
                nel = lane["h"][1].numel() // 4
                c._check(c.lib.bz_batch_invert_assigned_dev(c.h, 0, vp(lane["d_adv_e2e"].data_ptr()), vp(lane["d_den"].data_ptr()), vp(lane["d_adv_e2e"].data_ptr()), nel))
                ptrs = [vp(lane["h"][0].data_ptr()), vp(lane["d_adv_e2e"].data_ptr()), vp(lane["h"][2].data_ptr())]
        c._check(c.lib.bz_create_proofs(c.h, lane["pk"].h, self.B, ptrs[0], self.lens.ctypes.data_as(ctypes.c_void_p), self.stride,
                                        ptrs[1], ptrs[2], lane["proofs"].ctypes.data_as(ctypes.c_void_p)))

    def _run(self, device):
        futs = []
        for lane in self.lanes:
            futs.append(self.pool.submit(self._lane_run, lane, device))
        for f in futs:
            f.result()
        if self.which == "board_scaled" and getattr(self, "world", 1) > 1:
            return self.B * self.T / self.world          # one proof per step for the whole job
        return self.B * self.T

    def step_device(self):
        return self._run(True)

    def step_e2e(self):
        return self._run(False)

    def run_steps(self, device, steps):
        """K steps with the lanes free-running: every lane issues its K create_proof calls back to back, the way a proving
        service keeps its GPU fed.  With a barrier after every step all lanes would stage their next inputs (host -> device
        copies, witness inversion) at the same moment and leave the GPU idle meanwhile.  A sharded proof (collectives inside
        the call) stays in lockstep."""
        if getattr(self, "sharded", False) or len(self.lanes) == 1:
            return sum(self._run(device) for _ in range(steps))

        def loop(lane):
            for _ in range(steps):
                self._lane_run(lane, device)
        for f in [self.pool.submit(loop, lane) for lane in self.lanes]:
            f.result()
        return self.B * self.T * steps

    def outputs(self):
        """proof bytes of the last call of every lane; row t * B + i is proof i of lane t, whose witness and RNG stream
        depend on that row alone"""
        return {"proofs": np.concatenate([lane["proofs"] for lane in self.lanes])}

    def single_latency(self, reps=7):
        """latency of ONE proof (batch 1, one lane, device-resident inputs): median wall ms of `reps` calls"""
        import ctypes
        lane = self.lanes[0]
        c = lane["ctx"]
        out = np.zeros((1, lane["pk"].proof_size), dtype=np.uint8)
        ts = []
        for _ in range(reps + 2):
            t0 = time.perf_counter()
            c._check(c.lib.bz_create_proofs(c.h, lane["pk"].h, 1, ctypes.c_void_p(lane["d"][0].data_ptr()), self.lens.ctypes.data_as(ctypes.c_void_p), self.stride,
                                            ctypes.c_void_p(lane["d"][1].data_ptr()), ctypes.c_void_p(lane["d"][2].data_ptr()), out.ctypes.data_as(ctypes.c_void_p)))
            ts.append(1e3 * (time.perf_counter() - t0))
        return float(np.median(ts[2:]))

    def step_profile(self):
        self._lane_run(self.lanes[0], True)
        return self.B

    def all_contexts(self):
        return [l["ctx"] for l in self.lanes]

    def close(self):
        self.pool.shutdown()
        for lane in self.lanes:
            lane["d"] = lane["h"] = lane["d_den"] = lane["d_adv_e2e"] = None
            lane["pk"].close()
            if lane["ctx"] is not self.ctx:
                lane["ctx"].close()
        self.params.close()
        self.lanes = []
        if self.which == "board_scaled" and getattr(self, "world", 1) > 1:
            self.ctx.set_sharding(0, 1)

    def dominant(self):
        # fixed-base MSM: algorithmic bytes = one 64 B table point per mixed addition + 32 B per scalar read
        return "fixed_msm", None

    def check(self):
        """EVERY proof of the last step goes through verify_proof on the device (bz_verify_proofs: one verdict per proof);
        the restated reference verifier (oracle) cross-checks the first and last proof of the first and last lane."""
        PR = self.PR
        for lane in self.lanes:
            lane["pk"].vk_commitments()           # keygen_vk's commitments: once per key, not part of verify_proof
        t0 = time.perf_counter()
        total, accepted = 0, 0
        for lane in self.lanes:
            res = PR.verify_proofs(lane["pk"], [self.instances_d[s] for s in lane["sel"]], [bytes(lane["proofs"][b]) for b in range(self.B)])
            total += len(res); accepted += sum(res)
        dt = time.perf_counter() - t0
        self.verify_info = {"proofs": total, "accepted": accepted, "device_verify_proofs_per_sec": total / dt,
                            "note": "bz_verify_proofs, host transcript + device MSM check, single host thread"}
        if accepted != total:
            return False
        if getattr(self, "device_urs", False):
            return True
        from oracle import halo2 as H
        op = H.Params(self.k, 0, self.fx["g"], self.fx["g_lagrange"], self.fx["w"], self.fx["u"])
        opk = H.keygen(op, self.ir, self.asg0.fixed, self.asg0.permutation_mapping(), vk_repr=0x1234567890ABCDEF1234567890ABCDEF)
        for lane in (self.lanes[0], self.lanes[-1]):
            for b in sorted({0, self.B - 1}):
                if not H.verify_proof(op, opk, self.instances_d[lane["sel"][b]], bytes(lane["proofs"][b])):
                    return False
        self._oracle = (H, op, opk)
        return True

    def cpu(self, sample_log, steps=1):
        """restated halo2_proofs prover (oracle: Python protocol order over the C rayon-style arithmetic)"""
        from oracle import halo2 as H, c_oracle as co
        if not hasattr(self, "_oracle"):
            fx = self.fx if hasattr(self, "fx") else np.load(os.path.join(ROOT, "tests", "golden", f"params_vesta_k{self.k}.npz"))
            op = H.Params(self.k, 0, fx["g"], fx["g_lagrange"], fx["w"], fx["u"])
            opk = H.keygen(op, self.ir, self.asg0.fixed, self.asg0.permutation_mapping(), vk_repr=0x1234567890ABCDEF1234567890ABCDEF)
            self._oracle = (H, op, opk)
        H, op, opk = self._oracle
        nproofs = max(1, steps)
        co.call_timing(True)
        t = time.perf_counter()
        phases = {}
        for i in range(nproofs):
            T = H.Blake2bTranscript(0)
            trace = {}
            H.create_proof(op, opk, self.instances_d[0], [self.advice[0][g] for g in range(self.advice.shape[1])], H.Draws(self.wide[i % len(self.wide)]), T, trace=trace)
            for name, sec in trace.get("phase_s", {}).items():
                phases[name] = phases.get(name, 0.0) + 1e3 * sec / nproofs
        dt = (time.perf_counter() - t) / nproofs
        native_s, native_calls = co.call_timing(False)
        self.cpu_native = {"native_share": round(native_s / (dt * nproofs), 4), "native_calls_per_proof": native_calls // nproofs,
                           "note": "share of the CPU prover's wall time spent inside the C arithmetic library (the rest is the Python protocol driver)"}
        self.cpu_phases_ms = {k: round(v, 2) for k, v in phases.items()}        # the Amdahl picture of the CPU path (SURVEY 8d)
        return 1.0 / dt, (f"{nproofs} {self.which} proof(s) with the restated halo2_proofs 0.2.0 prover (oracle/halo2.py over the C restatement, "
                          f"{co.get_threads()} threads)"), co.get_threads(), dt


WORKLOADS = {"msm": MsmWorkload, "ntt": NttWorkload, "shot": lambda a: ProofWorkload(a, "shot"), "board": lambda a: ProofWorkload(a, "board"),
             "board_scaled": lambda a: ProofWorkload(a, "board_scaled"), "commit": CommitWorkload}


# ------------------------------------------------------------------------------------------------------
def run_reference(args, rank):
    """--impl reference: the CPU restatement of the reference path on this box's host cores (rank 0 only)."""
    if rank != 0:
        return
    wl = WORKLOADS[args.workload](args)
    if isinstance(wl, ProofWorkload):
        wl.advice = wl._jobs(0)[:1]
        wl.wide = wl._wide(0, 2)
    elif hasattr(wl, "host_inputs"):
        wl.scalars, wl.bases = wl.host_inputs(0)
    else:
        wl.a = rand_field(np.random.default_rng(99), wl.n)
    for _ in range(max(1, min(args.warmup, 1))):
        wl.cpu(args.cpu_sample_log - 2)
    vals, dts = [], []
    for _ in range(args.steps):
        v, sample, cores, dt = wl.cpu(args.cpu_sample_log)
        vals.append(v); dts.append(dt)
    v = float(np.median(vals))           # BASELINE.md section 3: median of the timed runs (the driver asks for 20)
    extra = {"runs": len(vals), "value_min_max": [float(min(vals)), float(max(vals))]}
    if isinstance(wl, ProofWorkload):
        from oracle import c_oracle as co
        extra["cpu_phases_ms"] = getattr(wl, "cpu_phases_ms", None)
        extra["cpu_native"] = getattr(wl, "cpu_native", None)
        nthreads = co.get_threads()
        co.set_threads(1)                    # the same proof on one host thread (SURVEY 8d asks for both figures)
        try:
            v1, _, _, _ = wl.cpu(args.cpu_sample_log)
            extra["one_thread"] = {"value": v1, "unit": wl.unit, "phases_ms": getattr(wl, "cpu_phases_ms", None)}
        finally:
            co.set_threads(nthreads)
    print(json.dumps({
        **extra,
        "impl": "reference", "metric": wl.metric, "value": v, "unit": wl.unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * float(np.median(dts)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
        "config": config_for(wl), "note": "restated halo2_proofs 0.2.0 arithmetic (C oracle); the rustc reference cannot be built here",
        "cpu_baseline": {"value": v, "unit": wl.unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def measure(args, wl, ctx, stream, rank, world, local_rank, want_cpu=True, steps=None, warmup=None, dump_dir=None):
    """One workload, three timed passes (device-resident, per-kernel profile, end-to-end with host buffers) -> dict.
    dump_dir: rank 0 writes the outputs of the device-resident pass's last step there (dump_outputs)."""
    import torch
    import torch.distributed as dist
    steps = steps or args.steps
    warmup = warmup or args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ----
    for _ in range(warmup):
        wl.step_device()
    barrier()
    ctxs = wl.all_contexts() if hasattr(wl, "all_contexts") else [ctx]
    launches0 = sum(c.kernel_launches() for c in ctxs)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    units = wl.run_steps(True, steps) if hasattr(wl, "run_steps") else sum(wl.step_device() for _ in range(steps))
    e1.record(stream)
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clocks = sampler.stop() if rank == 0 else None
    launches = sum(c.kernel_launches() for c in ctxs) - launches0
    if dump_dir and rank == 0:          # before the passes below overwrite the outputs
        dump_outputs(wl.outputs(), dump_dir)
    # ---- per-kernel pass: the same steps on ONE lane with the library's CUDA-event scopes on, so every kernel is
    # timed alone on the GPU (with several lanes in flight, kernels of different lanes overlap and a per-kernel
    # duration would measure the time-slicing, not the kernel).  The roofline / int_pipe objects come from here.
    ctx.profile_enable(True)
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for _ in range(steps):
        (wl.step_profile if hasattr(wl, "step_profile") else wl.step_device)()
    p1.record(stream)
    barrier()
    prof_ms = p0.elapsed_time(p1)
    prof = dict(ctx.profile_read())
    adds_total = ctx.profile_counter(0)
    ctx.profile_enable(False)

    # ---- end-to-end through the host-buffer ABI (H2D + D2H inside the timed region) ----
    for _ in range(min(warmup, 2)):
        wl.step_e2e()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    t0 = time.perf_counter()
    units_e = wl.run_steps(False, steps) if hasattr(wl, "run_steps") else sum(wl.step_e2e() for _ in range(steps))
    e3.record(stream)
    barrier()
    wall_e = time.perf_counter() - t0
    ms_e = torch.tensor([max(e2.elapsed_time(e3), 1e3 * wall_e)], device="cuda")   # host-synchronous calls: wall clock bounds it
    if world > 1:
        dist.all_reduce(ms_e, op=dist.ReduceOp.MAX)
    ms_e = float(ms_e.item())
    # a sharded proof exchanges partial sums in every MSM: its single-proof latency needs all ranks in the call
    single_ms = wl.single_latency() if hasattr(wl, "single_latency") and (rank == 0 or getattr(wl, "sharded", False)) else None
    if rank != 0:
        return None
    value = units * world / (ms / 1e3)
    e2e_value = units_e * world / (ms_e / 1e3)
    tag, alg_bytes = wl.dominant()
    if tag not in prof and prof:                     # e.g. k >= 18: commitments go through the bucket MSM
        tag = max(prof, key=lambda t: prof[t][0])
        alg_bytes = 0.0
    peak, peak_kind = peaks()
    roof = None
    int_pipe = None
    if tag == "fixed_msm" and tag in prof:
        adds = adds_total
        tot_ms, cnt = prof[tag]
        alg_bytes = adds * 64.0 / cnt      # per launch: one 64 B table entry per mixed addition
        imad_peak = ctx.imad_peak()
        # 10 field multiplications (8M + 2S) per mixed addition; I = fma-pipe issue slots per multiplication in the
        # shipped SASS (cuobjdump count, DESIGN.md)
        fmul_per_s = adds * 10.0 / (tot_ms / 1e3)
        int_pipe = {"kernel": tag, "mixed_adds_per_step": adds / steps, "field_mul_per_s": fmul_per_s, "fma_pipe_instr_per_field_mul_sass": FMA_PER_MUL,
                    "imad_peak_measured_per_s": imad_peak, "frac_of_imad_peak": fmul_per_s * FMA_PER_MUL / imad_peak}
    elif hasattr(wl, "field_muls") and tag in prof:
        tot_ms, cnt = prof[tag]
        imad_peak = ctx.imad_peak()
        fmul_per_s = wl.field_muls() * steps / (tot_ms / 1e3)
        int_pipe = {"kernel": tag, "field_mul_per_s": fmul_per_s, "fma_pipe_instr_per_field_mul_sass": FMA_PER_MUL,
                    "imad_peak_measured_per_s": imad_peak, "frac_of_imad_peak": fmul_per_s * FMA_PER_MUL / imad_peak}
    if tag in prof:
        tot_ms, cnt = prof[tag]
        avg_s = tot_ms / cnt / 1e3
        ach = alg_bytes / avg_s / 1e9
        # DRAM bytes per launch from the committed ncu --set full capture of this kernel (profiles/): fb_accumulate moves
        # 129.8 B per mixed addition (dram__bytes_read + write = 324.6 MB for 2.50 M additions, r1d) -- two 32 B sectors of
        # the table entry plus sector over-fetch on the entry list -- against 64 B algorithmic
        per_add, traffic_src = ncu_dram_bytes_per_add()
        traffic = (adds_total / cnt) * per_add if tag == "fixed_msm" and adds_total and per_add else None
        roof = {"bound": "hbm", "kernel": tag, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": traffic_src if traffic else None, "peak_kind": peak_kind, "avg_launch_ms": tot_ms / cnt, "launches": cnt,
                "share_of_step": tot_ms / prof_ms, "measured": "single-lane pass of the same steps, CUDA-event scopes in the library",
                "kernel_ms": {k: round(v[0], 4) for k, v in prof.items()}}
    cpu = None
    if want_cpu:
        v, sample, cores, _ = wl.cpu(args.cpu_sample_log)
        cpu = {"value": v, "unit": wl.unit, "cores": cores, "kind": "port", "sample": sample}
        if getattr(wl, "cpu_native", None):
            cpu.update(wl.cpu_native)
        if getattr(wl, "cpu_phases_ms", None):
            cpu["phases_ms"] = wl.cpu_phases_ms          # where the CPU prover spends its time, beside kernel_ms of the GPU arm
    return {
        "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": getattr(wl, "scaling", "weak"), "vs_baseline": None,
        "dtype": wl.dtype, "data": "synthetic",
        "config": config_for(wl),
        "e2e": {"value": e2e_value, "unit": wl.unit, "h2d_bytes_per_step": wl.h2d, "d2h_bytes_per_step": wl.d2h},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "int_pipe": int_pipe, "cpu_baseline": cpu,
        "verified": getattr(wl, "check", lambda: None)(), "verify": getattr(wl, "verify_info", None),
        "single_proof_ms": single_ms}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback")
    sched = set_sync_policy(args, local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        # a mismatched collective should fail in minutes, not after the default 10
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=int(os.environ.get("BZ_NCCL_TIMEOUT_S", "180"))))
    import battlezips_halo2_b200 as bz
    # a non-default torch stream: its handle is what libbzhalo2 launches on, so torch.cuda.Event timings on it
    # bracket exactly our kernels (the legacy default stream has handle 0, which the ABI reads as "private stream")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx = bz.Context(local_rank, stream=stream.cuda_stream)
    wl = WORKLOADS[args.workload](args)
    wl.setup(ctx, rank)
    line = measure(args, wl, ctx, stream, rank, world, local_rank, want_cpu=(rank == 0 and not os.environ.get("BZ_NO_CPU_BASELINE")),
                   dump_dir=args.dump_outputs)
    if line is not None:
        line["config"] = config_for(wl, sched)
        if getattr(wl, "setup_info", None):
            line["setup"] = wl.setup_info
    # ---- the other headline numbers of BASELINE.json's metric (Board proofs/s, MSM points/s, NTT GB/s) ride along in
    # the same JSON line as compact sub-benchmarks, so that one default run reports all of them
    extras = {}
    if args.workload == "shot" and args.extras:
        if hasattr(wl, "close"):
            wl.close()
        if os.environ.get("BZ_BENCH_VERBOSE"):
            print("free / total HBM after closing the headline workload:", torch.cuda.mem_get_info(local_rank), file=sys.stderr)
        names = ["board", "msm", "ntt", "commit", "scaled"] if world == 1 else ["board", "msm", "commit", "scaled"]
        for name in names:
            # an extra must never take the headline line down with it; under torchrun every rank takes the same branch
            # (setup errors are deterministic), so the collectives inside stay matched
            try:
                a2 = argparse.Namespace(**vars(args))
                if name == "commit":
                    a2.k, a2.columns = 18, 16
                if name == "scaled":                 # config 5 on the way up (k = 20 itself: --workload board_scaled --k 20, profiles/README.md)
                    a2.k = int(os.environ.get("BZ_SCALED_K", "16"))
                w2 = WORKLOADS["board_scaled" if name == "scaled" else name](a2)
                w2.setup(ctx, rank)
                r = measure(a2, w2, ctx, stream, rank, world, local_rank, want_cpu=False, steps=min(args.steps, 3), warmup=3)
                if hasattr(w2, "close"):
                    w2.close()
                if r is not None:
                    extras[name] = {k: r[k] for k in ("metric", "value", "unit", "ms_per_step", "scaling", "config", "e2e", "gpu_launches", "roofline", "int_pipe", "verified", "verify", "single_proof_ms")}
            except Exception as e:          # noqa: BLE001
                extras[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if rank == 0:
        if extras:
            line["extras"] = extras
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
