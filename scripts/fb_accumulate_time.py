"""Time the table MSM's accumulation kernel (fixedmsm.cu `fb_accumulate_kernel`) at the Shot circuit's size.

Params at k = 11 with the window the library picks for Shot (window_bits = 0), and two launch shapes through
Params.commit_batch_dev:

  ipa      128 MSMs of uniform scalars with half the points zero: the shape of one IPA round of a batch of proofs
  advice   512 witness-like columns (70 % zero, 20 % one, 5 % below 2^10, 5 % uniform) committed in the Lagrange basis

For each shape: the whole commit call (decode, accumulate, fold) timed with CUDA events over --launches calls after
--warmup, the kernels of --profiled calls timed by torch.profiler, and the exact number of mixed additions per call
from the library's profiling counter.  One JSON line per shape on stdout.  The library is the one the package loads
(BZ_LIB selects another build, e.g. to compare two builds on the same GPU in one session)."""
import argparse, json, os, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

K = 11
N = 1 << K


def uniform(rng, shape):
    """uint64 limbs < 2^253: valid Montgomery residues of either field"""
    a = rng.integers(0, 2**63, size=shape + (4,), dtype=np.uint64)
    a[..., 3] &= np.uint64((1 << 61) - 1)
    return a


def ipa_shape(rng, count):
    polys = uniform(rng, (count, N))
    polys[rng.random((count, N)) < 0.5] = 0
    return polys, uniform(rng, (count,))


def advice_shape(rng, count):
    from oracle import c_oracle as co
    sf = co.CURVES[0][1]                                                         # Vesta's scalar field
    u = rng.random((count, N))
    polys = uniform(rng, (count, N))
    polys[u < 0.7] = 0
    polys[(u >= 0.7) & (u < 0.9)] = co.to_mont(sf, [1])[0]
    small = (u >= 0.9) & (u < 0.95)
    polys[small] = co.to_mont(sf, [int(v) for v in rng.integers(2, 1 << 10, size=int(small.sum()))])
    return polys, uniform(rng, (count,))


SHAPES = {"ipa": (ipa_shape, 128, False), "advice": (advice_shape, 512, True)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--shapes", default="ipa,advice")
    ap.add_argument("--launches", type=int, default=400, help="timed commit calls per shape (>= 200)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--profiled", type=int, default=50, help="commit calls per shape under torch.profiler")
    ap.add_argument("--window", type=int, default=0, help="window bits of the tables (0: the library's choice for k = 11)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fb_accumulate_time.py: no CUDA device")
    import battlezips_halo2_b200 as bz
    from battlezips_halo2_b200 import arithmetic as ar
    from battlezips_halo2_b200.binding import lib_path
    from battlezips_halo2_b200.plonk import prover as PR
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = bz.Context(0, stream=stream.cuda_stream)
    urs = ar.params_new(ctx, K, curve=0)
    params = PR.Params(ctx, K, urs["g"], urs["g_lagrange"], urs["w"], urs["u"], window_bits=args.window)
    props = torch.cuda.get_device_properties(0)
    rng = np.random.default_rng(2024)
    try:
        for name in args.shapes.split(","):
            make, count, lagrange = SHAPES[name]
            polys, blinds = make(rng, count)
            d_p = torch.from_numpy(np.ascontiguousarray(polys).view(np.int64)).cuda()
            d_b = torch.from_numpy(np.ascontiguousarray(blinds).view(np.int64)).cuda()
            d_o = torch.zeros((count, 8), dtype=torch.int64, device="cuda")
            call = lambda: params.commit_batch_dev(d_p.data_ptr(), d_b.data_ptr(), count, d_o.data_ptr(), lagrange=lagrange)
            for _ in range(args.warmup):
                call()
            torch.cuda.synchronize()
            # exact additions per call: the accumulate kernel counts them while profiling is on
            ctx.profile_enable(True)
            ctx.profile_counter(0, reset=True)
            call()
            torch.cuda.synchronize()
            adds = ctx.profile_counter(0, reset=True)
            ctx.profile_enable(False)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.launches):
                call()
            e1.record(stream)
            torch.cuda.synchronize()
            call_ms = e0.elapsed_time(e1) / args.launches
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                for _ in range(args.profiled):
                    call()
                torch.cuda.synchronize()
            kern = {}
            for ev in prof.key_averages():
                if "fb_" in ev.key and ev.self_device_time_total > 0:
                    short = ev.key.split("(")[0].split("<")[0].replace("void ", "").replace("bz::", "")
                    t, c = kern.get(short, (0.0, 0))
                    kern[short] = (t + ev.self_device_time_total / 1e3, c + ev.count)     # microseconds -> ms
            acc_ms = kern["fb_accumulate_kernel"][0] / kern["fb_accumulate_kernel"][1] if "fb_accumulate_kernel" in kern else None
            print(json.dumps({
                "shape": name, "msms": count, "k": K, "lagrange": lagrange, "mixed_adds_per_call": adds,
                "call_ms": round(call_ms, 5), "calls_timed": args.launches,
                "adds_per_s_call": adds / (call_ms / 1e3),
                "fb_accumulate_ms": round(acc_ms, 5) if acc_ms else None,
                "adds_per_s_accumulate": adds / (acc_ms / 1e3) if acc_ms else None,
                "kernel_ms": {k: round(t / c, 5) for k, (t, c) in sorted(kern.items())},
                "gpu": props.name, "lib": os.path.relpath(lib_path(), ROOT)}), flush=True)
            del d_p, d_b, d_o
    finally:
        params.close()
        ctx.close()


if __name__ == "__main__":
    main()
