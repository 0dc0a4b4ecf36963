"""Blinding randomness from the host vs. from a seed: wall time of create_proofs fed a host-generated ChaCha20 keystream
(the `cryptography` package's C ChaCha20, the best case for generating the stream on the host) against create_proofs_seeded,
which uploads 32 bytes per proof and expands the same stream on the device.  Both paths give the same proof bytes; this script
checks that once per workload before timing.

Workloads: Shot (k = 11) and Board (k = 12) at batch 64, the scaled Board at k = 16 and k = 20 at batch 1.  The two paths are
timed alternately, --reps times each after --warmup rounds; every timed call ends with its proofs on the host (the calls are
synchronous).  Also reported: the host-side keystream generation alone, H2D bytes per proof of each path (computed from
num_random), and the fill kernel's device time from CUDA events (bz_chacha20_blocks into device memory with profiling on).

    python scripts/seeded_rng_time.py [--reps 20] [--warmup 2] [--workloads shot,board,board16,board20] [--out FILE]
"""
import argparse, json, os, statistics, subprocess, sys, time
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def host_keystream(seeds, blocks):
    """(B, blocks, 8) uint64 rand_wide from cryptography's ChaCha20 (all-zero 16-byte nonce = counter 0, stream id 0)."""
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms
    zeros = bytes(64 * blocks)
    out = np.empty((len(seeds), blocks * 8), dtype=np.uint64)
    for b, s in enumerate(seeds):
        enc = Cipher(algorithms.ChaCha20(bytes(s), b"\0" * 16), mode=None).encryptor()
        out[b] = np.frombuffer(enc.update(zeros), dtype="<u8")
    return out.reshape(len(seeds), blocks, 8)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def build(ctx, which):
    """(pk, params, instances, advice, batch) of one workload; URS from the fixtures or from Params::new on the device."""
    from battlezips_halo2_b200 import arithmetic as ar
    from battlezips_halo2_b200.plonk import prover as PR
    from battlezips_halo2_b200.circuits import shot_circuit, board_circuit, board_circuit_scaled
    if which in ("shot", "board"):
        cs, _, asg = (shot_circuit if which == "shot" else board_circuit)(0)
        batch = 64
    else:
        cs, _, asg = board_circuit_scaled(int(which[len("board"):]))
        batch = 1
    k = asg.k
    fx = os.path.join(ROOT, "tests", "golden", f"params_vesta_k{k}.npz")
    urs = dict(np.load(fx)) if os.path.exists(fx) else ar.params_new(ctx, k, curve=0)
    params = PR.Params(ctx, k, urs["g"], urs["g_lagrange"], urs["w"], urs["u"])
    pk = PR.ProvingKey(ctx, params, cs.to_ir(), asg.fixed, asg.permutation_mapping(), 0x1234567890ABCDEF1234567890ABCDEF)
    adv = np.stack([PR.mont(col) for col in asg.advice])
    return pk, params, [asg.instance] * batch, np.ascontiguousarray(np.stack([adv] * batch)), batch


def fill_kernel_ms(ctx, batch, blocks, reps):
    """Device time of one bz_chacha20_blocks launch of batch x blocks blocks (CUDA events, mean over reps)."""
    import torch
    from battlezips_halo2_b200 import arithmetic as ar
    buf = torch.empty(batch * blocks * 64, dtype=torch.uint8, device=f"cuda:{ctx.device}")
    seeds = np.frombuffer(os.urandom(32 * batch), dtype=np.uint8).reshape(batch, 32)
    ar.chacha20_blocks(ctx, seeds, blocks, out=buf.data_ptr())
    ctx.profile_enable(True)
    for _ in range(reps):
        ar.chacha20_blocks(ctx, seeds, blocks, out=buf.data_ptr())
    ms, count = ctx.profile_read()["other"]
    ctx.profile_enable(False)
    return ms / count


def run(ctx, which, reps, warmup):
    from battlezips_halo2_b200.plonk import prover as PR
    pk, params, inst, advice, B = build(ctx, which)
    R = pk.num_random
    new_seeds = lambda: np.frombuffer(os.urandom(32 * B), dtype=np.uint8).reshape(B, 32)
    s = new_seeds()
    assert PR.create_proofs_seeded(pk, inst, advice, s) == PR.create_proofs(pk, inst, advice, host_keystream(s, R)), which

    def host_path():
        t0 = time.perf_counter()
        wide = host_keystream(new_seeds(), R)
        t1 = time.perf_counter()
        PR.create_proofs(pk, inst, advice, wide)
        return time.perf_counter() - t0, t1 - t0

    def seeded_path():
        t0 = time.perf_counter()
        PR.create_proofs_seeded(pk, inst, advice, new_seeds())
        return time.perf_counter() - t0

    for _ in range(warmup):
        host_path(); seeded_path()
    th, tg, ts = [], [], []
    for _ in range(reps):
        a, g = host_path(); th.append(a); tg.append(g)
        ts.append(seeded_path())
    base = advice.nbytes // B + 4 * 8 * sum(len(c) for c in inst[0])          # advice + instance values per proof
    res = {
        "workload": which, "k": params.k, "batch": B, "num_random": R, "reps": reps,
        "host_path_ms_per_proof": round(1e3 * statistics.median(th) / B, 4),
        "host_keystream_ms_per_proof": round(1e3 * statistics.median(tg) / B, 4),
        "seeded_path_ms_per_proof": round(1e3 * statistics.median(ts) / B, 4),
        "host_path_h2d_bytes_per_proof": base + 64 * R, "seeded_path_h2d_bytes_per_proof": base + 32,
        "rng_h2d_bytes_per_proof": {"host": 64 * R, "seeded": 32},
        "fill_kernel_ms": round(fill_kernel_ms(ctx, B, R, reps), 5),
    }
    res["speedup"] = round(res["host_path_ms_per_proof"] / res["seeded_path_ms_per_proof"], 3)
    pk.close(); params.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="shot,board,board16,board20")
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    a = ap.parse_args()
    import battlezips_halo2_b200 as bz
    ctx = bz.Context(0)
    lines = [{"card": card()}]
    print(json.dumps(lines[0]), flush=True)
    for w in a.workloads.split(","):
        lines.append(run(ctx, w, a.reps, a.warmup))
        print(json.dumps(lines[-1]), flush=True)
    lines.append({"card_after": card()})
    print(json.dumps(lines[-1]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(l) for l in lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
