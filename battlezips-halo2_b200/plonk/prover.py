"""Host glue for the prover C ABI (include/bzhalo2.h): what the Rust shim does with `Params`, `ProvingKey` and
`create_proof` (reference call sites /root/reference/benches/shot.rs:58-71), expressed over ctypes.

Params / ProvingKey hold opaque device handles; create_proof returns exactly the bytes `transcript.finalize()`
yields in halo2_proofs 0.2.0."""
import ctypes
import numpy as np
from ..binding import _np_ptr, BzError

FP = 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001
_FP_ROOT = 0x2bce74deac30ebda362120830561f81aea322bf2b7bb7584bdad6fabd87ea32f
_FP_DELTA = 0x0a757d0f0006ab6cbd455b7112a5049df5e4f3f13eee56366a6ccd20dd7b9ba2


def mont(values, p=FP):
    """canonical ints -> (n,4) uint64 Montgomery limbs (pasta in-memory form)."""
    buf = b"".join(((int(v) << 256) % p).to_bytes(32, "little") for v in values)
    return np.frombuffer(buf, dtype=np.uint64).reshape(-1, 4).copy()


class bz_token(ctypes.Structure):
    _fields_ = [("op", ctypes.c_uint32), ("a", ctypes.c_uint32), ("b", ctypes.c_int32)]


class bz_circuit(ctypes.Structure):
    _fields_ = [
        ("k", ctypes.c_uint32), ("num_advice", ctypes.c_uint32), ("num_fixed", ctypes.c_uint32),
        ("num_instance", ctypes.c_uint32), ("degree", ctypes.c_uint32), ("blinding_factors", ctypes.c_uint32),
        ("n_advice_queries", ctypes.c_uint32), ("advice_queries", ctypes.c_void_p),
        ("n_fixed_queries", ctypes.c_uint32), ("fixed_queries", ctypes.c_void_p),
        ("n_instance_queries", ctypes.c_uint32), ("instance_queries", ctypes.c_void_p),
        ("n_perm_columns", ctypes.c_uint32), ("perm_columns", ctypes.c_void_p),
        ("n_constants", ctypes.c_uint32), ("constants", ctypes.c_void_p),
        ("n_tokens", ctypes.c_uint32), ("tokens", ctypes.c_void_p),
        ("n_gate_polys", ctypes.c_uint32), ("gate_poly_offsets", ctypes.c_void_p),
        ("n_lookups", ctypes.c_uint32), ("lookup_input_counts", ctypes.c_void_p), ("lookup_table_counts", ctypes.c_void_p),
        ("lookup_expr_offsets", ctypes.c_void_p),
        ("vk_transcript_repr", ctypes.c_uint8 * 32),
    ]


_KIND = {"advice": 0, "fixed": 1, "instance": 2}


def _bind(lib):
    vp, u32, i32 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int
    if getattr(lib, "_prover_bound", False):
        return
    lib.bz_params_create.restype = i32
    lib.bz_params_create.argtypes = [vp, u32, i32, vp, vp, vp, vp, i32, ctypes.POINTER(vp)]
    lib.bz_params_destroy.restype = None
    lib.bz_params_destroy.argtypes = [vp]
    lib.bz_params_commit.restype = i32
    lib.bz_params_commit.argtypes = [vp, vp, i32, vp, vp, vp]
    lib.bz_params_commit_batch_dev.restype = i32
    lib.bz_params_commit_batch_dev.argtypes = [vp, vp, i32, vp, vp, u32, vp]
    lib.bz_pk_create.restype = i32
    lib.bz_pk_create.argtypes = [vp, vp, ctypes.POINTER(bz_circuit), vp, vp, ctypes.POINTER(vp)]
    lib.bz_pk_create_from_assembly.restype = i32
    lib.bz_pk_create_from_assembly.argtypes = [vp, vp, ctypes.POINTER(bz_circuit), vp, vp, ctypes.POINTER(vp)]
    lib.bz_pk_vk_commitments.restype = i32
    lib.bz_pk_vk_commitments.argtypes = [vp, vp, vp, vp]
    lib.bz_verify_proofs.restype = i32
    lib.bz_verify_proofs.argtypes = [vp, vp, u32, vp, vp, u32, vp, u32, vp]
    lib.bz_vk_create.restype = i32
    lib.bz_vk_create.argtypes = [vp, vp, ctypes.POINTER(bz_circuit), vp, vp, ctypes.POINTER(vp)]
    lib.bz_vk_destroy.restype = None
    lib.bz_vk_destroy.argtypes = [vp]
    lib.bz_vk_proof_size.restype = u32
    lib.bz_vk_proof_size.argtypes = [vp]
    lib.bz_verify_proofs_vk.restype = i32
    lib.bz_verify_proofs_vk.argtypes = [vp, vp, u32, vp, vp, u32, vp, u32, vp]
    lib.bz_pk_destroy.restype = None
    lib.bz_pk_destroy.argtypes = [vp]
    lib.bz_pk_num_random.restype = u32
    lib.bz_pk_num_random.argtypes = [vp]
    lib.bz_pk_proof_size.restype = u32
    lib.bz_pk_proof_size.argtypes = [vp]
    lib.bz_pk_quotient_muls.restype = u32
    lib.bz_pk_quotient_muls.argtypes = [vp, u32, vp]
    lib.bz_create_proofs.restype = i32
    lib.bz_create_proofs.argtypes = [vp, vp, u32, vp, vp, u32, vp, vp, vp]
    lib._prover_bound = True


class Params:
    """`Params<vesta::Affine>` image on the device.  g, g_lagrange: (n,8) uint64 Montgomery affine; w, u: (8,)."""

    def __init__(self, ctx, k, g, g_lagrange, w, u, curve=0, window_bits=0):
        _bind(ctx.lib)
        self.ctx, self.k, self.n = ctx, k, 1 << k
        g = np.ascontiguousarray(g, dtype=np.uint64); gl = np.ascontiguousarray(g_lagrange, dtype=np.uint64)
        w = np.ascontiguousarray(w, dtype=np.uint64); u = np.ascontiguousarray(u, dtype=np.uint64)
        assert g.shape == (self.n, 8) and gl.shape == (self.n, 8)
        h = ctypes.c_void_p()
        ctx._check(ctx.lib.bz_params_create(ctx.h, k, curve, _np_ptr(g), _np_ptr(gl), _np_ptr(w), _np_ptr(u), window_bits, ctypes.byref(h)))
        self.h = h

    def commit(self, poly, blind, lagrange=False):
        """Params::commit / commit_lagrange followed by to_affine(): returns (8,) uint64 affine."""
        poly = np.ascontiguousarray(poly, dtype=np.uint64).reshape(self.n, 4)
        blind = np.ascontiguousarray(blind, dtype=np.uint64).reshape(4)
        out = np.zeros(8, dtype=np.uint64)
        self.ctx._check(self.ctx.lib.bz_params_commit(self.ctx.h, self.h, 1 if lagrange else 0, _np_ptr(poly), _np_ptr(blind), _np_ptr(out)))
        return out

    def commit_lagrange(self, poly, blind):
        return self.commit(poly, blind, lagrange=True)

    def commit_batch_dev(self, d_polys, d_blinds, count, d_out, lagrange=False):
        """`count` commitments, everything device-resident (int / c_void_p device addresses); d_out: count x 64 B."""
        as_ptr = lambda p: p if isinstance(p, ctypes.c_void_p) else ctypes.c_void_p(int(p))
        self.ctx._check(self.ctx.lib.bz_params_commit_batch_dev(self.ctx.h, self.h, 1 if lagrange else 0, as_ptr(d_polys), as_ptr(d_blinds), count, as_ptr(d_out)))

    def ipa_open(self, p_prime, x3, z, rounds):
        """poly::commitment::create_proof's folding loop through bz_ipa_begin / round / fold / finish.  rounds = k callables
        or tuples (l_rand, r_rand, u_of(L, R)) -- u_of maps the round's affine (L, R) to (u, u_inv) (the transcript side).
        Returns ([(L, R)], c)."""
        lib, ctx = self.ctx.lib, self.ctx
        sc = lambda v: np.ascontiguousarray(v, dtype=np.uint64).reshape(4)
        p_prime = np.ascontiguousarray(p_prime, dtype=np.uint64).reshape(-1, 4)
        h = ctypes.c_void_p()
        ctx._check(lib.bz_ipa_begin(ctx.h, self.h, _np_ptr(p_prime), _np_ptr(sc(x3)), ctypes.byref(h)))
        out = []
        try:
            for l_rand, r_rand, u_of in rounds:
                L, R = np.zeros(8, dtype=np.uint64), np.zeros(8, dtype=np.uint64)
                ctx._check(lib.bz_ipa_round(ctx.h, h, _np_ptr(sc(z)), _np_ptr(sc(l_rand)), _np_ptr(sc(r_rand)), _np_ptr(L), _np_ptr(R)))
                u, u_inv = u_of(L, R)
                ctx._check(lib.bz_ipa_fold(ctx.h, h, _np_ptr(sc(u)), _np_ptr(sc(u_inv))))
                out.append((L, R))
            c = np.zeros(4, dtype=np.uint64)
            ctx._check(lib.bz_ipa_finish(ctx.h, h, _np_ptr(c)))
            h = None
        finally:
            if h:
                lib.bz_ipa_destroy(h)
        return out, c

    def close(self):
        if self.h:
            self.ctx.lib.bz_params_destroy(self.h)
            self.h = None


def flatten_circuit(ir, k, vk_repr):
    """ConstraintSystem IR (plonk/circuit.py `to_ir`) -> bz_circuit + the numpy arrays that back its pointers."""
    p = ir["modulus"]
    consts, const_index = [], {}

    def cidx(v):
        v %= p
        if v not in const_index:
            const_index[v] = len(consts)
            consts.append(v)
        return const_index[v]

    tokens = []

    def emit(e):
        kind = e[0]
        if kind == "const":
            tokens.append((0, cidx(e[1]), 0))
        elif kind in ("advice", "fixed", "instance"):
            tokens.append(({"advice": 1, "fixed": 2, "instance": 3}[kind], e[1], e[2]))
        elif kind == "neg":
            emit(e[1]); tokens.append((4, 0, 0))
        elif kind == "sum":
            emit(e[1]); emit(e[2]); tokens.append((5, 0, 0))
        elif kind == "product":
            emit(e[1]); emit(e[2]); tokens.append((6, 0, 0))
        elif kind == "scaled":
            emit(e[1]); tokens.append((7, cidx(e[2]), 0))
        else:
            raise ValueError(kind)

    gate_off = [0]
    for gate in ir["gates"]:
        for poly in gate["polys"]:
            emit(poly)
            gate_off.append(len(tokens))
    lk_off, lk_in, lk_tab = [len(tokens)], [], []
    for lk in ir["lookups"]:
        lk_in.append(len(lk["input"])); lk_tab.append(len(lk["table"]))
        for e in lk["input"] + lk["table"]:
            emit(e)
            lk_off.append(len(tokens))
    keep = {}
    keep["aq"] = np.array(ir["advice_queries"], dtype=np.int32).reshape(-1, 2)
    keep["fq"] = np.array(ir["fixed_queries"], dtype=np.int32).reshape(-1, 2)
    keep["iq"] = np.array(ir["instance_queries"], dtype=np.int32).reshape(-1, 2)
    keep["perm"] = np.array([[_KIND[c[0]], c[1]] for c in ir["permutation"]], dtype=np.uint32).reshape(-1, 2)
    keep["consts"] = mont(consts, p) if consts else np.zeros((1, 4), np.uint64)
    tk = (bz_token * max(1, len(tokens)))()
    for i, (op, a, b) in enumerate(tokens):
        tk[i].op, tk[i].a, tk[i].b = op, a, b
    keep["tokens"] = tk
    keep["gate_off"] = np.array(gate_off, dtype=np.uint32)
    keep["lk_in"] = np.array(lk_in or [0], dtype=np.uint32)
    keep["lk_tab"] = np.array(lk_tab or [0], dtype=np.uint32)
    keep["lk_off"] = np.array(lk_off, dtype=np.uint32)
    c = bz_circuit()
    c.k, c.num_advice, c.num_fixed, c.num_instance = k, ir["num_advice"], ir["num_fixed"], ir["num_instance"]
    c.degree, c.blinding_factors = ir["degree"], ir["blinding_factors"]
    c.n_advice_queries, c.advice_queries = len(keep["aq"]), keep["aq"].ctypes.data
    c.n_fixed_queries, c.fixed_queries = len(keep["fq"]), keep["fq"].ctypes.data
    c.n_instance_queries, c.instance_queries = len(keep["iq"]), keep["iq"].ctypes.data
    c.n_perm_columns, c.perm_columns = len(keep["perm"]), keep["perm"].ctypes.data
    c.n_constants, c.constants = len(consts), keep["consts"].ctypes.data
    c.n_tokens, c.tokens = len(tokens), ctypes.addressof(tk)
    c.n_gate_polys, c.gate_poly_offsets = len(gate_off) - 1, keep["gate_off"].ctypes.data
    c.n_lookups = len(ir["lookups"])
    c.lookup_input_counts, c.lookup_table_counts = keep["lk_in"].ctypes.data, keep["lk_tab"].ctypes.data
    c.lookup_expr_offsets = keep["lk_off"].ctypes.data
    c.vk_transcript_repr[:] = list((vk_repr % p).to_bytes(32, "little"))
    return c, keep


def sigma_values(ir, k, mapping, p=FP):
    """pk.permutation.permutations: sigma_col[row] = delta^col' * omega^row' (U: permutation/keygen.rs build_pk)."""
    n = 1 << k
    omega = pow(_FP_ROOT, 1 << (32 - k), p)
    om = [1] * n
    for i in range(1, n):
        om[i] = om[i - 1] * omega % p
    m = len(ir["permutation"])
    dl = [pow(_FP_DELTA, i, p) for i in range(m)]
    return [[dl[c] * om[r] % p for (c, r) in mapping[i]] for i in range(m)]


class ProvingKey:
    """keygen_pk's device image for one circuit."""

    def __init__(self, ctx, params, ir, fixed_values, mapping, vk_repr, host_sigma=False):
        _bind(ctx.lib)
        self.ctx, self.params, self.ir, self.vk_repr = ctx, params, ir, vk_repr
        self.k, self.n = params.k, params.n
        circ, keep = flatten_circuit(ir, params.k, vk_repr)
        fixed = mont([v for col in fixed_values for v in col]) if fixed_values else np.zeros((1, 4), np.uint64)
        h = ctypes.c_void_p()
        if host_sigma:          # pk.permutation.permutations computed by the caller (what a patched keygen_pk may already hold)
            sig = sigma_values(ir, params.k, mapping)
            sigma = mont([v for col in sig for v in col]) if sig else np.zeros((1, 4), np.uint64)
            ctx._check(ctx.lib.bz_pk_create(ctx.h, params.h, ctypes.byref(circ), _np_ptr(fixed), _np_ptr(sigma), ctypes.byref(h)))
        else:                   # Assembly::build_pk on the device from the copy-constraint cycles
            mp = np.ascontiguousarray(np.array(mapping, dtype=np.uint32).reshape(-1, 2)) if len(mapping) else np.zeros((1, 2), np.uint32)
            ctx._check(ctx.lib.bz_pk_create_from_assembly(ctx.h, params.h, ctypes.byref(circ), _np_ptr(fixed), _np_ptr(mp), ctypes.byref(h)))
        self.h = h
        self.degree = ir["degree"]
        self.num_random = ctx.lib.bz_pk_num_random(h)
        self.proof_size = ctx.lib.bz_pk_proof_size(h)
        # (multiplications per point, points) of every h(X) evaluation tier: the quotient kernel's algorithmic work
        self.quotient_muls = []
        for t in range(3):
            pts = ctypes.c_uint32(0)
            self.quotient_muls.append((ctx.lib.bz_pk_quotient_muls(h, t, ctypes.byref(pts)), pts.value))

    def vk_commitments(self):
        """keygen_vk: (fixed_commitments (F, 8), permutation commitments (M, 8)) as Montgomery affine points."""
        F, M = self.ir["num_fixed"], len(self.ir["permutation"])
        fc, pc = np.zeros((max(F, 1), 8), dtype=np.uint64), np.zeros((max(M, 1), 8), dtype=np.uint64)
        self.ctx._check(self.ctx.lib.bz_pk_vk_commitments(self.ctx.h, self.h, _np_ptr(fc), _np_ptr(pc)))
        return fc[:F], pc[:M]

    def verifying_key(self):
        """keygen_vk's result as an independent VerifyingKey: it keeps no reference to this proving key, which may be closed."""
        fc, pc = self.vk_commitments()
        return VerifyingKey(self.ctx, self.params, self.ir, fc, pc, self.vk_repr)

    def quotient(self, polys, theta, beta, gamma, y):
        """vanishing::Argument::construct up to h(X)'s coefficients (bz_pk_quotient): polys = (slots, n, 4) coefficient
        forms in the order advice, instance, per lookup (A', S', Z), permutation z; challenges as (4,) Montgomery limbs.
        Returns ((degree - 1) * n, 4)."""
        lib = self.ctx.lib
        slots = lib.bz_pk_num_poly_slots(self.h)
        polys = np.ascontiguousarray(polys, dtype=np.uint64).reshape(slots, -1, 4)
        n = polys.shape[1]
        out = np.zeros(((self.degree - 1) * n, 4), dtype=np.uint64)
        sc = [np.ascontiguousarray(v, dtype=np.uint64).reshape(4) for v in (theta, beta, gamma, y)]
        self.ctx._check(lib.bz_pk_quotient(self.ctx.h, self.h, _np_ptr(polys), *[_np_ptr(v) for v in sc], _np_ptr(out)))
        return out

    def close(self):
        if self.h:
            self.ctx.lib.bz_pk_destroy(self.h)
            self.h = None


class VerifyingKey:
    """halo2's `VerifyingKey` on the device side: the constraint system, keygen_vk's commitments (fixed (F, 8) and permutation
    (M, 8) Montgomery affine points) and the vk.hash_into scalar.  Holds no fixed values and no sigma columns, and creating it
    allocates no device memory; `params` must stay open while it is used."""

    def __init__(self, ctx, params, ir, fixed_commitments, perm_commitments, vk_repr):
        _bind(ctx.lib)
        self.ctx, self.params, self.ir, self.vk_repr = ctx, params, ir, vk_repr
        self.k, self.n = params.k, params.n
        circ, keep = flatten_circuit(ir, params.k, vk_repr)
        F, M = ir["num_fixed"], len(ir["permutation"])
        fc = np.ascontiguousarray(fixed_commitments, dtype=np.uint64).reshape(-1, 8)
        pc = np.ascontiguousarray(perm_commitments, dtype=np.uint64).reshape(-1, 8)
        if fc.shape[0] != F or pc.shape[0] != M:
            raise ValueError(f"VerifyingKey: expected {F} fixed and {M} permutation commitments, got {fc.shape[0]} and {pc.shape[0]}")
        fc = fc if F else np.zeros((1, 8), np.uint64)
        pc = pc if M else np.zeros((1, 8), np.uint64)
        h = ctypes.c_void_p()
        ctx._check(ctx.lib.bz_vk_create(ctx.h, params.h, ctypes.byref(circ), _np_ptr(fc), _np_ptr(pc), ctypes.byref(h)))
        self.h = h
        self.proof_size = ctx.lib.bz_vk_proof_size(h)

    def close(self):
        if self.h:
            self.ctx.lib.bz_vk_destroy(self.h)
            self.h = None


def create_proofs(pk, instances, advice, rand_wide):
    """create_proof for a batch.  instances: (B, num_instance, stride, 4) uint64 + implied lens, or list of lists of
    int lists; advice: (B, num_advice, n, 4) uint64 Montgomery; rand_wide: (B, num_random, 8) uint64.
    Returns list of B proof byte strings."""
    ctx = pk.ctx
    advice = np.ascontiguousarray(advice, dtype=np.uint64)
    B = advice.shape[0]
    assert advice.shape == (B, pk.ir["num_advice"], pk.n, 4)
    rand_wide = np.ascontiguousarray(rand_wide, dtype=np.uint64)
    assert rand_wide.shape == (B, pk.num_random, 8), (rand_wide.shape, pk.num_random)
    ni = pk.ir["num_instance"]
    lens = np.array([len(instances[0][i]) for i in range(ni)] or [0], dtype=np.uint32)
    stride = max(1, int(lens.max()))
    inst = np.zeros((B, max(1, ni), stride, 4), dtype=np.uint64)
    for b in range(B):
        assert len(instances[b]) == ni, "Error::InvalidInstances"
        for i in range(ni):
            assert len(instances[b][i]) == lens[i]
            if lens[i]:
                inst[b, i, :lens[i]] = mont(instances[b][i])
    out = np.zeros((B, pk.proof_size), dtype=np.uint8)
    ctx._check(ctx.lib.bz_create_proofs(ctx.h, pk.h, B, _np_ptr(inst), _np_ptr(lens), stride, _np_ptr(advice), _np_ptr(rand_wide), _np_ptr(out)))
    return [bytes(out[b]) for b in range(B)]


def _pack_instances(pk, instances, B):
    ni = pk.ir["num_instance"]
    lens = np.array([len(instances[0][i]) for i in range(ni)] or [0], dtype=np.uint32)
    stride = max(1, int(lens.max()))
    inst = np.zeros((B, max(1, ni), stride, 4), dtype=np.uint64)
    for b in range(B):
        assert len(instances[b]) == ni, "Error::InvalidInstances"
        for i in range(ni):
            assert len(instances[b][i]) == lens[i]
            if lens[i]:
                inst[b, i, :lens[i]] = mont(instances[b][i])
    return inst, lens, stride


def verify_proofs(pk, instances, proofs):
    """plonk::verify_proof for a batch: pk = a VerifyingKey or a ProvingKey, instances[b] = list (num_instance) of int lists,
    proofs[b] = bytes (equal lengths).  Returns a list of bools (Ok / Err of the reference's SingleVerifier)."""
    ctx = pk.ctx
    B = len(proofs)
    plen = len(proofs[0])
    if any(len(p) != plen for p in proofs):
        raise ValueError("verify_proofs: proofs of one batch must have equal lengths")
    inst, lens, stride = _pack_instances(pk, instances, B)
    buf = np.frombuffer(b"".join(proofs) or b"\0", dtype=np.uint8).copy()
    res = np.zeros(B, dtype=np.uint8)
    verify = ctx.lib.bz_verify_proofs_vk if isinstance(pk, VerifyingKey) else ctx.lib.bz_verify_proofs
    ctx._check(verify(ctx.h, pk.h, B, _np_ptr(inst), _np_ptr(lens), stride, _np_ptr(buf), plen, _np_ptr(res)))
    return [bool(x) for x in res]
