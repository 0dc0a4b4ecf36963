"""ORACLE (test infrastructure; never shipped, never the thing measured as the product).

CPU restatement of the halo2_proofs 0.2.0 IPA prover and verifier over the Pasta curves -- the code path
behind the reference's `create_proof` / `verify_proof` calls
(/root/reference/benches/shot.rs:58-71, /root/reference/benches/board.rs:51-86,
/root/reference/src/circuits/shot.rs:915-940, /root/reference/src/circuits/board.rs:907-932).

The crate itself (pinned at /root/reference/Cargo.lock:382-393, checksum cff771b9...949a) is NOT vendored and
there is no Rust toolchain here, so this follows the published algorithm of these upstream files (SURVEY App. A,
D, H restate them step by step):
  src/plonk/prover.rs, src/plonk/verifier.rs, src/plonk/keygen.rs,
  src/plonk/{permutation,lookup,vanishing}/{prover,verifier}.rs, src/plonk/permutation/keygen.rs,
  src/poly/commitment.rs, src/poly/commitment/{prover,verifier}.rs, src/poly/multiopen{,/prover,/verifier}.rs,
  src/poly/domain.rs, src/arithmetic.rs, src/transcript.rs.

PARITY UNPINNED for proof bytes: the reference draws all randomness from OsRng and pins no proof, commitment,
MSM or NTT vector (SURVEY §0 fact 4, §8c).  What pins this file: (1) the Pallas hash-to-curve / scalar-mul KATs
that the underlying arithmetic passes (tests/test_oracle_kat.py), (2) prover/verifier round trips incl. tamper
rejection (tests/test_oracle_prover.py), i.e. the reference's own `production` test shape
(/root/reference/src/circuits/shot.rs:880-941).

Heavy loops run in the C restatement (oracle/c): best_multiexp, best_fft, eval_polynomial, kate_division,
batch_invert ... with the reference's rayon-style chunking; protocol order lives here.
One circuit instance per proof (all the reference ever passes: `&[circuit]`)."""
import hashlib, os, ctypes
from collections import OrderedDict
import numpy as np
from . import pasta, c_oracle as co
from .vec import Vec
from .domain import EvaluationDomain

_BUILD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_build")


# ------------------------------------------------------------------------------------------------------
# RngCore stand-in.  `Field::random(rng)` = from_u512 of 8 x next_u64 (little-endian limbs)  [U: pasta fields]
# ------------------------------------------------------------------------------------------------------
class Draws:
    """A pre-drawn stream of 64-byte RNG outputs, consumed strictly in protocol order (SURVEY App. A)."""

    def __init__(self, wide):
        self.wide = np.ascontiguousarray(wide, dtype=np.uint64).reshape(-1, 8)
        self.pos = 0

    def take(self, f, n):
        assert self.pos + n <= len(self.wide), "RNG stream exhausted"
        out = co.from_u512(f, self.wide[self.pos:self.pos + n])
        self.pos += n
        return out


def splitmix64_wide(seed, n):
    """n x 8 uint64 words from SplitMix64(seed) (test RNG; SURVEY §8d config 2)."""
    idx = np.arange(1, 8 * n + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + idx * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return z.reshape(n, 8)


# ------------------------------------------------------------------------------------------------------
# Transcript  [U: src/transcript.rs: Blake2bWrite / Blake2bRead / Challenge255]
# ------------------------------------------------------------------------------------------------------
class Blake2bTranscript:
    def __init__(self, curve_id=0, proof=None):
        self.curve, self.sf, self.bf = co.CURVES[curve_id]
        self.state = hashlib.blake2b(digest_size=64, person=b"Halo2-Transcript")
        self.out = bytearray()
        self.proof = proof
        self.rpos = 0

    def squeeze_challenge(self):
        self.state.update(b"\x00")
        return int.from_bytes(self.state.copy().digest(), "little") % self.curve.scalar.p

    def common_point(self, pt):
        if pt is None:
            raise IOError("cannot write points at infinity to the transcript")
        self.state.update(b"\x01" + pt[0].to_bytes(32, "little") + pt[1].to_bytes(32, "little"))

    def common_scalar(self, s):
        self.state.update(b"\x02" + (s % self.curve.scalar.p).to_bytes(32, "little"))

    def write_point(self, pt):
        self.common_point(pt)
        self.out += self.curve.to_bytes(pt)

    def write_scalar(self, s):
        self.common_scalar(s)
        self.out += (s % self.curve.scalar.p).to_bytes(32, "little")

    def read_point(self):
        b = bytes(self.proof[self.rpos:self.rpos + 32]); self.rpos += 32
        if len(b) != 32:
            raise IOError("proof too short")
        pt = self.curve.from_bytes(b)
        self.common_point(pt)
        return pt

    def read_scalar(self):
        b = bytes(self.proof[self.rpos:self.rpos + 32]); self.rpos += 32
        if len(b) != 32:
            raise IOError("proof too short")
        v = int.from_bytes(b, "little")
        if v >= self.curve.scalar.p:
            raise IOError("invalid field element encoding in proof")
        self.common_scalar(v)
        return v

    def finalize(self):
        return bytes(self.out)


# ------------------------------------------------------------------------------------------------------
# Params  [U: src/poly/commitment.rs]
# ------------------------------------------------------------------------------------------------------
class Params:
    def __init__(self, k, curve_id, g, g_lagrange, w, u):
        self.k, self.n, self.curve_id = k, 1 << k, curve_id
        self.g, self.g_lagrange, self.w, self.u = g, g_lagrange, w, u      # (n,8), (n,8), (8,), (8,) Montgomery affine
        self.sf = co.CURVES[curve_id][1]
        self._gw = np.concatenate([g, w[None, :]])
        self._glw = np.concatenate([g_lagrange, w[None, :]])

    @staticmethod
    def new(k, curve_id=0, cache=True):
        """`Params::new(k)`: g[i] = hash_to_curve("Halo2-Parameters")(0 || i_le32); g_lagrange = EC-iFFT(g);
        w = hasher([1]); u = hasher([2])."""
        path = os.path.join(_BUILD, f"params_c{curve_id}_k{k}.npz")
        if cache and os.path.exists(path):
            d = np.load(path)
            return Params(k, curve_id, d["g"], d["g_lagrange"], d["w"], d["u"])
        C, sf, bf = co.CURVES[curve_id]
        n = 1 << k
        hasher = C.hash_to_curve("Halo2-Parameters")
        g_pts = [hasher(b"\x00" + i.to_bytes(4, "little")) for i in range(n)]
        g = co.points_to_mont(curve_id, g_pts)
        # g_lagrange: best_fft over group elements with alpha_inv, then scale by 2^-k
        SF = co.FIELDS[sf]
        alpha_inv = SF.root_of_unity_inv
        for _ in range(k, pasta.S):
            alpha_inv = alpha_inv * alpha_inv % SF.p
        one = np.frombuffer(co.FIELDS[bf].to_mont_bytes(1), dtype=np.uint64)
        jac = np.concatenate([g, np.repeat(one[None, :], n, axis=0)], axis=1).copy()
        co.lib().orc_best_fft_ec(curve_id, co._p(jac), co._p(co.to_mont(sf, [alpha_inv])), ctypes.c_uint(k))
        aff = co.to_affine(curve_id, jac)
        minv = co.to_mont(sf, [pow(SF.two_inv, k, SF.p)])
        gl = np.empty_like(aff)
        tmp = np.empty(8, dtype=np.uint64)
        for i in range(n):
            co.lib().orc_point_mul(curve_id, co._p(aff[i]), co._p(minv), co._p(tmp))
            gl[i] = tmp
        w = co.points_to_mont(curve_id, [hasher(b"\x01")])[0]
        u = co.points_to_mont(curve_id, [hasher(b"\x02")])[0]
        if cache:
            os.makedirs(_BUILD, exist_ok=True)
            np.savez(path, g=g, g_lagrange=gl, w=w, u=u)
        return Params(k, curve_id, g, gl, w, u)

    def _commit(self, bases_w, poly, blind):
        V = Vec(self.sf)
        scalars = np.concatenate([np.ascontiguousarray(poly), V.m(blind)[None, :]])
        return co.best_multiexp(self.curve_id, scalars, bases_w)          # Jacobian (12,)

    def commit(self, poly, blind):
        assert len(poly) == self.n
        return self._commit(self._gw, poly, blind)

    def commit_lagrange(self, poly, blind):
        assert len(poly) == self.n
        return self._commit(self._glw, poly, blind)


def batch_invert_assigned(V, numerators, denominators):
    """poly::batch_invert_assigned (U: halo2_proofs 0.2.0 src/poly.rs): the denominators of one column's Assigned<F> cells
    go through ff::BatchInvert (zeros are skipped and stay zero), then every numerator is multiplied by its inverse --
    `Polynomial<Assigned<F>>::invert`.  Zero / Trivial cells are (0, 1) / (x, 1).  (n,4) Montgomery arrays in and out."""
    return V.mul(numerators, V.batch_invert(denominators))


def _affine_pts(curve_id, jacs):
    """list of Jacobian (12,) -> list of affine int tuples (batch_normalize)."""
    if not len(jacs):
        return []
    return co.points_from_mont(curve_id, co.to_affine(curve_id, np.stack(jacs)))


# ------------------------------------------------------------------------------------------------------
# Expression evaluation over whole columns (the reference's poly::Evaluator works the same way, node by node)
# ------------------------------------------------------------------------------------------------------
def eval_expr(V, e, leaf, n):
    k = e[0]
    if k == "const":
        return V.const(e[1], n)
    if k in ("fixed", "advice", "instance"):
        return leaf(k, e[1], e[2])
    if k == "neg":
        return V.neg(eval_expr(V, e[1], leaf, n))
    if k == "sum":
        return V.add(eval_expr(V, e[1], leaf, n), eval_expr(V, e[2], leaf, n))
    if k == "product":
        return V.mul(eval_expr(V, e[1], leaf, n), eval_expr(V, e[2], leaf, n))
    if k == "scaled":
        return V.scale(eval_expr(V, e[1], leaf, n), e[2])
    raise ValueError(k)


def eval_expr_scalar(p, e, leaf):
    """Same tree over single field values (verifier side)."""
    k = e[0]
    if k == "const": return e[1] % p
    if k in ("fixed", "advice", "instance"): return leaf(k, e[1], e[2])
    if k == "neg": return (-eval_expr_scalar(p, e[1], leaf)) % p
    if k == "sum": return (eval_expr_scalar(p, e[1], leaf) + eval_expr_scalar(p, e[2], leaf)) % p
    if k == "product": return eval_expr_scalar(p, e[1], leaf) * eval_expr_scalar(p, e[2], leaf) % p
    if k == "scaled": return eval_expr_scalar(p, e[1], leaf) * e[2] % p
    raise ValueError(k)


# ------------------------------------------------------------------------------------------------------
# keygen  [U: src/plonk/keygen.rs, src/plonk/permutation/keygen.rs]   (one-off per circuit; not timed)
# ------------------------------------------------------------------------------------------------------
class ProvingKey:
    pass


def keygen(params, ir, fixed_values, mapping, vk_repr):
    """fixed_values: list (num_fixed) of n canonical ints; mapping[col][row] = (col', row') from Assembly::copy."""
    f = params.sf
    V = Vec(f)
    pk = ProvingKey()
    pk.ir, pk.params = ir, params
    k, n = params.k, params.n
    pk.domain = dom = EvaluationDomain(f, ir["degree"], k)
    bf = ir["blinding_factors"]
    pk.fixed_values = [V.arr(col) for col in fixed_values]
    pk.fixed_polys = [dom.lagrange_to_coeff(v) for v in pk.fixed_values]
    pk.fixed_cosets = [dom.coeff_to_extended(p) for p in pk.fixed_polys]
    # permutation: sigma_col[row] = delta^col' * omega^row'
    p = V.p
    omega_pows = V.ints(V.powers(1, dom.omega, n))
    m = len(ir["permutation"])
    delta_pows = [pow(V.F.delta, i, p) for i in range(m)]
    pk.perm_values = []
    for i in range(m):
        col = [delta_pows[ci] * omega_pows[rj] % p for (ci, rj) in mapping[i]]
        pk.perm_values.append(V.arr(col))
    pk.perm_polys = [dom.lagrange_to_coeff(v) for v in pk.perm_values]
    pk.perm_cosets = [dom.coeff_to_extended(q) for q in pk.perm_polys]
    l0 = [0] * n; l0[0] = 1
    l_blind = [0] * n
    for i in range(n - bf, n):
        l_blind[i] = 1
    l_last = [0] * n; l_last[n - bf - 1] = 1
    pk.l0, pk.l_blind, pk.l_last = [dom.coeff_to_extended(dom.lagrange_to_coeff(V.arr(x))) for x in (l0, l_blind, l_last)]
    # verifying-key commitments (Blind::default() = 1)
    pk.fixed_commitments = _affine_pts(params.curve_id, [params.commit_lagrange(v, 1) for v in pk.fixed_values])
    pk.perm_commitments = _affine_pts(params.curve_id, [params.commit_lagrange(v, 1) for v in pk.perm_values])
    pk.vk_repr = vk_repr % p       # opaque transcript seed (vk.hash_into; SURVEY App. A step 0)
    return pk


# ------------------------------------------------------------------------------------------------------
# multiopen bookkeeping  [U: src/poly/multiopen.rs::construct_intermediate_sets]
# ------------------------------------------------------------------------------------------------------
def construct_intermediate_sets(queries):
    """queries: list of (commitment_id, point_int, payload).  Returns (commitment_map, point_sets) where
    commitment_map = [ {id, set_index, point_indices, payloads(evals ordered by point-index-set)} ] in first-
    appearance order and point_sets[set_index] = [points] ordered by point index."""
    commitment_map = []           # list of dicts in first-appearance order
    by_id = {}
    point_index_map = OrderedDict()
    for cid, point, payload in queries:
        if point not in point_index_map:
            point_index_map[point] = len(point_index_map)
        pi = point_index_map[point]
        if cid in by_id:
            by_id[cid]["point_indices"].append(pi)
        else:
            d = {"id": cid, "point_indices": [pi], "first_payload": payload}
            by_id[cid] = d
            commitment_map.append(d)
    inverse = {v: k for k, v in point_index_map.items()}
    point_idx_sets = OrderedDict()      # frozenset(sorted tuple) -> set_idx, insertion ordered
    for d in commitment_map:
        s = tuple(sorted(set(d["point_indices"])))
        d["point_index_set"] = s
        if s not in point_idx_sets:
            point_idx_sets[s] = len(point_idx_sets)
        d["set_index"] = point_idx_sets[s]
        d["evals"] = [None] * len(s)
    for cid, point, payload in queries:
        d = by_id[cid]
        d["evals"][d["point_index_set"].index(point_index_map[point])] = payload
    point_sets = [None] * len(point_idx_sets)
    for s, idx in point_idx_sets.items():
        point_sets[idx] = [inverse[i] for i in s]
    return commitment_map, point_sets


# ------------------------------------------------------------------------------------------------------
# argument inner loops  [U: src/plonk/lookup/prover.rs, src/plonk/permutation/prover.rs]
# ------------------------------------------------------------------------------------------------------
def permute_expression_pair(V, usable, cin, ctab):
    """lookup::prover::permute_expression_pair over the first `usable` rows of the compressed input / table ((n,4)
    Montgomery arrays) -> (A', S'), `usable` rows each.  A' is the input sorted by canonical value; S' holds the table
    value next to the first row of every run of equal inputs, and the left-over table values fill the repeated rows,
    last row first, in BTreeMap (ascending) order.  An input value missing from the table's usable rows raises
    ValueError("Error::ConstraintSystemFailure")."""
    a_keys = V.sort_keys(cin[:usable])
    s_keys = V.sort_keys(ctab[:usable])
    a_list = [bytes(r) for r in a_keys]
    order = sorted(range(usable), key=lambda i: a_list[i])
    permuted_input = np.ascontiguousarray(cin[:usable][order]).reshape(-1, 4)
    a_sorted = [a_list[i] for i in order]
    leftover = {}
    s_val = {}
    for i in range(usable):
        kb = bytes(s_keys[i])
        leftover[kb] = leftover.get(kb, 0) + 1
        s_val[kb] = ctab[i]
    permuted_table = V.zeros(usable)
    repeated = []
    for row in range(usable):
        if row == 0 or a_sorted[row] != a_sorted[row - 1]:
            permuted_table[row] = permuted_input[row]
            if a_sorted[row] not in leftover:
                raise ValueError("Error::ConstraintSystemFailure")     # input value not in table
            assert leftover[a_sorted[row]] > 0
            leftover[a_sorted[row]] -= 1
        else:
            repeated.append(row)
    for kb in sorted(leftover.keys()):            # BTreeMap iteration = ascending numeric order
        for _ in range(leftover[kb]):
            permuted_table[repeated.pop()] = s_val[kb]
    assert not repeated
    return permuted_input, permuted_table


def permutation_product(V, omega, values, sigmas, beta, gamma, delta_omega0, z0):
    """permutation::Argument::commit for one column set, before blinding: z[0] = z0,
    z[i+1] = z[i] * prod_j (v_j[i] + beta delta_omega0 delta^j omega^i + gamma) * inv0(prod_j (v_j[i] + beta sigma_j[i] + gamma)),
    where inv0 (ff::BatchInvert) leaves zero at zero.  values / sigmas: lists of (n,4) Montgomery arrays; scalars are ints."""
    n, p = len(values[0]), V.p
    modified = V.const(1, n)
    for v, s in zip(values, sigmas):
        modified = V.mul(modified, V.add(V.add_const(V.scale(s, beta), gamma), v))
    modified = V.batch_invert(modified)
    omega_pows = V.powers(1, omega, n)
    deltaomega = delta_omega0
    for v in values:
        modified = V.mul(modified, V.add(V.add_const(V.scale(omega_pows, deltaomega * beta % p), gamma), v))
        deltaomega = deltaomega * V.F.delta % p
    return V.running_product(z0, modified)


def lookup_product(V, cin, ctab, pin, ptab, beta, gamma):
    """lookup::Permuted::commit_product before blinding: z[0] = 1,
    z[i+1] = z[i] * (cin[i] + beta)(ctab[i] + gamma) * inv0((pin[i] + beta)(ptab[i] + gamma))."""
    prod = V.batch_invert(V.mul(V.add_const(pin, beta), V.add_const(ptab, gamma)))
    prod = V.mul(prod, V.add_const(cin, beta))
    prod = V.mul(prod, V.add_const(ctab, gamma))
    return V.running_product(1, prod)


# ------------------------------------------------------------------------------------------------------
# create_proof  [U: src/plonk/prover.rs and the argument provers; SURVEY App. A steps 0-21]
# ------------------------------------------------------------------------------------------------------
def create_proof(params, pk, instances, advice, draws, transcript, trace=None):
    """instances: list (num_instance) of lists of ints; advice: list (num_advice) of (n,4) Montgomery arrays
    whose last bf+1 rows are ignored (overwritten with blinding); draws: Draws; returns nothing -- bytes are in
    transcript.finalize().  `trace`, if a dict, receives named intermediates for the parity suite."""
    ir, dom = pk.ir, pk.domain
    f, cid = params.sf, params.curve_id
    V = Vec(f)
    p = V.p
    n, k = params.n, params.k
    bf = ir["blinding_factors"]
    usable = n - (bf + 1)
    ext_n = 1 << dom.extended_k
    rot_scale = 1 << (dom.extended_k - k)
    T = transcript
    tr = trace if trace is not None else {}
    import time as _time
    _clock = {"t": _time.perf_counter(), "name": "setup"}
    tr["phase_s"] = {}

    def _phase(name):          # wall-clock seconds per protocol phase (bench.py --impl reference reports them)
        now = _time.perf_counter()
        tr["phase_s"][_clock["name"]] = tr["phase_s"].get(_clock["name"], 0.0) + now - _clock["t"]
        _clock["t"], _clock["name"] = now, name

    def rnd(m):
        return draws.take(f, m)

    def rnd1():
        return V.int1(rnd(1)[0])

    assert len(instances) == ir["num_instance"], "Error::InvalidInstances"
    # step 0: vk.hash_into
    T.common_scalar(pk.vk_repr)

    _phase("instance + advice commitments")
    # step 1: instance columns
    instance_values, instance_polys, instance_cosets = [], [], []
    for vals in instances:
        if len(vals) > usable:
            raise ValueError("Error::InstanceTooLarge")
        col = V.zeros(n)
        if len(vals):
            col[:len(vals)] = V.arr(vals)
        instance_values.append(col)
    inst_comm = _affine_pts(cid, [params.commit_lagrange(v, 1) for v in instance_values])
    for c in inst_comm:
        T.common_point(c)
    instance_polys = [dom.lagrange_to_coeff(v) for v in instance_values]
    instance_cosets = [dom.coeff_to_extended(q) for q in instance_polys]

    # step 2: advice columns: blinding rows (column order), then one blind per column
    advice_values = [np.ascontiguousarray(a).copy() for a in advice]
    assert len(advice_values) == ir["num_advice"]
    for a in advice_values:
        assert len(a) == n
        a[usable:] = rnd(n - usable)
    advice_blinds = [rnd1() for _ in advice_values]
    adv_comm = _affine_pts(cid, [params.commit_lagrange(a, b) for a, b in zip(advice_values, advice_blinds)])
    for c in adv_comm:
        T.write_point(c)
    advice_polys = [dom.lagrange_to_coeff(a) for a in advice_values]
    advice_cosets = [dom.coeff_to_extended(q) for q in advice_polys]
    tr["advice_commitments"] = adv_comm

    # step 3
    theta = T.squeeze_challenge()
    tr["challenges"] = {"theta": theta}

    def lagrange_leaf(kind, col, rot):
        src = {"advice": advice_values, "fixed": pk.fixed_values, "instance": instance_values}[kind][col]
        return np.roll(src, -rot, axis=0) if rot else src

    def coset_leaf(kind, col, rot):
        src = {"advice": advice_cosets, "fixed": pk.fixed_cosets, "instance": instance_cosets}[kind][col]
        return np.roll(src, -rot * rot_scale, axis=0) if rot else src

    _phase("lookup permute + commitments")
    # steps 4-5: lookups: compress, permute, commit
    lookups = []
    for lk in ir["lookups"]:
        def compress(exprs, leaf, m):
            acc = V.zeros(m)
            for e in exprs:
                acc = V.add(V.scale(acc, theta), eval_expr(V, e, leaf, m))
            return acc
        L = {"compressed_input": compress(lk["input"], lagrange_leaf, n),
             "compressed_table": compress(lk["table"], lagrange_leaf, n)}
        permuted_input, permuted_table = permute_expression_pair(V, usable, L["compressed_input"], L["compressed_table"])
        permuted_input = np.concatenate([permuted_input, rnd(bf + 1)])
        permuted_table = np.concatenate([permuted_table, rnd(bf + 1)])
        L["permuted_input"], L["permuted_table"] = permuted_input, permuted_table
        # commit_values (input then table): poly, blind, commitment
        L["permuted_input_poly"] = dom.lagrange_to_coeff(permuted_input)
        L["permuted_input_blind"] = rnd1()
        ci = params.commit_lagrange(permuted_input, L["permuted_input_blind"])
        L["permuted_table_poly"] = dom.lagrange_to_coeff(permuted_table)
        L["permuted_table_blind"] = rnd1()
        ct = params.commit_lagrange(permuted_table, L["permuted_table_blind"])
        ci, ct = _affine_pts(cid, [ci, ct])
        T.write_point(ci)
        T.write_point(ct)
        L["permuted_commitments"] = (ci, ct)
        L["permuted_input_coset"] = dom.coeff_to_extended(L["permuted_input_poly"])
        L["permuted_table_coset"] = dom.coeff_to_extended(L["permuted_table_poly"])
        lookups.append(L)
    tr["lookups"] = lookups

    # step 6
    beta = T.squeeze_challenge()
    gamma = T.squeeze_challenge()
    tr["challenges"].update(beta=beta, gamma=gamma)
    tr["perm_sets"] = []

    _phase("grand products + commitments")
    # step 7: permutation argument
    chunk_len = ir["degree"] - 2
    perm_cols = ir["permutation"]
    sets = []
    deltaomega = 1
    last_z = 1

    def col_values(kind, col):
        return {"advice": advice_values, "fixed": pk.fixed_values, "instance": instance_values}[kind][col]

    for s0 in range(0, len(perm_cols), chunk_len):
        cols = perm_cols[s0:s0 + chunk_len]
        values, sigmas = [col_values(kind, col) for kind, col in cols], pk.perm_values[s0:s0 + len(cols)]
        tr["perm_sets"].append({"values": values, "sigmas": sigmas, "delta_omega0": deltaomega, "z0": last_z})
        z = permutation_product(V, dom.omega, values, sigmas, beta, gamma, deltaomega, last_z)
        deltaomega = deltaomega * pow(V.F.delta, len(cols), p) % p
        tr["perm_sets"][-1]["z_unblinded"] = z.copy()
        z[n - bf:] = rnd(bf)
        last_z = V.int1(z[n - (bf + 1)])
        blind = rnd1()
        comm = _affine_pts(cid, [params.commit_lagrange(z, blind)])[0]
        poly = dom.lagrange_to_coeff(z)
        coset = dom.coeff_to_extended(poly)
        T.write_point(comm)
        sets.append({"z": z, "poly": poly, "coset": coset, "blind": blind, "commitment": comm})
    tr["perm_z"] = [s["z"] for s in sets]

    # step 8: lookup products
    for L in lookups:
        L["z_unblinded"] = lookup_product(V, L["compressed_input"], L["compressed_table"], L["permuted_input"], L["permuted_table"], beta, gamma)
        z = np.concatenate([L["z_unblinded"][:n - bf], rnd(bf)])
        assert len(z) == n
        L["product_blind"] = rnd1()
        comm = _affine_pts(cid, [params.commit_lagrange(z, L["product_blind"])])[0]
        L["product_poly"] = dom.lagrange_to_coeff(z)
        T.write_point(comm)
        L["product_commitment"] = comm
        L["z"] = z
        L["product_coset"] = dom.coeff_to_extended(L["product_poly"])
    tr["lookup_z"] = [L["z"] for L in lookups]

    _phase("random polynomial")
    # step 9: vanishing argument: random polynomial
    random_poly = rnd(n)
    random_blind = rnd1()
    c = _affine_pts(cid, [params.commit(random_poly, random_blind)])[0]
    T.write_point(c)

    # step 10
    y = T.squeeze_challenge()
    tr["challenges"]["y"] = y
    tr["polys"] = (advice_polys + instance_polys + [q for L in lookups for q in (L["permuted_input_poly"], L["permuted_table_poly"], L["product_poly"])]
                   + [s_["poly"] for s_ in sets])          # the slot order of bz_pk_quotient

    _phase("h(X): coset NTTs + evaluation")
    # step 11: h(X) on the extended coset
    one_minus_lb = V.sub(V.const(1, ext_n), V.add(pk.l_last, pk.l_blind))      # 1 - (l_last + l_blind)
    exprs = []
    for gate in ir["gates"]:
        for poly in gate["polys"]:
            exprs.append(eval_expr(V, poly, coset_leaf, ext_n))

    def col_coset(kind, col):
        return {"advice": advice_cosets, "fixed": pk.fixed_cosets, "instance": instance_cosets}[kind][col]

    if sets:
        ones = V.const(1, ext_n)
        exprs.append(V.mul(V.sub(ones, sets[0]["coset"]), pk.l0))
        zl = sets[-1]["coset"]
        exprs.append(V.mul(V.sub(V.mul(zl, zl), zl), pk.l_last))
        last_rot = -(bf + 1)
        for i in range(1, len(sets)):
            prev = np.roll(sets[i - 1]["coset"], -last_rot * rot_scale, axis=0)
            exprs.append(V.mul(V.sub(sets[i]["coset"], prev), pk.l0))
        # the "X" of the linear term is the coset point zeta * w_ext^i
        coset_x = V.powers(V.F.zeta, dom.extended_omega, ext_n)
        for ci, s in enumerate(sets):
            cols = perm_cols[ci * chunk_len:(ci + 1) * chunk_len]
            left = np.roll(s["coset"], -rot_scale, axis=0)
            for j, (kind, col) in enumerate(cols):
                t = V.add_const(V.add(col_coset(kind, col), V.scale(pk.perm_cosets[ci * chunk_len + j], beta)), gamma)
                left = V.mul(left, t)
            right = s["coset"]
            cur_delta = beta * pow(V.F.delta, ci * chunk_len, p) % p
            for (kind, col) in cols:
                t = V.add_const(V.add(col_coset(kind, col), V.scale(coset_x, cur_delta)), gamma)
                right = V.mul(right, t)
                cur_delta = cur_delta * V.F.delta % p
            exprs.append(V.mul(V.sub(left, right), one_minus_lb))
    for L, lk in zip(lookups, ir["lookups"]):
        def compress_c(es):
            acc = V.zeros(ext_n)
            for e in es:
                acc = V.add(V.scale(acc, theta), eval_expr(V, e, coset_leaf, ext_n))
            return acc
        zc, ac, sc = L["product_coset"], L["permuted_input_coset"], L["permuted_table_coset"]
        ones = V.const(1, ext_n)
        exprs.append(V.mul(V.sub(ones, zc), pk.l0))
        exprs.append(V.mul(V.sub(V.mul(zc, zc), zc), pk.l_last))
        left = V.mul(V.mul(np.roll(zc, -rot_scale, axis=0), V.add_const(ac, beta)), V.add_const(sc, gamma))
        right = V.mul(V.mul(zc, V.add_const(compress_c(lk["input"]), beta)), V.add_const(compress_c(lk["table"]), gamma))
        exprs.append(V.mul(V.sub(left, right), one_minus_lb))
        exprs.append(V.mul(V.sub(ac, sc), pk.l0))
        a_prev = np.roll(ac, rot_scale, axis=0)
        exprs.append(V.mul(V.mul(V.sub(ac, sc), V.sub(ac, a_prev)), one_minus_lb))
    h = V.zeros(ext_n)
    for e in exprs:
        h = V.add(V.scale(h, y), e)
    tr["num_expressions"] = len(exprs)

    _phase("h(X): inverse NTT + piece commitments")
    # step 12: divide by t(X), back to coefficients, split, commit pieces
    tr["h_extended_before_division"] = h
    h = dom.divide_by_vanishing_poly(h)
    tr["h_extended"] = h
    h_coeffs = dom.extended_to_coeff(h)
    h_pieces = [h_coeffs[i * n:(i + 1) * n] for i in range(dom.quotient_poly_degree)]
    h_blinds = [rnd1() for _ in h_pieces]
    h_comm = _affine_pts(cid, [params.commit(pc, b) for pc, b in zip(h_pieces, h_blinds)])
    for cpt in h_comm:
        T.write_point(cpt)
    tr["h_commitments"] = h_comm
    tr["h_pieces"] = h_pieces

    # step 13
    x = T.squeeze_challenge()
    xn = pow(x, n, p)
    tr["challenges"]["x"] = x

    _phase("evaluations")
    # step 14: instance / advice / fixed evaluations
    for col, rot in ir["instance_queries"]:
        T.write_scalar(V.eval_polynomial(instance_polys[col], dom.rotate_omega(x, rot)))
    for col, rot in ir["advice_queries"]:
        T.write_scalar(V.eval_polynomial(advice_polys[col], dom.rotate_omega(x, rot)))
    for col, rot in ir["fixed_queries"]:
        T.write_scalar(V.eval_polynomial(pk.fixed_polys[col], dom.rotate_omega(x, rot)))

    # step 15: vanishing evaluate
    h_poly = V.zeros(n)
    h_blind = 0
    for pc, b in zip(reversed(h_pieces), reversed(h_blinds)):
        h_poly = V.add(V.scale(h_poly, xn), pc)
        h_blind = (h_blind * xn + b) % p
    T.write_scalar(V.eval_polynomial(random_poly, x))

    # step 16: permutation common evaluations
    for q in pk.perm_polys:
        T.write_scalar(V.eval_polynomial(q, x))
    # step 17: permutation product evaluations
    x_next = dom.rotate_omega(x, 1)
    x_prev = dom.rotate_omega(x, -1)
    x_last = dom.rotate_omega(x, -(bf + 1))
    for i, s in enumerate(sets):
        T.write_scalar(V.eval_polynomial(s["poly"], x))
        T.write_scalar(V.eval_polynomial(s["poly"], x_next))
        if i != len(sets) - 1:
            T.write_scalar(V.eval_polynomial(s["poly"], x_last))
    # step 18: lookup evaluations
    for L in lookups:
        T.write_scalar(V.eval_polynomial(L["product_poly"], x))
        T.write_scalar(V.eval_polynomial(L["product_poly"], x_next))
        T.write_scalar(V.eval_polynomial(L["permuted_input_poly"], x))
        T.write_scalar(V.eval_polynomial(L["permuted_input_poly"], x_prev))
        T.write_scalar(V.eval_polynomial(L["permuted_table_poly"], x))

    _phase("multiopen")
    # step 19: query list  (id, point, (poly, blind))
    Q = []
    for col, rot in ir["instance_queries"]:
        Q.append((("instance", col), dom.rotate_omega(x, rot), (instance_polys[col], 1)))
    for col, rot in ir["advice_queries"]:
        Q.append((("advice", col), dom.rotate_omega(x, rot), (advice_polys[col], advice_blinds[col])))
    for i, s in enumerate(sets):
        Q.append((("perm_z", i), x, (s["poly"], s["blind"])))
        Q.append((("perm_z", i), x_next, (s["poly"], s["blind"])))
    for i in reversed(range(len(sets) - 1)):
        Q.append((("perm_z", i), x_last, (sets[i]["poly"], sets[i]["blind"])))
    for i, L in enumerate(lookups):
        Q.append((("lk_z", i), x, (L["product_poly"], L["product_blind"])))
        Q.append((("lk_a", i), x, (L["permuted_input_poly"], L["permuted_input_blind"])))
        Q.append((("lk_s", i), x, (L["permuted_table_poly"], L["permuted_table_blind"])))
        Q.append((("lk_a", i), x_prev, (L["permuted_input_poly"], L["permuted_input_blind"])))
        Q.append((("lk_z", i), x_next, (L["product_poly"], L["product_blind"])))
    for col, rot in ir["fixed_queries"]:
        Q.append((("fixed", col), dom.rotate_omega(x, rot), (pk.fixed_polys[col], 1)))
    for i, q in enumerate(pk.perm_polys):
        Q.append((("sigma", i), x, (q, 1)))
    Q.append((("h",), x, (h_poly, h_blind)))
    Q.append((("random",), x, (random_poly, random_blind)))

    # step 20: multiopen
    x1 = T.squeeze_challenge()
    x2 = T.squeeze_challenge()
    tr["challenges"].update(x1=x1, x2=x2)
    tr["queries"] = Q
    cmap, point_sets = construct_intermediate_sets(Q)
    q_polys = [None] * len(point_sets)
    q_blinds = [0] * len(point_sets)
    for d in cmap:
        poly, blind = d["first_payload"]
        si = d["set_index"]
        q_polys[si] = poly if q_polys[si] is None else V.add(V.scale(q_polys[si], x1), poly)
        q_blinds[si] = (q_blinds[si] * x1 + blind) % p
    q_prime = None
    for pts, poly in zip(point_sets, q_polys):
        quo = poly
        for pt in pts:
            quo = V.kate_division(quo, pt)
        quo = np.concatenate([quo, V.zeros(n - len(quo))])
        q_prime = quo if q_prime is None else V.add(V.scale(q_prime, x2), quo)
    q_prime_blind = rnd1()
    qc = _affine_pts(cid, [params.commit(q_prime, q_prime_blind)])[0]
    T.write_point(qc)
    x3 = T.squeeze_challenge()
    for qp in q_polys:
        T.write_scalar(V.eval_polynomial(qp, x3))
    x4 = T.squeeze_challenge()
    tr["challenges"].update(x3=x3, x4=x4)
    tr["q_polys"], tr["q_prime"] = q_polys, q_prime
    p_poly, p_blind = q_prime, q_prime_blind
    for qp, qb in zip(q_polys, q_blinds):
        p_poly = V.add(V.scale(p_poly, x4), qp)
        p_blind = (p_blind * x4 + qb) % p
    tr["p_poly"] = p_poly
    tr["point_sets"] = point_sets

    _phase("inner product argument")
    # step 21: inner product argument
    ipa_create_proof(params, draws, T, p_poly, p_blind, x3, tr)
    _phase("done")


def ipa_create_proof(params, draws, T, p_poly, p_blind, x3, tr=None):
    """[U: src/poly/commitment/prover.rs::create_proof]"""
    f, cid = params.sf, params.curve_id
    V = Vec(f)
    p = V.p
    n, k = params.n, params.k
    s_poly = draws.take(f, n)
    s_at_x3 = V.eval_polynomial(s_poly, x3)
    s_poly[0] = V.m((V.int1(s_poly[0]) - s_at_x3) % p)
    s_blind = V.int1(draws.take(f, 1)[0])
    sc = _affine_pts(cid, [params.commit(s_poly, s_blind)])[0]
    T.write_point(sc)
    xi = T.squeeze_challenge()
    z = T.squeeze_challenge()
    p_prime = V.add(V.scale(s_poly, xi), p_poly)
    v = V.eval_polynomial(p_prime, x3)
    p_prime[0] = V.m((V.int1(p_prime[0]) - v) % p)
    fblind = (s_blind * xi + p_blind) % p
    if tr is not None:
        tr["ipa"] = {"p_prime": p_prime.copy(), "x3": x3, "z": z, "xi": xi, "rounds": []}
    b = V.powers(1, x3, n)
    g_prime = params.g.copy()
    u_w = np.stack([params.u, params.w])
    rounds = []
    for j in range(k):
        half = 1 << (k - j - 1)
        l_j = co.best_multiexp(cid, p_prime[half:2 * half], g_prime[:half])
        r_j = co.best_multiexp(cid, p_prime[:half], g_prime[half:2 * half])
        value_l = V.inner_product(p_prime[half:2 * half], b[:half])
        value_r = V.inner_product(p_prime[:half], b[half:2 * half])
        l_rand = V.int1(draws.take(f, 1)[0])
        r_rand = V.int1(draws.take(f, 1)[0])
        l2 = co.best_multiexp(cid, V.arr([value_l * z % p, l_rand]), u_w)
        r2 = co.best_multiexp(cid, V.arr([value_r * z % p, r_rand]), u_w)
        C = co.CURVES[cid][0]
        l_aff, l2_aff, r_aff, r2_aff = _affine_pts(cid, [l_j, l2, r_j, r2])
        l_pt, r_pt = C.add(l_aff, l2_aff), C.add(r_aff, r2_aff)
        T.write_point(l_pt)
        T.write_point(r_pt)
        u_j = T.squeeze_challenge()
        u_inv = pow(u_j, -1, p)
        p_prime = V.add(p_prime[:half], V.scale(p_prime[half:2 * half], u_inv))
        b = V.add(b[:half], V.scale(b[half:2 * half], u_j))
        g_prime = np.ascontiguousarray(g_prime[:2 * half]).copy()
        co.lib().orc_generator_collapse(cid, co._p(g_prime), ctypes.c_size_t(2 * half), co._p(V.m(u_j)))
        g_prime = g_prime[:half]
        fblind = (fblind + l_rand * u_inv + r_rand * u_j) % p
        rounds.append((l_pt, r_pt, u_j))
        if tr is not None:
            tr["ipa"]["rounds"].append({"L": l_pt, "R": r_pt, "u": u_j, "l_rand": l_rand, "r_rand": r_rand})
    c = V.int1(p_prime[0])
    T.write_scalar(c)
    T.write_scalar(fblind)
    if tr is not None:
        tr["ipa_rounds"] = rounds
        tr["ipa"]["c"] = c


# ------------------------------------------------------------------------------------------------------
# verify_proof  [U: src/plonk/verifier.rs + argument verifiers + poly/multiopen/verifier.rs +
#                poly/commitment/verifier.rs; SURVEY App. H].  SingleVerifier semantics: accept iff the final
#                MSM evaluates to the identity.
# ------------------------------------------------------------------------------------------------------
def verify_proof(params, pk, instances, proof):
    """pk supplies the verifying-key part only (ir, domain, fixed/perm commitments, vk_repr).  Returns bool."""
    try:
        return _verify(params, pk, instances, proof)
    except (IOError, AssertionError, ValueError):
        return False


def _verify(params, pk, instances, proof):
    ir, dom = pk.ir, pk.domain
    f, cid = params.sf, params.curve_id
    C = co.CURVES[cid][0]
    V = Vec(f)
    p = V.p
    n, k = params.n, params.k
    bf = ir["blinding_factors"]
    T = Blake2bTranscript(cid, proof)
    if len(instances) != ir["num_instance"]:
        return False
    inst_comm = []
    for vals in instances:
        if len(vals) > n - (bf + 1):
            return False
        col = V.zeros(n)
        if len(vals):
            col[:len(vals)] = V.arr(vals)
        inst_comm.append(params.commit_lagrange(col, 1))
    inst_comm = _affine_pts(cid, inst_comm)
    T.common_scalar(pk.vk_repr)
    for c in inst_comm:
        T.common_point(c)
    adv_comm = [T.read_point() for _ in range(ir["num_advice"])]
    theta = T.squeeze_challenge()
    lk_perm = [(T.read_point(), T.read_point()) for _ in ir["lookups"]]
    beta = T.squeeze_challenge()
    gamma = T.squeeze_challenge()
    chunk_len = ir["degree"] - 2
    perm_cols = ir["permutation"]
    nsets = (len(perm_cols) + chunk_len - 1) // chunk_len
    perm_z = [T.read_point() for _ in range(nsets)]
    lk_z = [T.read_point() for _ in ir["lookups"]]
    random_comm = T.read_point()
    y = T.squeeze_challenge()
    h_comm = [T.read_point() for _ in range(dom.quotient_poly_degree)]
    x = T.squeeze_challenge()
    instance_evals = [T.read_scalar() for _ in ir["instance_queries"]]
    advice_evals = [T.read_scalar() for _ in ir["advice_queries"]]
    fixed_evals = [T.read_scalar() for _ in ir["fixed_queries"]]
    random_eval = T.read_scalar()
    sigma_evals = [T.read_scalar() for _ in perm_cols]
    perm_evals = []
    for i in range(nsets):
        e = {"z": T.read_scalar(), "z_next": T.read_scalar()}
        if i != nsets - 1:
            e["z_last"] = T.read_scalar()
        perm_evals.append(e)
    lk_evals = []
    for _ in ir["lookups"]:
        lk_evals.append({"z": T.read_scalar(), "z_next": T.read_scalar(), "a": T.read_scalar(),
                         "a_inv": T.read_scalar(), "s": T.read_scalar()})

    # vanishing argument: expected h(x)
    xn = pow(x, n, p)
    # l_i_range(x, xn, -(bf+1)..=0):  l_i(x) = omega^i (x^n - 1) / (n (x - omega^i))
    n_inv = pow(n, -1, p)
    l_evals = []
    for rot in range(-(bf + 1), 1):
        w_i = dom.rotate_omega(1, rot)
        l_evals.append(w_i * (xn - 1) % p * n_inv % p * pow((x - w_i) % p, -1, p) % p)
    l_last = l_evals[0]
    l_blind = sum(l_evals[1:bf + 1]) % p
    l_0 = l_evals[bf + 1]

    aq = {tuple(q): i for i, q in enumerate(ir["advice_queries"])}
    fq = {tuple(q): i for i, q in enumerate(ir["fixed_queries"])}
    iq = {tuple(q): i for i, q in enumerate(ir["instance_queries"])}

    def leaf(kind, col, rot):
        if kind == "advice": return advice_evals[aq[(col, rot)]]
        if kind == "fixed": return fixed_evals[fq[(col, rot)]]
        return instance_evals[iq[(col, rot)]]

    exprs = []
    for gate in ir["gates"]:
        for poly in gate["polys"]:
            exprs.append(eval_expr_scalar(p, poly, leaf))
    if nsets:
        one_minus = (1 - (l_last + l_blind)) % p
        exprs.append(l_0 * (1 - perm_evals[0]["z"]) % p)
        zl = perm_evals[-1]["z"]
        exprs.append(l_last * (zl * zl - zl) % p)
        for i in range(1, nsets):
            exprs.append((perm_evals[i]["z"] - perm_evals[i - 1]["z_last"]) * l_0 % p)
        for ci in range(nsets):
            cols = perm_cols[ci * chunk_len:(ci + 1) * chunk_len]
            left = perm_evals[ci]["z_next"]
            for j, (kind, col) in enumerate(cols):
                left = left * (leaf(kind, col, 0) + beta * sigma_evals[ci * chunk_len + j] + gamma) % p
            right = perm_evals[ci]["z"]
            cur_delta = beta * x % p * pow(V.F.delta, ci * chunk_len, p) % p
            for (kind, col) in cols:
                right = right * (leaf(kind, col, 0) + cur_delta + gamma) % p
                cur_delta = cur_delta * V.F.delta % p
            exprs.append((left - right) * one_minus % p)
    for lk, e in zip(ir["lookups"], lk_evals):
        one_minus = (1 - (l_last + l_blind)) % p
        def compress(es):
            acc = 0
            for ex in es:
                acc = (acc * theta + eval_expr_scalar(p, ex, leaf)) % p
            return acc
        exprs.append(l_0 * (1 - e["z"]) % p)
        exprs.append(l_last * (e["z"] * e["z"] - e["z"]) % p)
        left = e["z_next"] * (e["a"] + beta) % p * (e["s"] + gamma) % p
        right = e["z"] * (compress(lk["input"]) + beta) % p * (compress(lk["table"]) + gamma) % p
        exprs.append((left - right) * one_minus % p)
        exprs.append(l_0 * (e["a"] - e["s"]) % p)
        exprs.append((e["a"] - e["s"]) * (e["a"] - e["a_inv"]) % p * one_minus % p)
    expected_h = 0
    for ev in exprs:
        expected_h = (expected_h * y + ev) % p
    expected_h = expected_h * pow((xn - 1) % p, -1, p) % p

    # h commitment = sum xn^i H_i  (an MSM in the reference; a point here)
    h_pt = None
    for cpt in reversed(h_comm):
        h_pt = C.add(C.mul(h_pt, xn), cpt)

    x_next = dom.rotate_omega(x, 1)
    x_prev = dom.rotate_omega(x, -1)
    x_last = dom.rotate_omega(x, -(bf + 1))
    Q = []      # (id, point, (commitment point, eval))
    for (col, rot), ev in zip(ir["instance_queries"], instance_evals):
        Q.append((("instance", col), dom.rotate_omega(x, rot), (inst_comm[col], ev)))
    for (col, rot), ev in zip(ir["advice_queries"], advice_evals):
        Q.append((("advice", col), dom.rotate_omega(x, rot), (adv_comm[col], ev)))
    for i in range(nsets):
        Q.append((("perm_z", i), x, (perm_z[i], perm_evals[i]["z"])))
        Q.append((("perm_z", i), x_next, (perm_z[i], perm_evals[i]["z_next"])))
    for i in reversed(range(nsets - 1)):
        Q.append((("perm_z", i), x_last, (perm_z[i], perm_evals[i]["z_last"])))
    for i, e in enumerate(lk_evals):
        Q.append((("lk_z", i), x, (lk_z[i], e["z"])))
        Q.append((("lk_a", i), x, (lk_perm[i][0], e["a"])))
        Q.append((("lk_s", i), x, (lk_perm[i][1], e["s"])))
        Q.append((("lk_a", i), x_prev, (lk_perm[i][0], e["a_inv"])))
        Q.append((("lk_z", i), x_next, (lk_z[i], e["z_next"])))
    for (col, rot), ev in zip(ir["fixed_queries"], fixed_evals):
        Q.append((("fixed", col), dom.rotate_omega(x, rot), (pk.fixed_commitments[col], ev)))
    for i, ev in enumerate(sigma_evals):
        Q.append((("sigma", i), x, (pk.perm_commitments[i], ev)))
    Q.append((("h",), x, (h_pt, expected_h)))
    Q.append((("random",), x, (random_comm, random_eval)))

    # multiopen verifier
    x1 = T.squeeze_challenge()
    x2 = T.squeeze_challenge()
    cmap, point_sets = construct_intermediate_sets(Q)
    q_comm = [None] * len(point_sets)
    q_eval_sets = [[0] * len(ps) for ps in point_sets]
    for d in cmap:
        si = d["set_index"]
        comm = d["first_payload"][0]
        q_comm[si] = C.add(C.mul(q_comm[si], x1), comm)
        for j, (_, ev) in enumerate(d["evals"]):
            q_eval_sets[si][j] = (q_eval_sets[si][j] * x1 + ev) % p
    q_prime_comm = T.read_point()
    x3 = T.squeeze_challenge()
    u_evals = [T.read_scalar() for _ in point_sets]
    msm_eval = 0
    for pts, evs, u_ev in zip(point_sets, q_eval_sets, u_evals):
        r_eval = _lagrange_eval(p, pts, evs, x3)
        den = 1
        for pt in pts:
            den = den * (x3 - pt) % p
        msm_eval = (msm_eval * x2 + (u_ev - r_eval) * pow(den, -1, p)) % p
    x4 = T.squeeze_challenge()
    M = q_prime_comm
    v = msm_eval
    for comm, u_ev in zip(q_comm, u_evals):
        M = C.add(C.mul(M, x4), comm)
        v = (v * x4 + u_ev) % p

    # IPA verifier
    g0 = co.points_from_mont(cid, params.g[:1])[0]
    w_pt = co.points_from_mont(cid, params.w[None, :])[0]
    u_pt = co.points_from_mont(cid, params.u[None, :])[0]
    M = C.add(M, C.mul(g0, (-v) % p))
    s_comm = T.read_point()
    xi = T.squeeze_challenge()
    M = C.add(M, C.mul(s_comm, xi))
    z = T.squeeze_challenge()
    us = []
    for _ in range(k):
        l_pt = T.read_point()
        r_pt = T.read_point()
        u_j = T.squeeze_challenge()
        us.append(u_j)
        M = C.add(M, C.add(C.mul(l_pt, pow(u_j, -1, p)), C.mul(r_pt, u_j)))
    c = T.read_scalar()
    fb = T.read_scalar()
    # compute_b
    tmp, cur = 1, x3
    for u_j in reversed(us):
        tmp = tmp * (1 + u_j * cur) % p
        cur = cur * cur % p
    b = tmp
    M = C.add(M, C.mul(u_pt, (-(c * b % p) * z) % p))
    M = C.add(M, C.mul(w_pt, (-fb) % p))
    # compute_s(u, -c) and the final G MSM
    s = [0] * n
    s[0] = (-c) % p
    for i, u_j in enumerate(reversed(us)):
        size = 1 << i
        for t in range(size):
            s[size + t] = s[t] * u_j % p
    gs = co.best_multiexp(cid, V.arr(s), params.g)
    M = C.add(M, _affine_pts(cid, [gs])[0])
    return M is None and T.rpos == len(proof)


def _lagrange_eval(p, points, evals, x):
    """arithmetic::lagrange_interpolate(points, evals) evaluated at x."""
    total = 0
    for j, (xj, yj) in enumerate(zip(points, evals)):
        num, den = 1, 1
        for m, xm in enumerate(points):
            if m != j:
                num = num * (x - xm) % p
                den = den * (xj - xm) % p
        total = (total + yj * num % p * pow(den, -1, p)) % p
    return total
