// Host check of the gate-DAG compiler (csrc/evalprog.h): random families of gate polynomials with shared
// sub-expressions and shared factors are compiled with every combination of {cse, hoist}; the emitted program is run
// by a scalar model of eval_program_kernel over F_p (p = 2^61 - 1) and must equal  sum_e y^(E-1-e) * expr_e  evaluated
// straight from the token streams.  Also reports the multiplication counts (the quantity the rewrite is for).
#include "../../battlezips-halo2_b200/csrc/evalprog.h"
#include <cstdio>
#include <cstdlib>
#include <random>
using namespace bz;
typedef unsigned long long u64;
static const u64 P = (1ull << 61) - 1;
static u64 mulm(u64 a, u64 b) { return (u64)((unsigned __int128)a * b % P); }
static u64 addm(u64 a, u64 b) { return (a + b) % P; }
static u64 subm(u64 a, u64 b) { return (a + P - b) % P; }

static std::mt19937_64 rng(12345);
static const int NADV = 6, NFIX = 4, NINST = 2, NCONST = 8, G = NADV;
static uint32_t g_inst_base = G;
static int g_max_tmp = -1;
static u64 val_const[4096], salt = 1;
static u64 hval(u64 kind, u64 col, long long rot) {           // pseudo-random value of a column cell at the evaluation point
  u64 z = salt * 0x9E3779B97F4A7C15ull + kind * 0xBF58476D1CE4E5B9ull + col * 0x94D049BB133111EBull + (u64)(rot + 1000) * 0xD6E8FEB86659FD93ull;
  z ^= z >> 31; z *= 0x7FB5D329728EA185ull; z ^= z >> 27; z *= 0x81DADEF4BC2DD44Dull; z ^= z >> 33;
  return z % P;
}
static std::vector<std::vector<Token>> pool;
// derived columns (split_fixed_subexpressions): shared slots >= g_derived_base hold the value of their sub-expression
static uint32_t g_derived_base = 0xffffffffu;
static std::vector<u64> g_derived;
static u64 sval(uint32_t slot, long long rot) { return slot >= g_derived_base ? g_derived[slot - g_derived_base] : hval(1, slot, rot); }

static std::vector<Token> gen(int depth) {
  if (!pool.empty() && depth < 4 && rng() % 10 < 3) return pool[rng() % pool.size()];
  std::vector<Token> r;
  if (depth == 0 || rng() % 6 == 0) {
    switch (rng() % 4) {
      case 0: r.push_back(Token{0, (uint32_t)(rng() % NCONST), 0}); break;
      case 1: r.push_back(Token{1, (uint32_t)(rng() % NADV), (int32_t)(rng() % 3) - 1}); break;
      case 2: r.push_back(Token{2, (uint32_t)(rng() % NFIX), (int32_t)(rng() % 3) - 1}); break;
      default: r.push_back(Token{3, (uint32_t)(rng() % NINST), (int32_t)(rng() % 3) - 1}); break;
    }
    return r;
  }
  const int kind = rng() % 8;
  std::vector<Token> a = gen(depth - 1);
  if (kind == 0) { r = a; r.push_back(Token{4, 0, 0}); }
  else if (kind == 1) { r = a; r.push_back(Token{7, (uint32_t)(rng() % NCONST), 0}); }
  else {
    std::vector<Token> b = (rng() % 8 == 0) ? a : gen(depth - 1);
    r = a; r.insert(r.end(), b.begin(), b.end());
    if (kind >= 5 && rng() % 2) { r.push_back(Token{4, 0, 0}); r.push_back(Token{5, 0, 0}); }     // a - b
    else r.push_back(Token{kind <= 4 ? 6u : 5u, 0, 0});
  }
  if (r.size() > 2 && r.size() < 40 && rng() % 3 == 0) pool.push_back(r);
  return r;
}

static u64 eval_tokens(const std::vector<Token>& t, uint32_t lo, uint32_t hi, u64& nmul) {
  std::vector<u64> st;
  for (uint32_t i = lo; i < hi; ++i) {
    const Token& k = t[i];
    switch (k.op) {
      case 0: st.push_back(val_const[k.a]); break;
      case 1: st.push_back(hval(0, k.a, k.b)); break;
      case 2: st.push_back(sval(k.a, k.b)); break;
      case 3: st.push_back(hval(0, g_inst_base + k.a, k.b)); break;
      case 4: st.back() = subm(0, st.back()); break;
      case 5: { u64 r = st.back(); st.pop_back(); st.back() = addm(st.back(), r); break; }
      case 6: { u64 r = st.back(); st.pop_back(); st.back() = mulm(st.back(), r); ++nmul; break; }
      case 7: st.back() = mulm(st.back(), val_const[k.a]); ++nmul; break;
    }
  }
  return st.back();
}

static u64 run_program(const ProgBuilder& pb, u64& nmul) {
  u64 st[EVAL_STACK], tmp[EVAL_TMP], acc = 0; int sp = 0;
  for (uint32_t ins : pb.code) {
    const uint32_t op = ins & 15u, x = (ins >> 4) & 0xfffu, y = ins >> 16;
    switch (op) {
      case OP_PUSH_P: st[sp++] = hval(0, x, pb.rot_table[y]); break;
      case OP_PUSH_S: st[sp++] = sval(x, pb.rot_table[y]); break;
      case OP_PUSH_C: st[sp++] = val_const[ins >> 4]; break;
      case OP_ADD: --sp; st[sp - 1] = addm(st[sp - 1], st[sp]); break;
      case OP_SUB: --sp; st[sp - 1] = subm(st[sp - 1], st[sp]); break;
      case OP_MUL: --sp; st[sp - 1] = mulm(st[sp - 1], st[sp]); ++nmul; break;
      case OP_NEG: st[sp - 1] = subm(0, st[sp - 1]); break;
      case OP_MULC: st[sp - 1] = mulm(st[sp - 1], val_const[ins >> 4]); ++nmul; break;
      case OP_ADDC: st[sp - 1] = addm(st[sp - 1], val_const[ins >> 4]); break;
      case OP_FOLD: --sp; acc = addm(mulm(acc, val_const[ins >> 4]), st[sp]); ++nmul; break;
      case OP_ACC_MULC: acc = mulm(acc, val_const[ins >> 4]); ++nmul; break;
      case OP_TEE: if ((ins >> 4) >= (uint32_t)EVAL_TMP) { printf("tmp overflow\n"); exit(1); } tmp[ins >> 4] = st[sp - 1]; if ((int)(ins >> 4) > g_max_tmp) g_max_tmp = (int)(ins >> 4); break;
      case OP_PUSH_T: st[sp++] = tmp[ins >> 4]; break;
      default: printf("bad op\n"); exit(1);
    }
    if (sp < 0 || sp > EVAL_STACK) { printf("stack out of range %d\n", sp); exit(1); }
  }
  if (sp != 0) { printf("stack not empty\n"); exit(1); }
  return acc;
}

// file mode: the gate polynomials of a real constraint system, one line per polynomial
//   "<tier> <e> <ntok> (<op> <a> <b>)*"   preceded by a header line "<E> <instance slot base> <#consts>"
// prints per tier: polynomials, multiplications as trees / as one DAG, deepest stack, temporaries used
static int file_mode(const char* path) {
  FILE* f = fopen(path, "r");
  if (!f) { printf("cannot open %s\n", path); return 1; }
  uint32_t E, ibase, nconst;
  if (fscanf(f, "%u %u %u", &E, &ibase, &nconst) != 3) return 1;
  g_inst_base = ibase;
  const uint32_t YP0 = nconst;
  if (YP0 + E + 1 > 4096) { printf("too many constants\n"); return 1; }
  struct PolyIn { uint32_t tier, e; std::vector<Token> t; };
  std::vector<PolyIn> in;
  for (;;) {
    PolyIn p; uint32_t nt;
    if (fscanf(f, "%u %u %u", &p.tier, &p.e, &nt) != 3) break;
    for (uint32_t i = 0; i < nt; ++i) { Token k; if (fscanf(f, "%u %u %d", &k.op, &k.a, &k.b) != 3) return 1; p.t.push_back(k); }
    in.push_back(p);
  }
  fclose(f);
  for (uint32_t tier = 0; tier < 3; ++tier) {
    salt = 77 + tier;
    for (uint32_t i = 0; i < nconst; ++i) val_const[i] = hval(2, i, 0);
    const u64 y = hval(3, 0, 0);
    { u64 p = 1; for (uint32_t d = 0; d <= E; ++d) { val_const[YP0 + d] = p; p = mulm(p, y); } }
    std::vector<Token> tokens; std::vector<uint32_t> lo, hi, eidx;
    for (const PolyIn& p : in) if (p.tier == tier) { lo.push_back((uint32_t)tokens.size()); tokens.insert(tokens.end(), p.t.begin(), p.t.end()); hi.push_back((uint32_t)tokens.size()); eidx.push_back(p.e); }
    if (eidx.empty()) { printf("tier %u polys 0\n", tier); continue; }
    u64 want = 0, naive = 0;
    for (size_t i = 0; i < eidx.size(); ++i) want = addm(want, mulm(eval_tokens(tokens, lo[i], hi[i], naive), val_const[YP0 + (E - 1 - eidx[i])]));
    naive += eidx.size();
    // what the library does before compiling: fixed-only sub-expressions (compressed selectors) become derived columns
    std::vector<DerivedColumn> derived; std::vector<Token> qtokens; std::vector<uint32_t> goff{0}, qoff;
    for (size_t i = 0; i < eidx.size(); ++i) goff.push_back(hi[i]);
    g_derived_base = 0xffffffffu; g_derived.clear();
    split_fixed_subexpressions(tokens, goff, 2000, derived, qtokens, qoff);
    { u64 dm = 0; std::vector<u64> vals; for (const DerivedColumn& d : derived) vals.push_back(eval_tokens(d.tokens, 0, (uint32_t)d.tokens.size(), dm)); g_derived = vals; g_derived_base = 2000; }
    tokens = qtokens;
    for (size_t i = 0; i < eidx.size(); ++i) { lo[i] = qoff[i]; hi[i] = qoff[i + 1]; }
    GateDag dag; dag.advice_slot_of_instance = ibase; dag.canon_mul = dag.sort_rest = getenv("BZ_NO_CANON") == nullptr;
    for (size_t i = 0; i < eidx.size(); ++i) dag.add(tokens, lo[i], hi[i], eidx[i]);
    dag.plan();
    ProgBuilder pb; int prev = -1;
    for (const GateDag::Group& g : dag.groups) { dag.emit_group(pb, g, prev, [&](uint32_t d) { return YP0 + d; }); prev = (int)dag.polys[g.first + g.count - 1].e; }
    if ((uint32_t)prev != E - 1) pb.accmul(YP0 + (E - 1 - (uint32_t)prev));
    if (pb.max_depth > EVAL_STACK) { printf("tier %u: stack depth %d exceeds EVAL_STACK\n", tier, pb.max_depth); return 1; }
    u64 nm = 0; g_max_tmp = -1;
    if (run_program(pb, nm) != want) { printf("MISMATCH tier %u\n", tier); return 1; }
    printf("tier %u polys %zu tree_muls %llu dag_muls %llu depth %d temporaries %d instructions %zu derived %zu\n", tier, eidx.size(), naive, nm, pb.max_depth, g_max_tmp + 1, pb.code.size(), derived.size());
    g_derived_base = 0xffffffffu;
  }
  printf("ok\n");
  return 0;
}

int main(int argc, char** argv) {
  if (argc > 1) return file_mode(argv[1]);
  u64 tot_naive = 0, tot[6] = {0, 0, 0, 0, 0, 0};
  int deepest = 0;
  for (int trial = 0; trial < 400; ++trial) {
    pool.clear();
    salt = rng();
    for (int i = 0; i < NCONST; ++i) val_const[i] = rng() % P;
    const uint32_t E = 4 + rng() % 30, YP0 = 16;               // constants 16.. : y^0 .. y^E
    const u64 y = rng() % P;
    { u64 p = 1; for (uint32_t d = 0; d <= E; ++d) { val_const[YP0 + d] = p; p = mulm(p, y); } }
    // polynomials: "gates" of 1..4 polynomials sharing a selector-like factor, at a random subset of the indices 0..E-1
    std::vector<Token> tokens; std::vector<uint32_t> lo, hi, eidx;
    for (uint32_t e = 0; e < E;) {
      const uint32_t m = 1 + rng() % 4;
      std::vector<Token> sel = rng() % 4 ? std::vector<Token>{Token{2, (uint32_t)(rng() % NFIX), 0}} : gen(2);
      for (uint32_t i = 0; i < m && e < E; ++i, ++e) {
        if (rng() % 4 == 0) continue;                          // this index belongs to another launch
        std::vector<Token> body = gen(1 + rng() % 4), poly;
        const int shape = rng() % 4;
        if (shape == 0) poly = body;                           // no common factor
        else if (shape == 1) { poly = body; poly.insert(poly.end(), sel.begin(), sel.end()); poly.push_back(Token{6, 0, 0}); }
        else { poly = sel; poly.insert(poly.end(), body.begin(), body.end()); poly.push_back(Token{6, 0, 0}); }
        lo.push_back((uint32_t)tokens.size()); tokens.insert(tokens.end(), poly.begin(), poly.end()); hi.push_back((uint32_t)tokens.size()); eidx.push_back(e);
      }
    }
    if (eidx.empty()) continue;
    u64 want = 0, naive = 0;
    for (size_t i = 0; i < eidx.size(); ++i) { want = addm(want, mulm(eval_tokens(tokens, lo[i], hi[i], naive), val_const[YP0 + (E - 1 - eidx[i])])); }
    naive += eidx.size();                                      // one fold multiplication per polynomial
    tot_naive += naive;
    for (int mode = 0; mode < 6; ++mode) {            // mode 4 = cse + hoist + hoisting through nested products, 5 = 4 + products as sorted chains
      GateDag dag; dag.cse = mode >= 4 || (mode & 1); dag.hoist = mode >= 4 || (mode & 2); dag.nested = mode >= 4; dag.canon_mul = dag.sort_rest = mode == 5; dag.advice_slot_of_instance = G;
      for (size_t i = 0; i < eidx.size(); ++i) dag.add(tokens, lo[i], hi[i], eidx[i]);
      dag.plan();
      ProgBuilder pb;
      int prev = -1;
      for (const GateDag::Group& g : dag.groups) { dag.emit_group(pb, g, prev, [&](uint32_t d) { if (d > E) { printf("y power out of range\n"); exit(1); } return YP0 + d; }); prev = (int)dag.polys[g.first + g.count - 1].e; }
      if ((uint32_t)prev != E - 1) pb.accmul(YP0 + (E - 1 - (uint32_t)prev));
      if (pb.max_depth > deepest) deepest = pb.max_depth;
      if (pb.max_depth > EVAL_STACK) { printf("trial %d mode %d: depth %d\n", trial, mode, pb.max_depth); continue; }   // the library rejects these with an error
      u64 nm = 0;
      const u64 got = run_program(pb, nm);
      if (got != want) { printf("MISMATCH trial %d mode %d\n", trial, mode); return 1; }
      tot[mode] += nm;
    }
  }
  printf("ok naive %llu plain %llu cse %llu hoist %llu both %llu nested %llu canon %llu deepest %d\n", tot_naive, tot[0], tot[1], tot[2], tot[3], tot[4], tot[5], deepest);
  return 0;
}
