// Program format of the expression evaluator (poly.cuh `eval_program_kernel`) and the host-side compiler that turns
// the gate polynomials of a constraint system into it.  Replaces what halo2_proofs 0.2.0 does with `poly::Evaluator`
// over an `Ast` (U: src/poly/evaluator.rs, src/plonk/prover.rs "Evaluate the h(X) polynomial's constraint system
// expressions"): there every gate polynomial is walked as a tree, one fresh Vec per node.  Here all gate polynomials that
// are evaluated in one launch are hash-consed into ONE DAG, so that
//   * a sub-expression that occurs several times (the curve equation of the ECC gates, (x_p - x_q), running-sum
//     differences, ...) is computed once per point and kept in a per-thread temporary (OP_TEE / OP_PUSH_T), and
//   * consecutive polynomials of one gate that share a factor (normally the selector:  s*e_1, s*e_2, ...) are folded as
//     acc <- acc*y^G + s*(e_1*y^.. + ... + e_m):  m + 1 multiplications instead of 2m.  The factor is also found through
//     nested products ((s*a)*e_1, (s*b)*e_2); the remaining factors are re-multiplied and interned, which for the ECC-style
//     gates exposes many more shared products.  Re-association can also lose sharing, so the caller compiles a tier both
//     ways and keeps the program with fewer multiplications.
// Both rewrites compute the same field element at every point (exact arithmetic), so h(X) and the proof bytes do not change.
// This header has no CUDA dependency: tests/host/evalprog_host_test.cc compiles it with g++ and checks the emitted
// programs against direct evaluation of the expression trees.
#pragma once
#include <algorithm>
#include <cstdint>
#include <map>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#define BZ_EP_CHECK(cond, msg) do { if (!(cond)) throw std::runtime_error(std::string(msg)); } while (0)

namespace bz {

enum : uint32_t { OP_PUSH_P = 0, OP_PUSH_S = 1, OP_PUSH_C = 2, OP_ADD = 3, OP_SUB = 4, OP_MUL = 5, OP_NEG = 6,
                  OP_MULC = 7, OP_ADDC = 8, OP_FOLD = 9, OP_STORE = 10, OP_END = 11, OP_MUL_T_STORE = 12, OP_ACC_MULC = 13,
                  OP_TEE = 14,        // tmp[x] = top of stack (stays on the stack)
                  OP_PUSH_T = 15 };   // push tmp[x]
constexpr int EVAL_STACK = 12;
constexpr int EVAL_TMP = 24;

// postfix token of a gate / lookup expression as it crosses the ABI (bz_circuit IR, SURVEY App. G):
// 0 const(a) 1 advice(a = column, b = rotation) 2 fixed 3 instance 4 neg 5 add 6 mul 7 scale by const(a)
struct Token { uint32_t op, a; int32_t b; };

// Fixed-only sub-expressions of the gate polynomials.  After keygen's selector compression every use of a simple selector is
// q * prod_{i != r} (i - q): up to 8 multiplications per use, all over one fixed column.  A maximal sub-expression built from
// constants and fixed queries at rotation 0 that contains a product is split off as a DERIVED column -- evaluated once per
// proving key on the extended coset -- and the gate polynomial queries it like a fixed column in slot base_slot + j.
// Same value at every point, so h(X) does not change.  `degree` keeps the true degree for the evaluation tiers.
struct DerivedColumn { std::vector<Token> tokens; uint32_t degree; };
inline void split_fixed_subexpressions(const std::vector<Token>& tokens, const std::vector<uint32_t>& gate_off, uint32_t base_slot,
                                       std::vector<DerivedColumn>& derived, std::vector<Token>& qtokens, std::vector<uint32_t>& qgate_off) {
  struct Node { Token t; int x = -1, y = -1; bool fixed_only = false, has_mul = false; uint32_t degree = 0; };
  std::map<std::vector<uint32_t>, uint32_t> index;
  derived.clear(); qtokens.clear(); qgate_off.assign(1, 0u);
  for (size_t g = 0; g + 1 < gate_off.size(); ++g) {
    std::vector<Node> nodes;
    std::vector<int> st;
    for (uint32_t t = gate_off[g]; t < gate_off[g + 1]; ++t) {
      Node n; n.t = tokens[t];
      switch (n.t.op) {
        case 0: n.fixed_only = true; break;
        case 2: n.fixed_only = n.t.b == 0; n.degree = 1; break;
        case 1: case 3: n.degree = 1; break;
        case 4: case 7: { BZ_EP_CHECK(!st.empty(), "bad expression"); n.x = st.back(); st.pop_back(); const Node& c = nodes[n.x]; n.fixed_only = c.fixed_only; n.has_mul = c.has_mul; n.degree = c.degree; break; }
        case 5: case 6: {
          BZ_EP_CHECK(st.size() >= 2, "bad expression");
          n.y = st.back(); st.pop_back(); n.x = st.back(); st.pop_back();
          const Node &a = nodes[n.x], &b = nodes[n.y];
          n.fixed_only = a.fixed_only && b.fixed_only; n.has_mul = a.has_mul || b.has_mul || n.t.op == 6;
          n.degree = n.t.op == 5 ? std::max(a.degree, b.degree) : a.degree + b.degree;
          break;
        }
        default: BZ_EP_CHECK(false, "bad token op");
      }
      nodes.push_back(n);
      st.push_back((int)nodes.size() - 1);
    }
    BZ_EP_CHECK(st.size() == 1, "bad expression");
    struct Walk {
      const std::vector<Node>& nodes; std::map<std::vector<uint32_t>, uint32_t>& index; std::vector<DerivedColumn>& derived; std::vector<Token>& out;
      uint32_t base_slot;
      void flat(int v, std::vector<Token>& o) const { const Node& n = nodes[v]; if (n.x >= 0) flat(n.x, o); if (n.y >= 0) flat(n.y, o); o.push_back(n.t); }
      void emit(int v) {
        const Node& n = nodes[v];
        if (n.fixed_only && n.has_mul && n.degree >= 2) {
          std::vector<Token> sub; flat(v, sub);
          std::vector<uint32_t> key;
          for (const Token& k : sub) { key.push_back(k.op); key.push_back(k.a); key.push_back((uint32_t)k.b); }
          auto it = index.find(key);
          if (it == index.end()) { it = index.emplace(key, (uint32_t)derived.size()).first; derived.push_back(DerivedColumn{sub, n.degree}); }
          out.push_back(Token{2, base_slot + it->second, 0});
          return;
        }
        if (n.x >= 0) emit(n.x);
        if (n.y >= 0) emit(n.y);
        out.push_back(n.t);
      }
    } walk{nodes, index, derived, qtokens, base_slot};
    walk.emit(st.back());
    qgate_off.push_back((uint32_t)qtokens.size());
  }
}

inline uint32_t enc(uint32_t op, uint32_t x = 0, uint32_t y = 0) { return op | (x << 4) | (y << 16); }
inline uint32_t encc(uint32_t op, uint32_t idx) { return op | (idx << 4); }

struct ProgBuilder {
  std::vector<uint32_t> code;
  std::vector<int32_t> rot_table;
  std::map<int, uint32_t> rot_index;
  int scale = 1;
  int depth = 0, max_depth = 0;
  uint32_t rot(int r) {
    auto it = rot_index.find(r);
    if (it != rot_index.end()) return it->second;
    uint32_t idx = (uint32_t)rot_table.size();
    rot_table.push_back(r * scale);
    rot_index[r] = idx;
    BZ_EP_CHECK(idx < 65536, "too many rotations");
    return idx;
  }
  void push() { if (++depth > max_depth) max_depth = depth; }
  void pop(int k = 1) { depth -= k; }
  void pp(uint32_t slot, int r) { BZ_EP_CHECK(slot < 4096, "slot overflow"); code.push_back(enc(OP_PUSH_P, slot, rot(r))); push(); }
  void ps(uint32_t slot, int r) { BZ_EP_CHECK(slot < 4096, "slot overflow"); code.push_back(enc(OP_PUSH_S, slot, rot(r))); push(); }
  void pc(uint32_t c) { code.push_back(encc(OP_PUSH_C, c)); push(); }
  void add() { code.push_back(OP_ADD); pop(); }
  void sub() { code.push_back(OP_SUB); pop(); }
  void mul() { code.push_back(OP_MUL); pop(); }
  void neg() { code.push_back(OP_NEG); }
  void mulc(uint32_t c) { code.push_back(encc(OP_MULC, c)); }
  void addc(uint32_t c) { code.push_back(encc(OP_ADDC, c)); }
  void fold(uint32_t c) { code.push_back(encc(OP_FOLD, c)); pop(); }
  void accmul(uint32_t c) { code.push_back(encc(OP_ACC_MULC, c)); }
  void store(uint32_t k) { code.push_back(encc(OP_STORE, k)); pop(); }
  void tee(uint32_t t) { code.push_back(encc(OP_TEE, t)); }
  void pt(uint32_t t) { code.push_back(encc(OP_PUSH_T, t)); push(); }
};

// The gate polynomials of one launch as a hash-consed DAG.  Usage: add() every polynomial in protocol order (with its
// index e among all expressions of h(X)), plan(), then emit_group() for the groups in order.
struct GateDag {
  struct Node {
    uint32_t op, a; int32_t b; int x, y;      // token op; children (-1: none)
    uint32_t uses = 0;                        // references the emitted program makes to this node
    uint32_t left = 0;                        // references not emitted yet
    int tmp = -1;                             // temporary holding the value, -1: none
    bool has_mul = false;                     // contains a multiplication: worth keeping
    int need = 1;                             // stack slots an emission needs (Sethi-Ullman estimate)
  };
  struct Poly { int root; uint32_t e; };
  struct Group { uint32_t first, count; int factor; std::vector<int> rest; };   // polys [first, first+count); factor -1: plain emission
  std::vector<Node> nodes;
  std::map<std::tuple<uint32_t, uint32_t, int32_t, int, int>, int> index;
  std::vector<Poly> polys;
  std::vector<Group> groups;
  bool sort_rest = false, canon_mul = false;
  bool cse = true, hoist = true, nested = true;      // nested: hoist common factors through nested products as well
  uint32_t advice_slot_of_instance = 0;       // instance column c lives in per-proof slot G + c
  std::vector<int> free_tmp;

  int intern(uint32_t op, uint32_t a, int32_t b, int x, int y) {
    if (canon_mul && op == 6) {                                         // products as sorted left-deep chains of their factors
      std::vector<int> fl = factors(x), fy = factors(y);
      fl.insert(fl.end(), fy.begin(), fy.end());
      std::sort(fl.begin(), fl.end());
      int prod = fl[0];
      for (size_t t = 1; t < fl.size(); ++t) prod = intern_raw(6, 0, 0, prod, fl[t]);
      return prod;
    }
    return intern_raw(op, a, b, x, y);
  }
  int intern_raw(uint32_t op, uint32_t a, int32_t b, int x, int y) {
    if ((op == 5 || op == 6) && x > y) std::swap(x, y);                // commutative
    auto key = std::make_tuple(op, a, b, x, y);
    if (cse) { auto it = index.find(key); if (it != index.end()) return it->second; }
    Node n; n.op = op; n.a = a; n.b = b; n.x = x; n.y = y;
    n.has_mul = op == 6 || op == 7 || (x >= 0 && nodes[x].has_mul) || (y >= 0 && nodes[y].has_mul);
    const int nx = x >= 0 ? nodes[x].need : 0, ny = y >= 0 ? nodes[y].need : 0;
    n.need = op <= 3 ? 1 : y < 0 ? nx : (nx == ny ? nx + 1 : std::max(nx, ny));
    nodes.push_back(n);
    const int id = (int)nodes.size() - 1;
    if (cse) index[key] = id;
    return id;
  }
  int from_tokens(const std::vector<Token>& tokens, uint32_t lo, uint32_t hi) {
    std::vector<int> st;
    for (uint32_t t = lo; t < hi; ++t) {
      const Token& k = tokens[t];
      switch (k.op) {
        case 0: st.push_back(intern(0, k.a, 0, -1, -1)); break;
        case 1: case 2: case 3: st.push_back(intern(k.op, k.a, k.b, -1, -1)); break;
        case 4: BZ_EP_CHECK(!st.empty(), "bad expression"); st.back() = intern(4, 0, 0, st.back(), -1); break;
        case 5: case 6: { BZ_EP_CHECK(st.size() >= 2, "bad expression"); int r = st.back(); st.pop_back(); st.back() = intern(k.op, 0, 0, st.back(), r); break; }
        case 7: BZ_EP_CHECK(!st.empty(), "bad expression"); st.back() = intern(7, k.a, 0, st.back(), -1); break;
        default: BZ_EP_CHECK(false, "bad token op");
      }
    }
    BZ_EP_CHECK(st.size() == 1, "bad expression");
    return st.back();
  }
  void add(const std::vector<Token>& tokens, uint32_t lo, uint32_t hi, uint32_t e) { polys.push_back(Poly{from_tokens(tokens, lo, hi), e}); }

  // the factors of a (nested) product, in emission order
  std::vector<int> factors(int v) const {
    std::vector<int> out, st{v};
    while (!st.empty()) {
      const int c = st.back(); st.pop_back();
      if (nodes[c].op == 6) { st.push_back(nodes[c].y); st.push_back(nodes[c].x); } else out.push_back(c);
    }
    return out;
  }
  // children as the emission references them: a + (-b) is emitted as a b SUB, so it references b, not the negation
  void refs(int v, int& c0, int& c1, bool& is_sub) const {
    const Node& n = nodes[v];
    c0 = n.x; c1 = n.y; is_sub = false;
    if (n.op == 5) {
      if (nodes[n.y].op == 4) { c1 = nodes[n.y].x; is_sub = true; }
      else if (nodes[n.x].op == 4) { c0 = n.y; c1 = nodes[n.x].x; is_sub = true; }
    }
  }
  void count(int v, std::vector<char>& seen) {
    nodes[v].uses++;
    if (seen[v]) return;
    seen[v] = 1;
    int c0, c1; bool s; refs(v, c0, c1, s);
    if (c0 >= 0) count(c0, seen);
    if (c1 >= 0) count(c1, seen);
  }
  void plan() {
    groups.clear();
    for (uint32_t i = 0; i < polys.size();) {
      Group g{i, 1, -1, {}};
      const Node r = nodes[polys[i].root];           // (a copy: interning below may grow `nodes`)
      if (hoist && r.op == 6) {
        std::vector<int> cand = {r.x, r.y};
        uint32_t j = i + 1;
        for (; j < polys.size(); ++j) {     // (a common factor is all it takes: the polynomials need not belong to one gate)
          const Node& q = nodes[polys[j].root];
          if (q.op != 6) break;
          std::vector<int> keep;
          for (int c : cand) if (c == q.x || c == q.y) keep.push_back(c);
          if (keep.empty()) break;
          cand = keep;
        }
        if (j - i >= 2) {
          g.count = j - i; g.factor = cand[0];
          for (uint32_t p = i; p < j; ++p) { const Node& q = nodes[polys[p].root]; g.rest.push_back(q.x == g.factor ? q.y : q.x); }
        }
      }
      if (hoist && cse && nested && g.factor < 0 && r.op == 6) {
        // no common DIRECT child: look through nested products -- (s*a)*e_1, (s*b)*e_2 share s.  One common factor (a
        // leaf if there is one: the selector) is pulled out, the other factors of every polynomial are re-multiplied
        // (interned, so they are still shared with the rest of the DAG).
        std::vector<int> cand = factors(polys[i].root);
        uint32_t j = i + 1;
        for (; j < polys.size() && nodes[polys[j].root].op == 6; ++j) {
          const std::vector<int> fj = factors(polys[j].root);
          std::vector<int> keep;
          for (int c : cand) if (std::find(fj.begin(), fj.end(), c) != fj.end() && std::find(keep.begin(), keep.end(), c) == keep.end()) keep.push_back(c);
          if (keep.empty()) break;
          cand = keep;
        }
        if (j - i >= 2) {
          int f = cand[0];
          for (int c : cand) if (nodes[c].op <= 3) { f = c; break; }
          std::vector<int> rest;
          bool ok = true;
          for (uint32_t p = i; p < j && ok; ++p) {
            std::vector<int> fp = factors(polys[p].root);
            fp.erase(std::find(fp.begin(), fp.end(), f));
            if (fp.empty()) { ok = false; break; }
            if (sort_rest) std::sort(fp.begin(), fp.end());          // same multiset of factors -> same chain of products
            int prod = fp[0];
            for (size_t t = 1; t < fp.size(); ++t) prod = intern(6, 0, 0, prod, fp[t]);
            rest.push_back(prod);
          }
          if (ok) { g.count = j - i; g.factor = f; g.rest = rest; }
        }
      }
      groups.push_back(g);
      i += g.count;
    }
    std::vector<char> seen(nodes.size(), 0);
    for (auto& n : nodes) { n.uses = 0; n.tmp = -1; }
    for (const Group& g : groups) {
      if (g.factor < 0) count(polys[g.first].root, seen);
      else { for (int r : g.rest) count(r, seen); count(g.factor, seen); }
    }
    for (auto& n : nodes) n.left = n.uses;
    free_tmp.clear();
    for (int t = EVAL_TMP - 1; t >= 0; --t) free_tmp.push_back(t);
  }

  void emit(ProgBuilder& pb, int v) {
    Node& n = nodes[v];
    if (n.left) --n.left;
    if (n.tmp >= 0) {
      pb.pt((uint32_t)n.tmp);
      if (!n.left) { free_tmp.push_back(n.tmp); n.tmp = -1; }
      return;
    }
    switch (n.op) {
      case 0: pb.pc(n.a); break;
      case 1: pb.pp(n.a, n.b); break;
      case 2: pb.ps(n.a, n.b); break;
      case 3: pb.pp(advice_slot_of_instance + n.a, n.b); break;
      case 4: emit(pb, n.x); pb.neg(); break;
      case 7: emit(pb, n.x); pb.mulc(n.a); break;
      case 5: case 6: {
        int c0, c1; bool is_sub; refs(v, c0, c1, is_sub);
        if (is_sub) { emit(pb, c0); emit(pb, c1); pb.sub(); }
        else {
          if (nodes[c1].need > nodes[c0].need) std::swap(c0, c1);        // deeper operand first: shallower stack
          emit(pb, c0); emit(pb, c1);
          if (n.op == 5) pb.add(); else pb.mul();
        }
        break;
      }
      default: BZ_EP_CHECK(false, "bad node");
    }
    Node& m = nodes[v];                                                    // (no reallocation happens during emission)
    if (m.left && m.has_mul && !free_tmp.empty()) { m.tmp = free_tmp.back(); free_tmp.pop_back(); pb.tee((uint32_t)m.tmp); }
  }
  // value of group g on the stack is folded into the accumulator:  acc <- acc * y^(gap_total) + (terms of the group).
  // `yp(d)` = constant index of y^d; `prev_e` = index of the last expression folded before this group (-1: none).
  template <class YP> void emit_group(ProgBuilder& pb, const Group& g, int prev_e, YP yp) {
    const uint32_t e0 = polys[g.first].e, e_last = polys[g.first + g.count - 1].e;
    const uint32_t gap0 = prev_e < 0 ? 1u : e0 - (uint32_t)prev_e;
    if (g.factor < 0) { emit(pb, polys[g.first].root); pb.fold(yp(gap0)); return; }
    emit(pb, g.rest[0]);
    for (uint32_t i = 1; i < g.count; ++i) {
      pb.mulc(yp(polys[g.first + i].e - polys[g.first + i - 1].e));
      emit(pb, g.rest[i]);
      pb.add();
    }
    emit(pb, g.factor);
    pb.mul();
    pb.fold(yp(gap0 + (e_last - e0)));
  }
};

}  // namespace bz
