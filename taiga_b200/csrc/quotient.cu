// Row-parallel evaluation of the PLONKish gate / lookup / permutation constraint polynomial (the quotient numerator)
// and the grand-product helpers, for sm_100a.
//
// Replaces the h(X) construction of halo2_proofs `plonk::create_proof` + `vanishing::Argument::construct`,
// `permutation::Argument::commit` and `lookup::Argument::commit_product` (EXT; SURVEY.md §8a rows H3-H5, App. A.1
// step 8, App. E.3/E.6).  The extended domain is never materialised per column: for each of the R = 2^(ext_k-k)
// sub-cosets zeta*w_ext^k1*<w> the per-proof columns are NTT'd onto that sub-coset (n rows), every constraint is
// evaluated one thread per row, and the result is scaled by the (constant on the sub-coset) 1/(X^n - 1).
//
// Algorithmic bytes per sub-coset row: 32*(C+1), C = distinct column-cosets read (SURVEY §8d).
#include <map>
#define TB_NOINLINE_MUL 0  // loop-structured kernels: small code, keep the multiply inline
#include "common.cuh"
#include "prover_kernels.cuh"

namespace tb {

// ---------------------------------------------------------------- expression compiler (host)
namespace {
// A constraint list is compiled as a sequence of ITEMS.  Consecutive constraints of one gate usually share their selector
// factor, root_j = S * X_j: since  acc <- acc * y + S * X_j  over such a run equals  acc * y^len + S * (Horner of the X_j in y),
// the run is evaluated as a group with len + 1 multiplications instead of 2 * len (the result is the same field element, so
// the proof bytes do not change).  A program may hold any subset of the constraints: every fold multiplies by y^(gap to the
// previous constraint of the program), read from a per-proof table of powers of y.
struct Item { bool group; uint32_t root; uint32_t S; std::vector<uint32_t> xs; std::vector<uint32_t> pos; };   // pos: constraint index of every element

std::vector<Item> build_items(const tb_cs_desc* cs, const std::vector<uint32_t>& idx) {
  std::vector<Item> items;
  auto factors = [&](uint32_t r, uint32_t* f) -> int { const tb_expr_node& nd = cs->nodes[r]; if (nd.op != TB_EX_MUL) return 0; f[0] = nd.a; f[1] = nd.b; return nd.a == nd.b ? 1 : 2; };
  size_t i = 0;
  while (i < idx.size()) {
    uint32_t f[2]; int nf = factors(cs->constraint_roots[idx[i]], f);
    size_t j = i + 1;
    while (nf && j < idx.size()) {
      uint32_t g[2]; int ng = factors(cs->constraint_roots[idx[j]], g);
      uint32_t keep[2]; int nk = 0;
      for (int x = 0; x < nf; ++x) for (int y = 0; y < ng; ++y) if (f[x] == g[y]) { keep[nk++] = f[x]; break; }
      if (!nk) break;
      nf = nk; f[0] = keep[0]; if (nk > 1) f[1] = keep[1];
      ++j;
    }
    Item it; it.S = 0; it.root = 0;
    if (j - i >= 2) {
      it.group = true; it.S = f[0];
      for (size_t q = i; q < j; ++q) { const tb_expr_node& nd = cs->nodes[cs->constraint_roots[idx[q]]]; it.xs.push_back(nd.a == it.S ? nd.b : nd.a); it.pos.push_back(idx[q]); }
    } else {
      it.group = false; it.root = cs->constraint_roots[idx[i]]; it.pos.push_back(idx[i]); j = i + 1;
    }
    items.push_back(it);
    i = j;
  }
  return items;
}

struct Compiler {
  const tb_cs_desc* cs;
  std::vector<int> refc;          // remaining uses per node
  std::vector<int> reg_of;        // register holding node value (-1 = none)
  std::vector<int> free_regs; int next_reg = 0, max_regs = 0;
  std::vector<QInstr> code;
  struct Opnd { int kind; uint32_t v; int node; };

  explicit Compiler(const tb_cs_desc* c) : cs(c), refc(c->num_nodes, 0), reg_of(c->num_nodes, -1) {}
  void count(uint32_t node, std::vector<char>& seen) {
    refc[node]++;
    if (seen[node]) return;
    seen[node] = 1;
    const tb_expr_node& nd = cs->nodes[node];
    if (nd.op == TB_EX_NEG || nd.op == TB_EX_SCALE) count(nd.a, seen);
    else if (nd.op == TB_EX_ADD || nd.op == TB_EX_MUL) { count(nd.a, seen); count(nd.b, seen); }
  }
  int alloc() {
    int r;
    if (!free_regs.empty()) { r = free_regs.back(); free_regs.pop_back(); } else r = next_reg++;
    if (next_reg > max_regs) max_regs = next_reg;
    return r;
  }
  void release(const Opnd& o) {
    if (o.node < 0) return;
    if (--refc[o.node] == 0 && reg_of[o.node] >= 0) { free_regs.push_back(reg_of[o.node]); reg_of[o.node] = -1; }
  }
  static uint32_t leaf(const tb_query& q) {   // column << 8 | (rotation + 128): the kernel needs no query table
    TB_REQUIRE(q.rotation >= -128 && q.rotation < 128 && q.column < (1u << 24), "query rotation / column out of the encodable range");
    return (q.column << 8) | (uint32_t)(q.rotation + 128);
  }
  bool is_two(uint32_t const_index) const {
    const uint8_t* c = cs->constants + 32 * (size_t)const_index;
    if (c[0] != 2) return false;
    for (int i = 1; i < 32; ++i) if (c[i]) return false;
    return true;
  }
  Opnd emit(uint32_t node) {
    const tb_expr_node& nd = cs->nodes[node];
    switch (nd.op) {
      case TB_EX_CONST: return {K_CONST, nd.a, (int)node};
      case TB_EX_ADVICE: return {K_ADV, leaf(cs->advice_queries[nd.a]), (int)node};
      case TB_EX_FIXED: return {K_FIX, leaf(cs->fixed_queries[nd.a]), (int)node};
      case TB_EX_INSTANCE: return {K_INST, leaf(cs->instance_queries[nd.a]), (int)node};
      default: break;
    }
    if (reg_of[node] >= 0) return {K_REG, (uint32_t)reg_of[node], (int)node};
    int op; Opnd oa, ob; bool binary = true;
    if (nd.op == TB_EX_NEG) { oa = emit(nd.a); ob = {K_CONST, 0, -1}; op = Q_NEG; binary = false; }
    else if (nd.op == TB_EX_SCALE) {
      oa = emit(nd.a);
      if (is_two(nd.b)) { ob = oa; ob.node = -1; op = Q_ADD; }   // 2 x = x + x: an addition instead of a multiplication
      else { ob = {K_CONST, nd.b, -1}; op = Q_MUL; }
    }
    else if (nd.op == TB_EX_MUL) { oa = emit(nd.a); ob = emit(nd.b); op = Q_MUL; }
    else {  // ADD, with a - b peephole when the negation is used only here
      const tb_expr_node& na = cs->nodes[nd.a]; const tb_expr_node& nb = cs->nodes[nd.b];
      if (nb.op == TB_EX_NEG && refc[nd.b] == 1 && reg_of[nd.b] < 0) {
        oa = emit(nd.a); refc[nd.b]--; ob = emit(nb.a); op = Q_SUB;
      } else if (na.op == TB_EX_NEG && refc[nd.a] == 1 && reg_of[nd.a] < 0) {
        oa = emit(nd.b); refc[nd.a]--; ob = emit(na.a); op = Q_SUB;
      } else { oa = emit(nd.a); ob = emit(nd.b); op = Q_ADD; }
    }
    // operands of leaves carry node ids only for refcounting; leaves hold no register
    release(oa); if (binary) release(ob);
    int r = alloc();
    code.push_back(q_make(op, r, oa.kind, oa.v, ob.kind, ob.v));
    reg_of[node] = r;
    return {K_REG, (uint32_t)r, (int)node};
  }
  // the constraints `idx` (ascending) folded with y; returns the index of the last one
  int compile_constraints(const std::vector<uint32_t>& idx) {
    std::vector<Item> items = build_items(cs, idx);
    std::vector<char> seen(cs->num_nodes, 0);
    for (auto& it : items) {
      if (!it.group) count(it.root, seen);
      else { count(it.S, seen); for (uint32_t x : it.xs) count(x, seen); }
    }
    int prev = -1;
    for (auto& it : items) {
      if (!it.group) {
        Opnd o = emit(it.root);
        code.push_back(q_make(Q_FOLD_Y, 0, o.kind, o.v, K_CONST, prev < 0 ? 1u : (uint32_t)((int)it.pos[0] - prev))); release(o);
        prev = (int)it.pos[0];
        continue;
      }
      for (size_t j = 0; j < it.xs.size(); ++j) {
        Opnd o = emit(it.xs[j]);
        code.push_back(q_make(j == 0 ? Q_GBEGIN : Q_GFOLD, 0, o.kind, o.v, K_CONST, j == 0 ? 0u : it.pos[j] - it.pos[j - 1])); release(o);
      }
      Opnd os = emit(it.S);
      code.push_back(q_make(Q_GEND, 0, os.kind, os.v, K_CONST, prev < 0 ? 1u : (uint32_t)((int)it.pos.back() - prev))); release(os);
      prev = (int)it.pos.back();
    }
    return prev;
  }
};
void finish_program(Compiler& c, QProgram* out) {
  out->host = c.code; out->nregs = c.max_regs < 1 ? 1 : c.max_regs; out->ninstr = (int)c.code.size();
  TB_REQUIRE(out->nregs <= 48, "constraint expressions need too many live temporaries");
  if (out->dev) cudaFree(out->dev);
  out->dev = nullptr;
  if (out->ninstr) {
    TB_CUDA(cudaMalloc(&out->dev, out->ninstr * sizeof(QInstr)));
    TB_CUDA(cudaMemcpy(out->dev, out->host.data(), out->ninstr * sizeof(QInstr), cudaMemcpyHostToDevice));
  }
}
}  // namespace

std::vector<int> q_constraint_degrees(const tb_cs_desc* cs) {
  std::vector<int> deg(cs->num_nodes, -1);
  for (uint32_t i = 0; i < cs->num_nodes; ++i) {   // nodes are in topological order (checked at circuit load)
    const tb_expr_node& nd = cs->nodes[i];
    switch (nd.op) {
      case TB_EX_CONST: deg[i] = 0; break;
      case TB_EX_ADVICE: case TB_EX_FIXED: case TB_EX_INSTANCE: deg[i] = 1; break;
      case TB_EX_NEG: case TB_EX_SCALE: deg[i] = deg[nd.a]; break;
      case TB_EX_ADD: deg[i] = deg[nd.a] > deg[nd.b] ? deg[nd.a] : deg[nd.b]; break;
      default: deg[i] = deg[nd.a] + deg[nd.b]; break;
    }
  }
  std::vector<int> out(cs->num_constraints);
  for (uint32_t j = 0; j < cs->num_constraints; ++j) out[j] = deg[cs->constraint_roots[j]];
  return out;
}

void q_compile_gates_split(const tb_cs_desc* cs, const std::vector<uint32_t>& subset, int parts, std::vector<QProgram>* out) {
  // cost of a root = instructions of its stand-alone program; contiguous (within the subset) groups with roughly equal cumulative cost
  std::vector<size_t> cost(subset.size());
  size_t total = 0;
  for (size_t i = 0; i < subset.size(); ++i) {
    Compiler c(cs); std::vector<char> seen(cs->num_nodes, 0);
    c.count(cs->constraint_roots[subset[i]], seen);
    Compiler::Opnd o = c.emit(cs->constraint_roots[subset[i]]); (void)o;
    cost[i] = c.code.size() + 1; total += cost[i];
  }
  if (parts > (int)subset.size()) parts = subset.empty() ? 1 : (int)subset.size();
  out->clear();
  size_t r0 = 0, acc = 0;
  for (int p = 0; p < parts; ++p) {
    size_t r1 = r0;
    const size_t target = total * (p + 1) / parts;
    while (r1 < subset.size() && (acc < target || p == parts - 1)) acc += cost[r1++];
    if (p == parts - 1) r1 = subset.size();
    Compiler c(cs);
    const int last = c.compile_constraints(std::vector<uint32_t>(subset.begin() + r0, subset.begin() + r1));
    out->emplace_back();
    finish_program(c, &out->back());
    out->back().last = last;
    r0 = r1;
  }
}

void q_compile_lookups(const tb_cs_desc* cs, QProgram* out) {
  Compiler c(cs);
  std::vector<char> seen(cs->num_nodes, 0);
  for (uint32_t l = 0; l < cs->num_lookups; ++l)
    for (uint32_t e = 0; e < cs->lookups[l].num_exprs; ++e) { c.count(cs->lookups[l].input_roots[e], seen); c.count(cs->lookups[l].table_roots[e], seen); }
  for (uint32_t l = 0; l < cs->num_lookups; ++l) {
    c.code.push_back(q_make(Q_LK_BEGIN, 0, K_CONST, 0, K_CONST, 0));
    for (uint32_t e = 0; e < cs->lookups[l].num_exprs; ++e) {
      Compiler::Opnd o = c.emit(cs->lookups[l].input_roots[e]);
      c.code.push_back(q_make(Q_FOLD_A, 0, o.kind, o.v, K_CONST, 0)); c.release(o);
    }
    for (uint32_t e = 0; e < cs->lookups[l].num_exprs; ++e) {
      Compiler::Opnd o = c.emit(cs->lookups[l].table_roots[e]);
      c.code.push_back(q_make(Q_FOLD_S, 0, o.kind, o.v, K_CONST, 0)); c.release(o);
    }
    c.code.push_back(q_make(Q_LK_STORE, 0, K_CONST, l, K_CONST, 0));
  }
  finish_program(c, out);
}

void q_compile_check_gates(const tb_cs_desc* cs, QProgram* out) {
  Compiler c(cs);
  std::vector<char> seen(cs->num_nodes, 0);
  for (uint32_t j = 0; j < cs->num_constraints; ++j) c.count(cs->constraint_roots[j], seen);
  for (uint32_t j = 0; j < cs->num_constraints; ++j) {
    Compiler::Opnd o = c.emit(cs->constraint_roots[j]);
    c.code.push_back(q_make(Q_CK_TEST, 0, o.kind, o.v, K_CONST, j)); c.release(o);
  }
  finish_program(c, out);
}

void q_compile_check_lookups(const tb_cs_desc* cs, bool tables, QProgram* out) {
  Compiler c(cs);
  std::vector<char> seen(cs->num_nodes, 0);
  auto root = [&](uint32_t l, uint32_t e) { return tables ? cs->lookups[l].table_roots[e] : cs->lookups[l].input_roots[e]; };
  for (uint32_t l = 0; l < cs->num_lookups; ++l)
    for (uint32_t e = 0; e < cs->lookups[l].num_exprs; ++e) c.count(root(l, e), seen);
  uint32_t slot = 0;
  for (uint32_t l = 0; l < cs->num_lookups; ++l)
    for (uint32_t e = 0; e < cs->lookups[l].num_exprs; ++e) {
      Compiler::Opnd o = c.emit(root(l, e));
      QInstr in = q_make(Q_CK_STORE, 0, o.kind, o.v, K_CONST, slot++); in.pad = l;
      c.code.push_back(in); c.release(o);
    }
  finish_program(c, out);
}

// ---------------------------------------------------------------- interpreter kernel
// One thread per (row, constraint part).  ALL values, including the running folds, live in the shared-memory register file
// [nregs + 2][T] x 32 B (slot nregs = the y / theta fold accumulator, slot nregs + 1 = the group / table fold): the loop carries
// no 256-bit value in registers, which kept the compiler from shuffling 16-24 registers on every interpreted instruction
// (ncu source view of the previous version: 30 % of the executed instructions were MOV / CS2R / SEL / BRA).
__global__ void __launch_bounds__(128) q_interp_kernel(QPartList pl, int nregs, QData d) {
  const uint4* __restrict__ prog = reinterpret_cast<const uint4*>(pl.prog[blockIdx.z]);
  const int ninstr = pl.ninstr[blockIdx.z];
  extern __shared__ uint4 q_smem[];
  const int T = blockDim.x, tid = threadIdx.x;
  uint4* rlo = q_smem + tid;
  uint4* rhi = q_smem + (size_t)(nregs + 2) * T + tid;
  const int row = blockIdx.x * T + tid, b = blockIdx.y;
  if (row >= d.n) return;
  const int nm = d.n - 1, ACC = nregs * T, G = (nregs + 1) * T;
  const Fp* adv = d.adv + (long long)b * d.adv_pstride;
  const Fp* inst = d.inst + (long long)b * d.inst_pstride;
  const Fp* chal = d.chal + (long long)b * d.chal_stride;

  auto lds = [&](int idx) -> Fp { uint4 x = rlo[idx], z = rhi[idx]; Fp r;
    r.l[0] = x.x; r.l[1] = x.y; r.l[2] = x.z; r.l[3] = x.w; r.l[4] = z.x; r.l[5] = z.y; r.l[6] = z.z; r.l[7] = z.w; return r; };
  auto sts = [&](int idx, const Fp& r) {
    rlo[idx] = make_uint4(r.l[0], r.l[1], r.l[2], r.l[3]); rhi[idx] = make_uint4(r.l[4], r.l[5], r.l[6], r.l[7]); };
  auto fetch = [&](int kind, uint32_t v) -> Fp {
    if (kind == K_REG) return lds((int)v * T);
    const Fp* p;
    if (kind == K_CONST) p = d.consts + v;
    else {
      const int rot = (int)(v & 255u) - 128; const size_t col = v >> 8;
      const Fp* base = kind == K_ADV ? adv + col * d.n : kind == K_INST ? inst + col * d.n : d.fix + (col * d.R + d.k1) * d.n;
      p = base + ((row + rot + d.n) & nm);
    }
    return ldg_fe(p);
  };
  sts(ACC, Fp::zero()); sts(G, Fp::zero());
  uint4 in = __ldg(prog);
  for (int pc = 0; pc < ninstr; ++pc) {
    const uint32_t w0 = in.x, ia = in.y, ib = in.z;
    if (pc + 1 < ninstr) in = __ldg(prog + pc + 1);   // next instruction word in flight while this one executes
    const int op = w0 & 0xff, ak = (w0 >> 16) & 0xff, bk = w0 >> 24;
    int dst = ((w0 >> 8) & 0xff) * T;
    Fp r;
    switch (op) {
      case Q_MOV: r = fetch(ak, ia); break;
      case Q_NEG: r = fetch(ak, ia).neg(); break;
      case Q_ADD: r = fetch(ak, ia) + fetch(bk, ib); break;
      case Q_SUB: r = fetch(ak, ia) - fetch(bk, ib); break;
      case Q_MUL: r = fetch(ak, ia) * fetch(bk, ib); break;
      case Q_FOLD_Y: r = lds(ACC) * chal[d.ytab_slot + ib] + fetch(ak, ia); dst = ACC; break;   // acc = acc * y^gap + e
      case Q_FOLD_A: r = lds(ACC) * chal[d.theta_slot] + fetch(ak, ia); dst = ACC; break;
      case Q_FOLD_S: r = lds(G) * chal[d.theta_slot] + fetch(ak, ia); dst = G; break;
      case Q_GFOLD: r = lds(G) * chal[d.ytab_slot + ib] + fetch(ak, ia); dst = G; break;
      case Q_GBEGIN: r = fetch(ak, ia); dst = G; break;
      case Q_GEND: r = lds(ACC) * chal[d.ytab_slot + ib] + fetch(ak, ia) * lds(G); dst = ACC; break;   // acc = acc * y^gap + S * g
      case Q_LK_BEGIN: r = Fp::zero(); sts(G, r); dst = ACC; break;
      case Q_LK_STORE: {
        const size_t o = (size_t)b * d.lk_pstride + (size_t)ia * d.n + row;
        st_fe(d.lkA + o, lds(ACC)); st_fe(d.lkS + o, lds(G)); continue; }
      default: continue;
    }
    sts(dst, r);
  }
  if (d.gate_out) st_fe(d.gate_out + (long long)blockIdx.z * pl.part_stride + (long long)b * d.gate_pstride + row, lds(ACC));
}

static double program_muls(const QProgram& p) {   // field multiplications per evaluated row
  double m = 0;
  for (const QInstr& in : p.host) { const int op = in.w0 & 0xff; m += (op == Q_MUL || op == Q_FOLD_Y || op == Q_FOLD_A || op == Q_FOLD_S || op == Q_GFOLD) ? 1.0 : op == Q_GEND ? 2.0 : 0.0; }
  return m;
}
static void q_launch(Ctx* c, const QPartList& pl, int nregs, const QData& d, int B) {
  ProfScope prof_scope(c, PC_QUOT_GATES);
  c->opt_in_smem(q_interp_kernel, 96 * 1024);
  // T threads evaluate T rows; the register file [nregs + 2][T] x 32 B lives in shared memory
  int T = (96 * 1024) / ((nregs + 2) * 32);
  const int tmax = tb_tune("TB_Q_THREADS", 128);
  T = T >= tmax ? tmax : (T / 16) * 16;
  TB_REQUIRE(T >= 16 && T <= 128, "constraint program register file does not fit shared memory");
  while (T > d.n && T > 1) T >>= 1;
  const size_t smem = (size_t)(nregs + 2) * T * 32;
  q_interp_kernel<<<dim3((d.n + T - 1) / T, B, pl.nparts), T, smem, c->stream>>>(pl, nregs, d);
  TB_LAUNCH_CHECK(); c->launches++;
}
void q_run(Ctx* c, const QProgram& prog, const QData& d, int B) {
  QPartList pl; memset(&pl, 0, sizeof(pl));
  pl.prog[0] = prog.dev; pl.ninstr[0] = prog.ninstr; pl.nparts = 1; pl.part_stride = 0;
  c->work[PC_QUOT_GATES] += program_muls(prog) * (double)d.n * B;
  q_launch(c, pl, prog.nregs, d, B);
}
void q_run_parts(Ctx* c, const std::vector<QProgram>& progs, QData d, long long part_stride, int B) {
  QPartList pl; memset(&pl, 0, sizeof(pl));
  int nregs = 1;
  pl.nparts = (int)progs.size(); pl.part_stride = part_stride;
  for (int p = 0; p < pl.nparts; ++p) c->work[PC_QUOT_GATES] += program_muls(progs[p]) * (double)d.n * B;
  for (int p = 0; p < pl.nparts; ++p) { pl.prog[p] = progs[p].dev; pl.ninstr[p] = progs[p].ninstr; nregs = nregs > progs[p].nregs ? nregs : progs[p].nregs; }
  q_launch(c, pl, nregs, d, B);
}

}  // namespace tb
