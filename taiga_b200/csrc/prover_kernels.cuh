// Declarations for lookup.cu and quotient.cu (kernel drivers used by prover.cu).
#pragma once
#include "prover.cuh"

namespace tb {

// ---------------------------------------------------------------- lookup.cu
void lookup_keys(Ctx* c, Fp* keys, const Fp* vals, int n, int usable, int arrays);      // Montgomery -> canonical sort keys (+ sentinels)
void sort_keys(Ctx* c, Fp* keys, int n, int arrays);                                      // ascending, canonical-integer order
void lookup_arrange(Ctx* c, const Fp* sortedA, const Fp* sortedT, Fp* scratch, Fp* S, int n, int usable, int arrays, uint32_t* d_err);

// ---------------------------------------------------------------- quotient.cu
// Row-parallel expression interpreter (SURVEY.md App. E.6).  Temporaries live in a shared-memory register file laid
// out [reg][thread] as two 16-byte halves; leaves (column queries, constants) are read straight from global memory.
// Q_CK_TEST / Q_CK_STORE end the constraint-check programs (check.cu): test the operand as constraint `b`, or store it as lookup
// expression `b` of lookup `pad`.
enum QOp { Q_MOV = 0, Q_NEG, Q_ADD, Q_SUB, Q_MUL, Q_FOLD_Y, Q_LK_BEGIN, Q_FOLD_A, Q_FOLD_S, Q_LK_STORE, Q_GBEGIN, Q_GFOLD, Q_GEND, Q_CK_TEST, Q_CK_STORE };
enum QKind { K_REG = 0, K_ADV, K_FIX, K_INST, K_CONST };
struct alignas(16) QInstr { uint32_t w0; uint32_t a, b, pad; };  // w0 = op | dst << 8 | akind << 16 | bkind << 24 (one 128-bit load)
inline QInstr q_make(int op, int dst, int ak, uint32_t a, int bk, uint32_t b) { QInstr i; i.w0 = op | (dst << 8) | (ak << 16) | (bk << 24); i.a = a; i.b = b; i.pad = 0; return i; }

struct QProgram {           // compiled once per circuit (host), resident on the device
  std::vector<QInstr> host; int nregs = 0;
  QInstr* dev = nullptr; int ninstr = 0;
  int last = -1;            // index of the last constraint the program folds: its result is sum_j y^(last - j) e_j over its constraints
};
// Flattens the expression DAG reachable from `roots` into a register-allocated instruction list.
// mode 0: gate constraints folded with y (Q_FOLD_Y per root);  mode 1: lookup compression (theta folds + stores)
// The (sorted) constraint subset `subset` split into `parts` groups of similar cost, one program each (row-parallel AND
// constraint-parallel evaluation).  Folds are gap-aware: program p yields S_p = sum_{j in p} y^(last_p - j) e_j, so any
// set of programs combines as sum_p y^(J - 1 - last_p) S_p, whatever subset of the J constraints each one holds.
constexpr int Q_MAX_PARTS = 16;
void q_compile_gates_split(const tb_cs_desc* cs, const std::vector<uint32_t>& subset, int parts, std::vector<QProgram>* out);
// polynomial degree of every constraint (a column query counts 1): decides which sub-cosets a constraint must be evaluated on
std::vector<int> q_constraint_degrees(const tb_cs_desc* cs);
struct QPartList { const QInstr* prog[Q_MAX_PARTS]; int ninstr[Q_MAX_PARTS]; int nparts; long long part_stride; };
void q_compile_lookups(const tb_cs_desc* cs, QProgram* out);
// constraint-check programs: every constraint root followed by Q_CK_TEST j; or every lookup input (tables = false) / table
// (tables = true) expression followed by Q_CK_STORE, expressions numbered lookup-major across all lookups
void q_compile_check_gates(const tb_cs_desc* cs, QProgram* out);
void q_compile_check_lookups(const tb_cs_desc* cs, bool tables, QProgram* out);

struct QData {
  const Fp* adv; long long adv_pstride;     // [B][num_advice][n]
  const Fp* inst; long long inst_pstride;   // [B][num_instance][n]
  const Fp* fix; int R; int k1;             // [num_fixed][R][n]  (R = 1: Lagrange values)
  const Fp* consts;                         // Montgomery
  const Fp* chal; long long chal_stride; int y_slot, theta_slot, ytab_slot;   // chal[ytab_slot + i] = y^i (0 <= i <= constraints + permutation / lookup terms)
  Fp* gate_out; long long gate_pstride;     // [B][n]
  Fp* lkA; Fp* lkS; long long lk_pstride;   // [B][L][n]
  int n;
};
void q_run(Ctx* c, const QProgram& prog, const QData& d, int B);
void q_run_parts(Ctx* c, const std::vector<QProgram>& progs, QData d, long long part_stride, int B);

// permutation + lookup terms of the quotient, folded onto the gate accumulator, times 1/(X^n - 1) (constant per sub-coset)
struct QFinish {
  const Fp* gate;          // [nparts][B][n] partial Horner sums of the gate constraints
  int nparts; long long gate_part_stride; int ytab_slot; int gexp[Q_MAX_PARTS];   // numerator += chal[ytab_slot + gexp[p]] * gate[p]
  const Fp* rlo; long long rlo_pstride;   // remainder of the low-degree numerator modulo X^n - 1 on this sub-coset (or null): added before the division
  const Fp* adv; long long adv_pstride; const Fp* inst; long long inst_pstride;   // sub-coset evaluations
  const Fp* fix; const Fp* sig; int R; int k1;      // [nf][R][n], [P][R][n]
  const Fp* l0; const Fp* l_last; const Fp* l_blind; // [R][n]
  const Fp* pz; long long pz_pstride;                // [B][nsets][n]
  const Fp* lz; const Fp* lpin; const Fp* lptab; long long lk_pstride;  // per-proof stride of the three (merged coset buffer)
  long long lkc_pstride;                             // per-proof stride of lkA / lkS
  const Fp* lkA; const Fp* lkS;                      // [B][L][n] compressed input / table on this sub-coset
  const int2* perm_cols; int P; int chunk; int nsets; int L; int bf;
  const Fp* chal; long long chal_stride; int y_slot, beta_slot, gamma_slot;
  Fp delta; Fp zeta; Fp t_inv;                       // DELTA, ZETA, 1/((zeta w^k1)^n - 1)
  Fp delta_c0[16];                                   // DELTA^(s*chunk) per permutation set
  TwiddleTables<Fp> tw;                              // forward tables
  int ext_k; int k;
  Fp* out; long long out_pstride;                    // H[b][k1][row]  (out + b*out_pstride + k1*n + row)
  int n;
};
void q_finish(Ctx* c, const QFinish& f, int B);

// extended_to_coeff step B: size-R inverse transform across sub-cosets + zeta^-i, keeps `pieces` * n coefficients
void h_cross(Ctx* c, const Fp* V, long long v_pstride, Fp* hcoef, long long h_pstride, int n, int R, int pieces, const Fp* d_wr_inv /* R * wr_step */,
             int wr_step, Fp r_inv, Fp zeta_inv, int B);
// low-degree numerator (SURVEY 8a H3, evaluated on every second sub-coset only):
//   out[b][k][row] = sum_p chal[b][ytab_slot + gexp[p]] * gate[p][b][row]      (combination of the low programs on one sub-coset)
void q_combine(Ctx* c, const Fp* gate, int nparts, long long part_stride, const int* gexp, const Fp* chal, long long chal_stride, int ytab_slot, Fp* out, long long out_pstride,
               int n, int B);
//   c[b][j][i], j < m: coefficients of H_lo.  r[b][i] = sum_j c[b][j][i] (= H_lo mod X^n - 1);  q[b][j][i] = sum_{t > j} c[b][t][i], j < m - 1 (= H_lo div X^n - 1)
void q_lo_split(Ctx* c, const Fp* coef, long long c_pstride, int m, Fp* r, long long r_pstride, Fp* q, long long q_pstride, int n, int B);
// h[b][j][i] += q[b][j][i], j < m
void q_add_blocks(Ctx* c, Fp* h, long long h_pstride, const Fp* q, long long q_pstride, int m, int n, int B);

// grand products (permutation / lookup)
struct PermFrac {
  const Fp* adv; long long adv_pstride; const Fp* inst; long long inst_pstride; const Fp* fix;   // Lagrange values
  const Fp* sig;                     // [P][n] sigma values
  const int2* perm_cols; int P; int chunk; int nsets;
  const Fp* chal; long long chal_stride; int beta_slot, gamma_slot;
  Fp delta, omega;
  Fp delta_c0[16];
  TwiddleTables<Fp> tw;
  Fp* num; Fp* den; long long pstride;   // [B][nsets][n]
  int n; int k;
};
void perm_fractions(Ctx* c, const PermFrac& p, int B);
// a[i] *= b[i]
void vec_mul(Ctx* c, Fp* a, const Fp* b, size_t count);
// z[b][s][i] *= carry, where carry_s = prod_{s' < s} zlocal[b][s'][u]; applied in place (u = last usable row)
void perm_chain(Ctx* c, Fp* z, long long pstride, int nsets, int n, int u, int B);
// lookup: den = (A'+beta)(S'+gamma), num = (A+beta)(S+gamma)
void lookup_fractions(Ctx* c, const Fp* A, const Fp* S, const Fp* Ap, const Fp* Sp, Fp* num, Fp* den, long long pstride, int L, int n,
                      const Fp* chal, long long chal_stride, int beta_slot, int gamma_slot, int B);

}  // namespace tb
