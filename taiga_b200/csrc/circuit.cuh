// The device-resident proving key of one circuit (tb_pk) shared by prover.cu and verifier.cu.
#pragma once
#include <atomic>
#include <map>
#include <mutex>
#include <set>
#include <memory>
#include <vector>
#include "prover_kernels.cuh"

namespace tb {

enum PolyKind { PK_INST = 0, PK_ADV, PK_PZ, PK_LZ, PK_LPIN, PK_LPTAB, PK_FIXED, PK_SIG, PK_H, PK_RANDOM };
struct PolyId { int kind, idx; bool operator<(const PolyId& o) const { return kind != o.kind ? kind < o.kind : idx < o.idx; } bool operator==(const PolyId& o) const { return kind == o.kind && idx == o.idx; } };
struct QueryRef { PolyId poly; int rot; };
struct WsBlock { void* p = nullptr; size_t bytes = 0; };
// Scratch of one (context, batch size) pair: device blocks in request order and the small tables uploaded on first use.
// A tb_pk may be shared by several contexts (= host threads); each gets its own workspace, and a second thread entering
// with the SAME context and batch size while a call is in flight is refused (TB_ERR_INVALID) instead of corrupting it.
struct ProveWs { std::vector<WsBlock> blocks; std::vector<void*> tables; std::vector<std::vector<uint8_t>> table_bytes; std::atomic<int> busy{0}; };

// What tb_check_batch needs of a key beyond the prover's tables (check.cu), built on the first check and read-only afterwards.
struct CheckKey {
  QProgram gates, lk_in, lk_tab;   // Q_CK_TEST per constraint; Q_CK_STORE per lookup input / table expression
  int E = 0;                       // lookup expressions over all lookups
  int2* d_lk = nullptr;            // per lookup: (first expression slot, expressions)
  uint32_t* perm_map = nullptr;    // [P][n]: the cell sigma sends (column p, row r) to, packed p' << 24 | r'
  // tables that read only fixed columns and constants, evaluated and sorted once: [L][n] row order, [E][n] values, [L][n] poison
  bool tables_fixed = false;
  uint32_t* tab_idx = nullptr; Fp* tab_vals = nullptr; uint8_t* tab_pois = nullptr;
  ~CheckKey() {
    for (void* p : {(void*)d_lk, (void*)perm_map, (void*)tab_idx, (void*)tab_vals, (void*)tab_pois, (void*)gates.dev, (void*)lk_in.dev, (void*)lk_tab.dev})
      if (p) cudaFree(p);
  }
};

struct Circuit {
  Ctx* ctx; const Srs* srs;
  // deep copy of the description
  uint32_t k, na, nf, ni, degree, bf, P, L, chunk, nsets, pieces; int ext_k, R; size_t n, usable;
  std::vector<tb_query> aq, fq, iq; std::vector<tb_column> perm;
  std::vector<tb_expr_node> nodes; std::vector<uint32_t> roots; std::vector<uint8_t> consts_bytes; uint32_t nconsts;
  std::vector<std::vector<uint32_t>> lk_in, lk_tab; std::vector<tb_lookup> lk_desc;
  Fp vk_repr;  // canonical
  // device tables
  Fp *fixed_vals = nullptr, *fixed_polys = nullptr, *fixed_cosets = nullptr, *sig_vals = nullptr, *sig_polys = nullptr, *sig_cosets = nullptr;
  Fp *l0 = nullptr, *l_last = nullptr, *l_blind = nullptr, *consts = nullptr, *wr_inv = nullptr;
  Fp* coset_pre = nullptr;   // [R][n]: zeta^(i mod 3) * w_ext^(i * k1), the factor the forward coset NTT applies to coefficient i for sub-coset k1
  int2 *d_aq = nullptr, *d_fq = nullptr, *d_iq = nullptr, *d_perm = nullptr;
  QProgram prog_lookups;
  // gate programs keyed by number of parts: `gate_parts` holds the constraints evaluated on every sub-coset (all of them when the
  // circuit is not split), `gate_parts_lo` the low-degree ones (degree <= R / 2) that are evaluated on every second sub-coset only
  std::map<int, std::vector<QProgram>> gate_parts, gate_parts_lo;
  bool split = false; uint32_t num_constraints = 0, t_pl = 0;   // t_pl: permutation + lookup terms folded after the gates
  std::vector<Fp> t_inv; Fp delta, zeta, omega, r_inv;
  Fp delta_c0[16];
  // evaluation / multiopen structure (host)
  std::vector<QueryRef> evals;            // transcript order of the evaluation section
  std::vector<QueryRef> queries;          // multiopen query order
  std::vector<int> rots;                  // distinct rotations (evaluation points), in order of first appearance in `queries`
  std::vector<PolyId> uniq; std::vector<int> uniq_set; std::vector<std::vector<int>> point_sets;
  uint32_t proof_len;
  // persistent per-batch-size workspace and cached small tables (see prove_batch)
  mutable std::mutex mu;                                                   // guards the three caches below
  mutable std::map<std::pair<const Ctx*, int>, std::unique_ptr<ProveWs>> ws;
  mutable std::vector<Aff<Fq>> vk_fixed, vk_sigma;   // verifying-key commitments (Montgomery, host), filled on first verification
  mutable std::unique_ptr<CheckKey> check;           // constraint-check tables, filled on the first tb_check_batch
  ProveWs& workspace(const Ctx* c, int B) const {
    std::lock_guard<std::mutex> lk(mu);
    auto& slot = ws[std::make_pair(c, B)];
    if (!slot) slot.reset(new ProveWs());
    return *slot;
  }

  ~Circuit() {
    for (auto& kv : ws) { for (auto& b : kv.second->blocks) cudaFree(b.p); for (void* p : kv.second->tables) cudaFree(p); }
    for (void* p : {(void*)fixed_vals, (void*)fixed_polys, (void*)fixed_cosets, (void*)sig_vals, (void*)sig_polys, (void*)sig_cosets, (void*)l0, (void*)l_last,
                    (void*)l_blind, (void*)consts, (void*)wr_inv, (void*)coset_pre, (void*)d_aq, (void*)d_fq, (void*)d_iq, (void*)d_perm, (void*)prog_lookups.dev})
      if (p) cudaFree(p);
    for (auto& kv : gate_parts) for (auto& qp : kv.second) if (qp.dev) cudaFree(qp.dev);
    for (auto& kv : gate_parts_lo) for (auto& qp : kv.second) if (qp.dev) cudaFree(qp.dev);
  }
};

}  // namespace tb
