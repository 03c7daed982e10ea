// Constraint check of a batch of witnesses on the device: halo2 `dev::MockProver::verify` for the data-driven tb_cs_desc
// (the reference runs it in verify_transparently, resource_logic_circuit.rs:597-606).
//
// Cell values follow halo2's dev::Value: advice cells in rows >= usable are POISON whatever the caller's bytes hold
// (tb_prove_batch overwrites them with blinding scalars).  Negation, addition and scaling propagate poison; a product is a
// real zero when either factor is a real zero, else poison when a factor is.  Checked, per witness:
//   gates    every constraint at every row 0..n: unsatisfied if real and non-zero, poisoned if poison;
//   lookups  for rows < usable, the input tuple must equal, element for element, the table tuple of some row < usable whose
//            elements are all real (exact membership: no theta compression);
//   copies   for permutation column p and rows r < usable, value(p, r) must equal value(sigma(p, r)) and neither be poison.
// Failures go to per-(witness, slot) counters with atomicAdd and the lowest failing row with atomicMin: the result does not
// depend on the order in which threads run.  oracle/mock_prover.py restates the same semantics in Python.
#include <algorithm>
#include <unordered_map>
#define TB_NOINLINE_MUL 0  // loop-structured kernels: small code, keep the multiply inline
#include "capi_internal.cuh"
#include "kernels.cuh"
#include "prover_kernels.cuh"
#include "circuit.cuh"

namespace tb {

constexpr uint32_t CK_MAX_BATCH = 4096;
constexpr int CK_CHUNK = 32;                            // witnesses per internal pass
constexpr size_t CK_CHUNK_BYTES = size_t(1) << 30;      // device bytes one pass may hold (advice, instance, lookup values)

struct CkData {
  const Fp* adv; long long adv_pstride;    // [B][num_advice][n] Montgomery
  const Fp* inst; long long inst_pstride;  // [B][num_instance][n]
  const Fp* fix;                           // [num_fixed][n]
  const Fp* consts;
  int n, usable, rows;                     // rows evaluated: n (gates) or usable (lookup expressions)
  uint32_t* fail; uint32_t* first; int S, J;   // per-witness slot counters, witness stride S; J constraints
  Fp* vals; long long vals_pstride;        // Q_CK_STORE: [B][E][n]
  uint8_t* pois; long long pois_pstride;   //             [B][L][n], 1 = some element of the tuple is poison
};

__device__ __forceinline__ void ck_record(uint32_t* fail, uint32_t* first, int slot, int row) {
  atomicAdd(fail + slot, 1u);
  atomicMin(first + slot, (uint32_t)row);
}

// One thread per (row, witness).  Temporaries live in a shared-memory register file [nregs][T] (two 16-byte halves) as in
// q_interp_kernel; the poison bit of register i is bit i of `pm` (nregs <= 48).
__global__ void __launch_bounds__(128) ck_interp_kernel(const QInstr* __restrict__ prog_, int ninstr, int nregs, CkData d) {
  const uint4* __restrict__ prog = reinterpret_cast<const uint4*>(prog_);
  extern __shared__ uint4 ck_smem[];
  const int T = blockDim.x, tid = threadIdx.x;
  uint4* rlo = ck_smem + tid;
  uint4* rhi = ck_smem + (size_t)nregs * T + tid;
  const int row = blockIdx.x * T + tid, b = blockIdx.y;
  if (row >= d.rows) return;
  const int nm = d.n - 1;
  const Fp* adv = d.adv + (long long)b * d.adv_pstride;
  const Fp* inst = d.inst + (long long)b * d.inst_pstride;
  uint64_t pm = 0;

  auto lds = [&](int r) -> Fp { uint4 x = rlo[r * T], z = rhi[r * T]; Fp v;
    v.l[0] = x.x; v.l[1] = x.y; v.l[2] = x.z; v.l[3] = x.w; v.l[4] = z.x; v.l[5] = z.y; v.l[6] = z.z; v.l[7] = z.w; return v; };
  auto fetch = [&](int kind, uint32_t v, bool& p) -> Fp {
    if (kind == K_REG) { p = (pm >> v) & 1u; return lds((int)v); }
    p = false;
    if (kind == K_CONST) return ldg_fe(d.consts + v);
    const int rot = (int)(v & 255u) - 128; const size_t col = v >> 8;
    const int r = (row + rot + d.n) & nm;
    if (kind == K_ADV) { p = r >= d.usable; return ldg_fe(adv + col * d.n + r); }
    return ldg_fe((kind == K_INST ? inst : d.fix) + col * d.n + r);
  };
  uint4 in = __ldg(prog);
  for (int pc = 0; pc < ninstr; ++pc) {
    const uint32_t w0 = in.x, ia = in.y, ib = in.z, ipad = in.w;
    if (pc + 1 < ninstr) in = __ldg(prog + pc + 1);
    const int op = w0 & 0xff, ak = (w0 >> 16) & 0xff, bk = w0 >> 24, dst = (w0 >> 8) & 0xff;
    bool pa, pb, p;
    Fp r;
    switch (op) {
      case Q_MOV: r = fetch(ak, ia, pa); p = pa; break;
      case Q_NEG: r = fetch(ak, ia, pa).neg(); p = pa; break;
      case Q_ADD: r = fetch(ak, ia, pa) + fetch(bk, ib, pb); p = pa | pb; break;
      case Q_SUB: r = fetch(ak, ia, pa) - fetch(bk, ib, pb); p = pa | pb; break;
      case Q_MUL: {
        const Fp x = fetch(ak, ia, pa), y = fetch(bk, ib, pb);
        r = x * y;
        p = (pa | pb) && !(!pa && x.is_zero()) && !(!pb && y.is_zero());   // real zero times poison is a real zero
        break; }
      case Q_CK_TEST: {
        r = fetch(ak, ia, pa);
        if (pa) ck_record(d.fail, d.first, b * d.S + d.J + (int)ib, row);
        else if (!r.is_zero()) ck_record(d.fail, d.first, b * d.S + (int)ib, row);
        continue; }
      case Q_CK_STORE:
        r = fetch(ak, ia, pa);
        st_fe(d.vals + (long long)b * d.vals_pstride + (size_t)ib * d.n + row, r);
        if (pa) d.pois[(long long)b * d.pois_pstride + (size_t)ipad * d.n + row] = 1;
        continue;
      default: continue;
    }
    rlo[dst * T] = make_uint4(r.l[0], r.l[1], r.l[2], r.l[3]); rhi[dst * T] = make_uint4(r.l[4], r.l[5], r.l[6], r.l[7]);
    pm = (pm & ~(1ull << dst)) | ((uint64_t)p << dst);
  }
}

// Lookup tables as sorted row orders.  Key of table row t of lookup l: (excluded, tuple), excluded = t >= usable or poison,
// excluded rows last; tuples compared element by element on their Montgomery residues (any total order serves exact membership).
struct CkTable {
  const Fp* vals; long long vals_pstride;       // [Bt][E][n]
  const uint8_t* pois; long long pois_pstride;  // [Bt][L][n]
  uint32_t* idx;                                // [Bt][L][n]
  const int2* lk;                               // (first slot, expressions) per lookup
  int L, n, usable;
};
__device__ __forceinline__ bool ck_excluded(const CkTable& t, int a, uint32_t row) {
  return (int)row >= t.usable || t.pois[(long long)(a / t.L) * t.pois_pstride + (size_t)(a % t.L) * t.n + row];
}
// compares table row x with the tuple at (v, y): v points at expression 0 of the lookup, expressions n apart
__device__ __forceinline__ int ck_tuple_cmp(const Fp* tv, uint32_t x, const Fp* v, uint32_t y, int m, int n) {
  for (int e = 0; e < m; ++e) {
    const int c = Fp::cmp_raw(ldg_fe(tv + (size_t)e * n + x), ldg_fe(v + (size_t)e * n + y));
    if (c) return c;
  }
  return 0;
}
__global__ void ck_iota_kernel(uint32_t* idx, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) idx[(size_t)blockIdx.y * n + i] = (uint32_t)i;
}
// one compare-exchange step (k, j) of a bitonic sort of every [Bt][L] row order
__global__ void ck_sort_step_kernel(CkTable t, int k, int j) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x, a = blockIdx.y;
  if (s >= (t.n >> 1)) return;
  const int l = a % t.L;
  const Fp* tv = t.vals + (long long)(a / t.L) * t.vals_pstride + (size_t)t.lk[l].x * t.n;
  uint32_t* I = t.idx + (size_t)a * t.n;
  const int i = ((s & ~(j - 1)) << 1) | (s & (j - 1));
  const bool asc = (i & k) == 0;
  const uint32_t x = I[i], y = I[i | j];
  const bool ex = ck_excluded(t, a, x), ey = ck_excluded(t, a, y);
  const int c = ex != ey ? (ex ? 1 : -1) : ex ? 0 : ck_tuple_cmp(tv, x, tv, y, t.lk[l].y, t.n);
  if (c != 0 && (c > 0) == asc) { I[i] = y; I[i | j] = x; }
}
// one thread per (usable row, lookup, witness): binary search of the input tuple among the sorted table rows
__global__ void ck_lookup_search_kernel(CkTable t, bool shared_table, const Fp* iv, long long iv_pstride, const uint8_t* ip, long long ip_pstride,
                                        uint32_t* fail, uint32_t* first, int S, int slot0) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x, l = blockIdx.y, b = blockIdx.z;
  if (row >= t.usable) return;
  const int n = t.n, m = t.lk[l].y, slot = b * S + slot0 + l;
  if (ip[(long long)b * ip_pstride + (size_t)l * n + row]) { ck_record(fail, first, slot, row); return; }   // poisoned input
  const int a = (shared_table ? 0 : b) * t.L + l;
  const Fp* tv = t.vals + (long long)(a / t.L) * t.vals_pstride + (size_t)t.lk[l].x * n;
  const Fp* v = iv + (long long)b * iv_pstride + (size_t)t.lk[l].x * n;
  const uint32_t* I = t.idx + (size_t)a * n;
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const uint32_t x = I[mid];
    if (!ck_excluded(t, a, x) && ck_tuple_cmp(tv, x, v, row, m, n) < 0) lo = mid + 1; else hi = mid;
  }
  if (lo == n || ck_excluded(t, a, I[lo]) || ck_tuple_cmp(tv, I[lo], v, row, m, n) != 0) ck_record(fail, first, slot, row);
}

// one thread per (usable row, permutation column, witness)
struct CkCopy {
  const Fp* adv; long long adv_pstride; const Fp* inst; long long inst_pstride; const Fp* fix;
  const int2* perm; const uint32_t* map; int n, usable;
  uint32_t* fail; uint32_t* first; int S, slot0;
};
__device__ __forceinline__ Fp ck_cell(const CkCopy& c, int b, int2 col, int row, bool& poison) {
  poison = col.x == TB_COL_ADVICE && row >= c.usable;
  const Fp* base = col.x == TB_COL_ADVICE ? c.adv + (long long)b * c.adv_pstride : col.x == TB_COL_INSTANCE ? c.inst + (long long)b * c.inst_pstride : c.fix;
  return ldg_fe(base + (size_t)col.y * c.n + row);
}
__global__ void ck_copy_kernel(CkCopy c) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y, b = blockIdx.z;
  if (row >= c.usable) return;
  const uint32_t to = c.map[(size_t)p * c.n + row];
  bool pa, pb;
  const Fp x = ck_cell(c, b, c.perm[p], row, pa), y = ck_cell(c, b, c.perm[to >> 24], (int)(to & 0xffffffu), pb);
  if (pa || pb || x != y) ck_record(c.fail, c.first, b * c.S + c.slot0 + p, row);
}

// ---------------------------------------------------------------- host
static void ck_run(Ctx* ctx, const QProgram& prog, const CkData& d, int B) {
  if (!prog.ninstr) return;
  ctx->opt_in_smem(ck_interp_kernel, 96 * 1024);
  int T = (96 * 1024) / (prog.nregs * 32);
  T = T >= 128 ? 128 : (T / 16) * 16;
  TB_REQUIRE(T >= 16, "constraint program register file does not fit shared memory");
  while (T > d.rows && T > 16) T >>= 1;
  ck_interp_kernel<<<dim3((d.rows + T - 1) / T, B), T, (size_t)prog.nregs * T * 32, ctx->stream>>>(prog.dev, prog.ninstr, prog.nregs, d);
  TB_LAUNCH_CHECK(); ctx->launches++;
}

static void ck_sort_tables(Ctx* ctx, const CkTable& t, int arrays) {
  ck_iota_kernel<<<dim3((t.n + 255) / 256, arrays), 256, 0, ctx->stream>>>(t.idx, t.n);
  TB_LAUNCH_CHECK(); ctx->launches++;
  for (int k = 2; k <= t.n; k <<= 1)
    for (int j = k >> 1; j >= 1; j >>= 1) {
      ck_sort_step_kernel<<<dim3((t.n / 2 + 255) / 256, arrays), 256, 0, ctx->stream>>>(t, k, j);
      TB_LAUNCH_CHECK(); ctx->launches++;
    }
}

static tb_cs_desc desc_of(const Circuit& C, std::vector<tb_lookup>& lks) {
  tb_cs_desc d; memset(&d, 0, sizeof(d));
  d.k = C.k; d.num_advice = C.na; d.num_fixed = C.nf; d.num_instance = C.ni; d.cs_degree = C.degree; d.blinding_factors = C.bf;
  d.num_advice_queries = (uint32_t)C.aq.size(); d.advice_queries = C.aq.data();
  d.num_fixed_queries = (uint32_t)C.fq.size(); d.fixed_queries = C.fq.data();
  d.num_instance_queries = (uint32_t)C.iq.size(); d.instance_queries = C.iq.data();
  d.num_perm_columns = C.P; d.perm_columns = C.perm.data();
  d.num_constants = C.nconsts; d.constants = C.consts_bytes.data();
  d.num_nodes = (uint32_t)C.nodes.size(); d.nodes = C.nodes.data();
  d.num_constraints = (uint32_t)C.roots.size(); d.constraint_roots = C.roots.data();
  lks.clear();
  for (uint32_t l = 0; l < C.L; ++l) lks.push_back({(uint32_t)C.lk_in[l].size(), C.lk_in[l].data(), C.lk_tab[l].data()});
  d.num_lookups = C.L; d.lookups = lks.data();
  return d;
}

// sigma[p][r] = delta^p' * omega^r' decoded back to the cell (p', r'); throws if a value names no cell (malformed key)
static std::vector<uint32_t> decode_sigma(Ctx* ctx, const Circuit& C) {
  const size_t n = C.n, P = C.P;
  std::vector<Fp> sig(P * n), ident(P * n);
  TB_CUDA(cudaMemcpyAsync(sig.data(), C.sig_vals, P * n * sizeof(Fp), cudaMemcpyDeviceToHost, ctx->stream));
  ctx->sync();
  std::unordered_map<uint64_t, uint32_t> where;
  where.reserve(P * n);
  Fp dp = Fp::one();
  for (size_t p = 0; p < P; ++p) {
    Fp v = dp;
    for (size_t r = 0; r < n; ++r) {
      ident[p * n + r] = v;
      const uint64_t key = (uint64_t)v.l[0] | (uint64_t)v.l[1] << 32;
      if (!where.emplace(key, (uint32_t)(p << 24 | r)).second) throw std::runtime_error("sigma decode: 64-bit key collision");
      v = v * C.omega;
    }
    dp = dp * C.delta;
  }
  std::vector<uint32_t> map(P * n);
  for (size_t i = 0; i < P * n; ++i) {
    const Fp& s = sig[i];
    auto it = where.find((uint64_t)s.l[0] | (uint64_t)s.l[1] << 32);
    const uint32_t to = it == where.end() ? 0xffffffffu : it->second;
    TB_REQUIRE(to != 0xffffffffu && ident[(size_t)(to >> 24) * n + (to & 0xffffffu)] == s, "malformed key: a permutation value decodes to no cell");
    map[i] = to;
  }
  return map;
}

static bool reads_only_fixed(const Circuit& C, uint32_t node) {
  const tb_expr_node& nd = C.nodes[node];
  switch (nd.op) {
    case TB_EX_ADVICE: case TB_EX_INSTANCE: return false;
    case TB_EX_NEG: case TB_EX_SCALE: return reads_only_fixed(C, nd.a);
    case TB_EX_ADD: case TB_EX_MUL: return reads_only_fixed(C, nd.a) && reads_only_fixed(C, nd.b);
    default: return true;
  }
}

template <class T> static T* ck_upload(const std::vector<T>& v) {
  T* p = nullptr;
  TB_CUDA(cudaMalloc(&p, std::max<size_t>(1, v.size()) * sizeof(T)));
  if (!v.empty()) TB_CUDA(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return p;
}

// Set-up of one key, once: programs, sigma map, and the sorted tables when they read only fixed columns.  Key-lifetime
// tables are plain device allocations, like the rest of the key; per-call scratch comes from the stream-ordered pool.
static const CheckKey& check_key(Ctx* ctx, const Circuit& C) {
  std::lock_guard<std::mutex> lk(C.mu);
  if (C.check) return *C.check;
  std::unique_ptr<CheckKey> K(new CheckKey());
  const size_t n = C.n;
  std::vector<tb_lookup> lks;
  const tb_cs_desc d = desc_of(C, lks);
  TB_REQUIRE(C.k <= 24 && C.P <= 256, "key too large for the packed copy map");
  q_compile_check_gates(&d, &K->gates);
  std::vector<int2> lkinfo;
  for (uint32_t l = 0; l < C.L; ++l) { lkinfo.push_back(make_int2(K->E, (int)C.lk_in[l].size())); K->E += (int)C.lk_in[l].size(); }
  K->d_lk = ck_upload(lkinfo);
  if (C.L) {
    q_compile_check_lookups(&d, false, &K->lk_in);
    q_compile_check_lookups(&d, true, &K->lk_tab);
    K->tables_fixed = true;
    for (uint32_t l = 0; l < C.L; ++l) for (uint32_t r : C.lk_tab[l]) K->tables_fixed = K->tables_fixed && reads_only_fixed(C, r);
    if (K->tables_fixed) {
      TB_CUDA(cudaMalloc(&K->tab_vals, (size_t)K->E * n * sizeof(Fp)));
      TB_CUDA(cudaMalloc(&K->tab_pois, (size_t)C.L * n));
      TB_CUDA(cudaMalloc(&K->tab_idx, (size_t)C.L * n * sizeof(uint32_t)));
      TB_CUDA(cudaMemsetAsync(K->tab_pois, 0, (size_t)C.L * n, ctx->stream));
      CkData cd; memset(&cd, 0, sizeof(cd));
      cd.fix = C.fixed_vals; cd.consts = C.consts; cd.n = (int)n; cd.usable = (int)C.usable; cd.rows = (int)C.usable;
      cd.vals = K->tab_vals; cd.pois = K->tab_pois;
      ck_run(ctx, K->lk_tab, cd, 1);
      CkTable t{K->tab_vals, 0, K->tab_pois, 0, K->tab_idx, K->d_lk, (int)C.L, (int)n, (int)C.usable};
      ck_sort_tables(ctx, t, (int)C.L);
    }
  }
  if (C.P) K->perm_map = ck_upload(decode_sigma(ctx, C));
  ctx->sync();
  C.check = std::move(K);
  return *C.check;
}

static void check_batch(Ctx* ctx, const Circuit& C, uint32_t B, const uint8_t* advice, const uint8_t* instance, const uint32_t* instance_len,
                        uint32_t* fail_out, uint32_t* first_out) {
  size_t inst_total = 0;
  for (uint32_t c = 0; c < C.ni; ++c) { TB_REQUIRE(instance_len[c] <= C.usable, "InstanceTooLarge"); inst_total += instance_len[c]; }
  const CheckKey& K = check_key(ctx, C);
  const size_t n = C.n; const long long nn = (long long)n;
  const int na = C.na, ni = C.ni, ni1 = std::max(1, ni), L = C.L, L1 = std::max(1, L), E1 = std::max(1, K.E), J = (int)C.num_constraints;
  const int S = 2 * J + L + (int)C.P;
  cudaStream_t st = ctx->stream;
  // witnesses per pass: at most CK_CHUNK, and no more than CK_CHUNK_BYTES of per-witness device buffers
  const size_t per = 32 * n * (size_t)(na + ni1 + E1 * (K.tables_fixed || !L ? 1 : 2)) + 2 * (size_t)L1 * n + (K.tables_fixed ? 0 : 4 * (size_t)L1 * n);
  const int chunk = (int)std::max<size_t>(1, std::min<size_t>({(size_t)CK_CHUNK, (size_t)B, CK_CHUNK_BYTES / per}));
  DevBuf<uint32_t> dfail(ctx, (size_t)B * S), dfirst(ctx, (size_t)B * S);
  TB_CUDA(cudaMemsetAsync(dfail.get(), 0, (size_t)B * S * 4, st));
  TB_CUDA(cudaMemsetAsync(dfirst.get(), 0xff, (size_t)B * S * 4, st));
  DevBuf<Fp> adv(ctx, (size_t)chunk * na * n), inst(ctx, (size_t)chunk * ni1 * n);
  DevBuf<Fp> ivals, tvals; DevBuf<uint8_t> ipois, tpois; DevBuf<uint32_t> tidx;
  if (L) {
    ivals = DevBuf<Fp>(ctx, (size_t)chunk * K.E * n); ipois = DevBuf<uint8_t>(ctx, (size_t)chunk * L * n);
    if (!K.tables_fixed) { tvals = DevBuf<Fp>(ctx, (size_t)chunk * K.E * n); tpois = DevBuf<uint8_t>(ctx, (size_t)chunk * L * n); tidx = DevBuf<uint32_t>(ctx, (size_t)chunk * L * n); }
  }
  for (uint32_t b0 = 0; b0 < B; b0 += (uint32_t)chunk) {
    const int Bc = (int)std::min<uint32_t>((uint32_t)chunk, B - b0);
    uint32_t* fail = dfail.get() + (size_t)b0 * S; uint32_t* first = dfirst.get() + (size_t)b0 * S;
    TB_CUDA(cudaMemcpyAsync(adv.get(), advice + (size_t)b0 * na * n * 32, (size_t)Bc * na * n * 32, cudaMemcpyDefault, st));   // host, pinned or device
    fe_to_mont<Fp>(ctx, adv.get(), (size_t)Bc * na * n);
    if (ni) {
      TB_CUDA(cudaMemsetAsync(inst.get(), 0, (size_t)Bc * ni * n * sizeof(Fp), st));
      size_t off = 0;
      for (int c = 0; c < ni; ++c) {
        if (instance_len[c])
          TB_CUDA(cudaMemcpy2DAsync(inst.get() + (size_t)c * n, (size_t)ni * n * 32, instance + 32 * ((size_t)b0 * inst_total + off), inst_total * 32,
                                    (size_t)instance_len[c] * 32, Bc, cudaMemcpyDefault, st));
        off += instance_len[c];
      }
      fe_to_mont<Fp>(ctx, inst.get(), (size_t)Bc * ni * n);
    }
    CkData cd; memset(&cd, 0, sizeof(cd));
    cd.adv = adv.get(); cd.adv_pstride = (long long)na * nn; cd.inst = inst.get(); cd.inst_pstride = (long long)ni1 * nn; cd.fix = C.fixed_vals;
    cd.consts = C.consts; cd.n = (int)n; cd.usable = (int)C.usable; cd.fail = fail; cd.first = first; cd.S = S; cd.J = J;
    cd.rows = (int)n;
    ck_run(ctx, K.gates, cd, Bc);
    if (L) {
      CkTable t{K.tab_vals, 0, K.tab_pois, 0, K.tab_idx, K.d_lk, L, (int)n, (int)C.usable};
      cd.rows = (int)C.usable;
      if (!K.tables_fixed) {
        TB_CUDA(cudaMemsetAsync(tpois.get(), 0, (size_t)Bc * L * n, st));
        cd.vals = tvals.get(); cd.vals_pstride = (long long)K.E * nn; cd.pois = tpois.get(); cd.pois_pstride = (long long)L * nn;
        ck_run(ctx, K.lk_tab, cd, Bc);
        t = CkTable{tvals.get(), (long long)K.E * nn, tpois.get(), (long long)L * nn, tidx.get(), K.d_lk, L, (int)n, (int)C.usable};
        ck_sort_tables(ctx, t, Bc * L);
      }
      TB_CUDA(cudaMemsetAsync(ipois.get(), 0, (size_t)Bc * L * n, st));
      cd.vals = ivals.get(); cd.vals_pstride = (long long)K.E * nn; cd.pois = ipois.get(); cd.pois_pstride = (long long)L * nn;
      ck_run(ctx, K.lk_in, cd, Bc);
      ck_lookup_search_kernel<<<dim3((unsigned)((C.usable + 255) / 256), L, Bc), 256, 0, st>>>(t, K.tables_fixed, ivals.get(), (long long)K.E * nn, ipois.get(),
                                                                                             (long long)L * nn, fail, first, S, 2 * J);
      TB_LAUNCH_CHECK(); ctx->launches++;
    }
    if (C.P) {
      CkCopy cc{adv.get(), (long long)na * nn, inst.get(), (long long)ni1 * nn, C.fixed_vals, C.d_perm, K.perm_map, (int)n, (int)C.usable, fail, first, S, 2 * J + L};
      ck_copy_kernel<<<dim3((unsigned)((C.usable + 255) / 256), C.P, Bc), 256, 0, st>>>(cc);
      TB_LAUNCH_CHECK(); ctx->launches++;
    }
  }
  TB_CUDA(cudaMemcpyAsync(fail_out, dfail.get(), (size_t)B * S * 4, cudaMemcpyDefault, st));
  TB_CUDA(cudaMemcpyAsync(first_out, dfirst.get(), (size_t)B * S * 4, cudaMemcpyDefault, st));
  ctx->sync();
}

}  // namespace tb

using namespace tb;

extern "C" {

size_t tb_pk_check_slots(const tb_pk* pk) {
  const Circuit* C = reinterpret_cast<const Circuit*>(pk);
  return C ? 2 * (size_t)C->num_constraints + C->L + C->P : 0;
}

tb_status tb_check_batch(tb_ctx* ctx, const tb_pk* pk, uint32_t n_proofs, const uint8_t* advice, const uint8_t* instance, const uint32_t* instance_len,
                         uint32_t* fail_rows, uint32_t* first_row) {
  TB_API_BEGIN(ctx)
  const Circuit* C = reinterpret_cast<const Circuit*>(pk);
  TB_REQUIRE(C && n_proofs >= 1 && n_proofs <= CK_MAX_BATCH && advice && fail_rows && first_row && (C->ni == 0 || (instance && instance_len)),
             "tb_check_batch arguments");
  TB_CUDA(cudaSetDevice(ctx->c.device));
  check_batch(&ctx->c, *C, n_proofs, advice, instance, instance_len, fail_rows, first_row);
  TB_API_END(ctx)
}

}  // extern "C"
