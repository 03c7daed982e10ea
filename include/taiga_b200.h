/* taiga_b200.h - C ABI of libtaiga_b200.so, the B200-native (sm_100a) prover hot path for anoma/taiga.
 *
 * The reference has NO FFI on this path: the seam is the Rust call
 *     taiga_halo2/src/proof.rs:25-42   Proof::create(pk, params, circuit, instance, rng) -> Result<Proof, plonk::Error>
 * which forwards to halo2_proofs::plonk::create_proof (un-vendored git dependency, taiga_halo2/Cargo.toml:14-15).
 * This header is what a Rust shim (cc + bindgen, see INTEGRATION.md) binds in place of that body.
 *
 * Conventions
 *   - field element: 32 bytes, little-endian canonical integer < modulus (what `to_repr()` returns in Rust).
 *   - point: 64 bytes affine x||y (each a field element of the curve's base field); identity = 64 zero bytes
 *     (the coordinates `vesta::Affine` holds, taiga_halo2/src/proof.rs:26).
 *   - field ids : TB_FP = circuit field (pallas::Base = vesta::Scalar), TB_FQ = vesta::Base.
 *   - curve ids : TB_VESTA = commitment curve of Taiga's proofs (base Fq, scalars Fp), TB_PALLAS (base Fp, scalars Fq).
 *   - every call returns tb_status (0 = OK); nothing throws or panics across the ABI; the message for the last
 *     failure on a context is available from tb_last_error().  A tb_ctx is bound to one GPU and one host thread.
 *   - there is no CPU fallback: every entry point fails with TB_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef TAIGA_B200_H
#define TAIGA_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef int tb_status;
enum { TB_OK = 0, TB_ERR_INVALID = 1, TB_ERR_CUDA = 2, TB_ERR_CONSTRAINT = 3, TB_ERR_INTERNAL = 4 };
enum { TB_FP = 0, TB_FQ = 1 };
enum { TB_VESTA = 0, TB_PALLAS = 1 };

typedef struct tb_ctx tb_ctx;
typedef struct tb_srs tb_srs;

/* ---- context (owns a CUDA stream, twiddle tables, stream-ordered scratch memory) */
tb_status tb_ctx_create(int device, tb_ctx** out);
void tb_ctx_destroy(tb_ctx* ctx);
const char* tb_last_error(const tb_ctx* ctx);
const char* tb_version(void);
tb_status tb_ctx_sync(tb_ctx* ctx);
uint64_t tb_ctx_stream(const tb_ctx* ctx);        /* cudaStream_t, for event timing by the caller */
uint64_t tb_ctx_launch_count(const tb_ctx* ctx);  /* kernels launched through this context so far */
/* Built-in CUDA-event profiler: when enabled every kernel group is bracketed by events on the context's stream;
 * tb_prof_read synchronises and returns accumulated milliseconds and group counts per category, then resets. */
int tb_prof_categories(void);
const char* tb_prof_category_name(int category);
tb_status tb_prof_enable(tb_ctx* ctx, int on);
tb_status tb_prof_read(tb_ctx* ctx, double* ms_out, uint64_t* counts_out);
/* 255-bit Montgomery multiplications executed per category since the last call (the path is bound by the integer pipe, so
 * this is the numerator of its roofline; see bench.py int_util).  Synchronises. */
tb_status tb_prof_work(tb_ctx* ctx, double* modmuls_out);

/* ---- primitives over HOST buffers (copies in and out inside the call).
 * tb_ntt   replaces halo2_proofs arithmetic::best_fft / EvaluationDomain::{lagrange_to_coeff, coeff_to_lagrange}
 *          (EXT; reached from taiga_halo2/src/proof.rs:33-40).  inverse != 0 also scales by 1/n.
 *          coset: 0 = plain; 1 = halo2 zeta-coset (input coefficient i pre-scaled by ZETA^(i mod 3) for the forward
 *          transform, output coefficient i post-scaled by ZETA^-(i mod 3) for the inverse one).
 * tb_msm   replaces halo2_proofs arithmetic::best_multiexp (EXT).  `batch` scalar vectors share one base vector.
 *          window_bits = 0 selects the default window. */
tb_status tb_ntt(tb_ctx* ctx, int field, uint32_t logn, int inverse, int coset, uint32_t batch, const uint8_t* in, uint8_t* out);
tb_status tb_msm(tb_ctx* ctx, int curve, size_t n, uint32_t batch, const uint8_t* scalars, const uint8_t* points,
                 uint32_t window_bits, uint8_t* out_points);

/* ---- the same primitives over DEVICE memory owned by the caller (e.g. torch tensors).  Device field elements
 * are 32-byte Montgomery residues (R = 2^256); convert with tb_dev_{to,from}_mont.  Work is enqueued on the
 * context's stream; call tb_ctx_sync (or wait on the stream) before reading results. */
tb_status tb_dev_to_mont(tb_ctx* ctx, int field, void* d_elems, size_t n);
tb_status tb_dev_from_mont(tb_ctx* ctx, int field, void* d_elems, size_t n);
tb_status tb_dev_ntt(tb_ctx* ctx, int field, uint32_t logn, int inverse, int coset, uint32_t batch, const void* d_in, void* d_out,
                     void* d_scratch /* batch << logn elements; may alias d_in if the input may be destroyed */);
tb_status tb_dev_msm(tb_ctx* ctx, int curve, size_t n, uint32_t batch, const void* d_scalars, const void* d_points,
                     uint32_t window_bits, void* d_out_points /* batch affine points, Montgomery */);

/* ---- circuit description.  Replaces what halo2_proofs keeps inside ProvingKey<vesta::Affine> / VerifyingKey.cs
 * (COMPLIANCE_PROVING_KEY, taiga_halo2/src/constant.rs:145-152; TRIVIAL_RESOURCE_LOGIC_PK,
 * taiga_halo2/src/circuit/resource_logic_examples.rs:50-61).  The Rust shim walks `pk.get_vk().cs()` once per circuit
 * and fills this flat, pointer-based description (INTEGRATION.md); nothing here is Taiga specific. */
typedef struct { uint32_t column; int32_t rotation; } tb_query;             /* (column index within its kind, Rotation) */
enum { TB_COL_ADVICE = 0, TB_COL_FIXED = 1, TB_COL_INSTANCE = 2 };
typedef struct { uint32_t kind; uint32_t index; } tb_column;                /* halo2 Column<Any> */
/* halo2 `Expression<F>` flattened to a DAG in topological order (operands refer to earlier nodes):
 *   CONST a=constant index | ADVICE/FIXED/INSTANCE a=index into the matching *_queries array | NEG a=node
 *   ADD/MUL a,b=nodes | SCALE a=node, b=constant index.  (Selectors are already fixed columns after keygen.) */
enum { TB_EX_CONST = 0, TB_EX_ADVICE = 1, TB_EX_FIXED = 2, TB_EX_INSTANCE = 3, TB_EX_NEG = 4, TB_EX_ADD = 5, TB_EX_MUL = 6, TB_EX_SCALE = 7 };
typedef struct { uint32_t op, a, b; } tb_expr_node;
typedef struct { uint32_t num_exprs; const uint32_t* input_roots; const uint32_t* table_roots; } tb_lookup;  /* lookup::Argument */
typedef struct {
  uint32_t k;                       /* rows = 2^k (PARAMS_SIZE = 15 for Taiga, constant.rs:123-125) */
  uint32_t num_advice, num_fixed, num_instance;
  uint32_t cs_degree;               /* cs.degree() */
  uint32_t blinding_factors;        /* cs.blinding_factors() */
  uint32_t num_advice_queries;   const tb_query* advice_queries;    /* cs.advice_queries, in order */
  uint32_t num_fixed_queries;    const tb_query* fixed_queries;
  uint32_t num_instance_queries; const tb_query* instance_queries;
  uint32_t num_perm_columns;     const tb_column* perm_columns;     /* cs.permutation.columns, in order */
  uint32_t num_constants;        const uint8_t* constants;          /* 32-byte field elements */
  uint32_t num_nodes;            const tb_expr_node* nodes;
  uint32_t num_constraints;      const uint32_t* constraint_roots;  /* every gate's polynomials, gate-major (halo2 order) */
  uint32_t num_lookups;          const tb_lookup* lookups;
  uint8_t vk_transcript_repr[32];  /* vk.transcript_repr (hash of the pinned vk; owned by the Rust side) */
} tb_cs_desc;

/* ---- structured reference string.  Replaces halo2_proofs poly::commitment::Params<vesta::Affine> as held in
 * SETUP_PARAMS_MAP (taiga_halo2/src/constant.rs:128-139).  g / g_lagrange: 2^k affine points each; w, u: one point.
 * The call copies everything to the device and precomputes the fixed-base window tables. */
tb_status tb_srs_load(tb_ctx* ctx, uint32_t k, const uint8_t* g, const uint8_t* g_lagrange, const uint8_t* w, const uint8_t* u,
                      tb_srs** out);
void tb_srs_free(tb_srs* srs);
/* Params::commit (lagrange = 0) / Params::commit_lagrange (lagrange = 1):  out[b] = MSM(scalars[b], basis) + blinds[b] * w.
 * blinds may be NULL (no blinding term). */
tb_status tb_srs_commit(tb_ctx* ctx, const tb_srs* srs, int lagrange, uint32_t batch, const uint8_t* scalars, const uint8_t* blinds,
                        uint8_t* out_points);

/* ---- proving key + batched prover: the drop-in for the body of Proof::create (taiga_halo2/src/proof.rs:25-42).
 * tb_circuit_load replaces halo2_proofs keygen_pk's table building (COMPLIANCE_PROVING_KEY, constant.rs:145-152):
 *   fixed_values : num_fixed columns x 2^k field elements (pk.fixed_values, Lagrange basis), column-major
 *   sigma_values : num_perm_columns x 2^k field elements (pk.permutation.permutations, Lagrange basis)
 * and builds coefficient forms, extended cosets (sub-coset major), l0/l_last/l_blind and the expression programs on
 * the device.  tb_prove_batch replaces plonk::create_proof for n_proofs independent instances of that circuit:
 *   advice       : n_proofs x num_advice x 2^k field elements (the table `synthesize` produced, after
 *                  batch_invert_assigned; the last blinding_factors+1 rows are overwritten with blinding scalars)
 *   instance     : per proof the instance columns concatenated (sum(instance_len) elements); instance_len[num_instance]
 *   seed         : 32 bytes drawn from the caller's RNG (proof.rs:30); blinding scalars of proof i are derived from
 *                  (seed, first_proof_index + i), so results are reproducible for a given seed.  A (seed, index) pair must never
 *                  be reused for a different witness (it would reuse every blinding scalar): draw a fresh seed per call
 *   proofs_out   : n_proofs records of tb_pk_proof_len(pk) bytes at distance proof_stride
 * Errors: TB_ERR_CONSTRAINT mirrors plonk::Error::ConstraintSystemFailure (lookup input missing from its table),
 * TB_ERR_INVALID covers InstanceTooLarge and malformed arguments. */
typedef struct tb_pk tb_pk;
tb_status tb_circuit_load(tb_ctx* ctx, const tb_srs* srs, const tb_cs_desc* cs, const uint8_t* fixed_values, const uint8_t* sigma_values,
                          tb_pk** out);
void tb_pk_free(tb_pk* pk);
size_t tb_pk_proof_len(const tb_pk* pk);
/* keygen_vk on the device (constant.rs:150): commit_lagrange(column, Blind::default()) of every fixed column and of every
 * permutation sigma column, as 64-byte affine points (vk.fixed_commitments, vk.permutation.commitments). */
tb_status tb_pk_commitments(tb_ctx* ctx, const tb_pk* pk, uint8_t* fixed_commitments, uint8_t* sigma_commitments);
tb_status tb_prove_batch(tb_ctx* ctx, const tb_pk* pk, uint32_t n_proofs, const uint8_t* advice, const uint8_t* instance,
                         const uint32_t* instance_len, const uint8_t seed[32], uint32_t first_proof_index, uint8_t* proofs_out,
                         size_t proof_stride);

/* Batched verifier, the counterpart of Proof::verify (taiga_halo2/src/proof.rs:45-54; plonk::verify_proof with
 * SingleVerifier) for n_proofs proofs of one circuit: the transcript is replayed on the host, the final IPA check
 * (one fixed-base MSM over the SRS + one ~100-term MSM per proof) runs on the device.  ok_out[i] = 1 iff proof i is
 * accepted.  instance / instance_len as in tb_prove_batch. */
tb_status tb_verify_batch(tb_ctx* ctx, const tb_pk* pk, uint32_t n_proofs, const uint8_t* instance, const uint32_t* instance_len,
                          const uint8_t* proofs, size_t proof_stride, size_t proof_len, uint8_t* ok_out);

/* Constraint check of n_proofs witnesses of one circuit (halo2 dev::MockProver::verify; the reference's
 * verify_transparently, resource_logic_circuit.rs:597-606).  advice / instance / instance_len as in tb_prove_batch
 * (host, pinned-host or device memory; instance_len on the host).  Advice cells in the last blinding_factors+1 rows are
 * poison whatever they hold.  Per proof, tb_pk_check_slots(pk) = 2C + L + P slots:
 *   [0, C) constraint j unsatisfied | [C, 2C) constraint j poisoned | [2C, 2C+L) lookup l | [2C+L, 2C+L+P) copy, permutation column p
 * fail_rows[i*S + s] = number of failing rows, first_row[i*S + s] = lowest failing row (0xFFFFFFFF if none).
 * Proof i satisfies the circuit iff all its fail_rows are 0.  1 <= n_proofs <= 4096.  Errors: TB_ERR_INVALID for
 * malformed arguments, instance_len > usable rows (InstanceTooLarge) and a sigma value that names no cell. */
size_t    tb_pk_check_slots(const tb_pk* pk);
tb_status tb_check_batch(tb_ctx* ctx, const tb_pk* pk, uint32_t n_proofs, const uint8_t* advice, const uint8_t* instance,
                         const uint32_t* instance_len, uint32_t* fail_rows, uint32_t* first_row);

#ifdef __cplusplus
}
#endif
#endif /* TAIGA_B200_H */
