/*
 * cortex_b200.h — C ABI of the B200-native belief-propagation engine that sits behind
 * Cortex.jl's InferenceEngine / update_marginals! hot path.
 *
 * Every entry point names the reference interface it replaces (paths relative to the
 * ReactiveBayes/Cortex.jl v0.3.0 tree).  The reference has no FFI of its own (pure Julia);
 * these are exactly the calls a `CortexB200` Julia package extension binds with `ccall`
 * (see INTEGRATION.md) and that the Python ctypes mirror in `cortex.jl_b200/` binds for the
 * parity tests.
 *
 * Conventions
 *   - one opaque handle = one engine on one CUDA device, one host thread per handle, one stream;
 *   - every function returns an int32 status (CXB_OK = 0) unless stated; the message of the
 *     last failure is available from cxb_last_error(h);
 *   - the library owns all device memory; host arrays are borrowed for the call only;
 *   - ids (variables and factors) live in ONE shared id space [0, n_ids) like
 *     BipartiteFactorGraphs.jl (ext/BipartiteFactorGraphsExt/BipartiteFactorGraphsExt.jl:22-48);
 *     neighbour iteration order is ascending id;
 *   - "signal id" (sid) is the dense index of a Signal (src/signal.jl:82-115):
 *         marginal(v)      = rank of v among the variables in ascending id order
 *         m2v(connection c)= n_variables + 2c,   m2f(connection c) = n_variables + 2c + 1
 *         (c = position of the (variable,factor) edge in the edge list given to cxb_graph_build)
 *         then ProductOfMessages nodes / free signals in creation order;
 *   - values are `value_dim` scalars per signal, stored on the device in the engine dtype and
 *     exchanged with the host as float64 (cxb_set_values / cxb_get_values) or in the native
 *     dtype (the *_native bulk calls of the structured graphs).
 *
 * There is no CPU fallback: every call that computes requires the CUDA device and fails with
 * CXB_ERR_CUDA otherwise.
 */
#ifndef CORTEX_B200_H
#define CORTEX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cxb_engine cxb_engine; /* opaque */

/* ---- status codes (Julia-side mapping in INTEGRATION.md) --------------------------------- */
enum {
    CXB_OK = 0,
    CXB_ERR_NOT_PENDING = 1,     /* -> ArgumentError, src/signal.jl:399-405                 */
    CXB_ERR_NO_RULE = 2,         /* -> ErrorException, src/inference_engine.jl:358-360      */
    CXB_ERR_OUT_OF_CONTRACT = 3, /* level-synchronous schedule would differ from A.4 order  */
    CXB_ERR_BAD_ARG = 4,
    CXB_ERR_UNSUPPORTED_ENGINE = 5, /* -> UnsupportedModelEngineError, src/model_engine.jl:252 */
    CXB_ERR_CUDA = 6,
    CXB_ERR_STATE = 7,           /* call order violated (e.g. compute before graph build)    */
    CXB_ERR_INTERNAL = 8         /* host allocation failure / C++ exception stopped at the ABI */
};

/* ---- dtype ------------------------------------------------------------------------------- */
enum { CXB_F32 = 0, CXB_F64 = 1 };

/* ---- signal kinds: InferenceSignalVariants, src/inference_signal.jl:16-96 ----------------- */
enum {
    CXB_KIND_UNSPECIFIED = 0,
    CXB_KIND_M2F = 1,      /* MessageToFactor(variable_id, factor_id)    */
    CXB_KIND_M2V = 2,      /* MessageToVariable(variable_id, factor_id)  */
    CXB_KIND_PRODUCT = 3,  /* ProductOfMessages(variable_id, range, factors) */
    CXB_KIND_MARGINAL = 4, /* IndividualMarginal(variable_id)            */
    CXB_KIND_JOINT = 5     /* JointMarginal(factor_id, variable_ids)     */
};

/* ---- dependency flags: add_dependency! kwargs, src/signal.jl:286-293 ---------------------- */
enum {
    CXB_DEP_INTERMEDIATE = 1, /* nibble bit 0x1, src/signal.jl:507 */
    CXB_DEP_WEAK = 2,         /* nibble bit 0x2, src/signal.jl:508 */
    CXB_DEP_NO_LISTEN = 16,   /* listen = false                    */
    CXB_DEP_NO_CHECK_COMPUTED = 32 /* check_computed = false       */
};
/* nibble bits reported by cxb_get_dependencies (src/signal.jl:507-510) */
enum { CXB_NIB_INTERMEDIATE = 1, CXB_NIB_WEAK = 2, CXB_NIB_COMPUTED = 4, CXB_NIB_FRESH = 8 };

/* ---- value families: how m2f / ProductOfMessages / marginal combine their dependencies ---- */
enum {
    CXB_FAMILY_GAUSS_CANON = 0, /* (precision, precision*mean): component-wise sum  (SURVEY App. C) */
    CXB_FAMILY_CATEGORICAL = 1, /* element-wise product, normalised to sum 1       (SURVEY App. C) */
    CXB_FAMILY_GAUSS_MV = 2,    /* (mean, variance) product of test/runtests.jl:40-46              */
    CXB_FAMILY_BETA = 3,        /* (a1+a2-1, b1+b2-1), test/inference_engine_tests.jl:273-294      */
    CXB_FAMILY_SUM = 4,         /* plain sum, test/inference_engine_tests.jl:1179                   */
    /* value types of the variational (VMP) models, test/inference_engine_tests.jl:593-809; assigned per
     * variable with cxb_set_variable_families (a model mixes them), value_dim = 2: */
    CXB_FAMILY_GAUSS_MP = 5,    /* NormalMeanPrecision (mean, precision): product of test/runtests.jl:89-95 */
    CXB_FAMILY_GAMMA = 6,       /* Gamma (shape, scale): product of test/runtests.jl:97-99               */
    CXB_FAMILY_POINT = 7        /* observed value (value[0]); has no product                              */
};

/* ---- message-to-variable rules, registered per factor type (Factor.functional_form,
 *      src/model_engine.jl:119-122; dispatch as test/inference_engine_tests.jl:256-259) --------- */
enum {
    CXB_RULE_NONE = 0,
    CXB_RULE_GAUSS_OBS = 1,    /* canonical: (1/r, y/r); y = value[0] of the single dependency; r = factor param */
    CXB_RULE_GAUSS_RW = 2,     /* canonical random walk: (L,h) -> (L/(1+qL), h/(1+qL)); q = factor param        */
    CXB_RULE_CAT_TABLE = 3,    /* out[x_v] = sum_{x_u} psi[x_lo][x_hi] * in[x_u], normalised; params = psi K*K  */
    CXB_RULE_POTTS = 4,        /* psi[a][b] = exp(beta*[a==b]); params = {beta}                                  */
    CXB_RULE_HMM_EMIT = 5,     /* out = normalise(E[:, o]); o = value[0] of the dependency; params = {M, E K*M}  */
                               /* (o outside [0, M): CXB_ERR_BAD_ARG)                                           */
    CXB_RULE_GAUSS_MV_OBS = 6, /* N(y, r)            test/inference_engine_tests.jl:425-426 (r = 1.0 there)      */
    CXB_RULE_GAUSS_MV_RW = 7,  /* N(m, v + q)        test/inference_engine_tests.jl:427-428 (q = 1.0 there)      */
    CXB_RULE_BETA_BERNOULLI = 8, /* Beta(1 + r, 2 - r) test/inference_engine_tests.jl:256-258                    */
    CXB_RULE_SCALE2 = 9,       /* 2 * x              test/inference_engine_tests.jl:1163-1166                    */
    /* Normal node N(out | mean, precision^-1) under the mean-field factorisation; the m2v rule of BOTH factor types
     * of test/inference_engine_tests.jl:652-695 (two dependencies = the marginals of the other two variables):
     *   one of them Gamma (the precision) -> NormalMeanPrecision(mean(other), mean(precision))        (:666-676)
     *   none of them Gamma (target = precision) -> Gamma(1.5, 2 / (var(a) + var(b) + (mean(a) - mean(b))^2)) (:678-692)
     * mean / var by the dependency's family (POINT: value, 0). */
    CXB_RULE_NORMAL_MEAN_FIELD = 10,
    /* Normal node with the two states of a transition kept JOINT (structured VMP), the :transition branch of
     * test/inference_engine_tests.jl:942-973, 1008-1028. One registration covers every signal of the factor:
     *   JointMarginal <- (m2f a, m2f b, marginal of the precision):  W = [Wa+w  -w; -w  Wb+w], mu = W^-1 [xi_a; xi_b],
     *       value = (mu1, mu2, W11, W12, W21, W22) = MvNormalMeanPrecision, value_dim >= 6            (:942-973)
     *   m2v <- (m2f of the other state, marginal of the precision): NormalMeanPrecision(mean, 1/(var + 1/w)) (:1013-1020)
     *   m2v <- (JointMarginal): Gamma(1.5, 2 / (V11 - V12 - V21 + V22 + (mu1 - mu2)^2)), V = W^-1      (:1021-1026)
     * with w = mean of the Gamma marginal. */
    CXB_RULE_NORMAL_STRUCTURED = 11,
    /* USER-DEFINED rule: a small stack program evaluated per signal, so that a new factor type needs no rebuild of the library
     * (the counterpart of writing a new method of compute_message_to_variable!, src/inference_engine.jl:351-361, for fixed-size
     * values, value_dim <= 8). params = { n_consts, consts[n_consts], code... }; code is a sequence of opcodes with their
     * immediate operands, all stored as doubles (CXB_OP_*). The per-factor parameter (cxb_set_factor_params) defaults to
     * consts[0]. A program error (stack under/overflow, dependency or component out of range) fails the request with
     * CXB_ERR_NO_RULE. The oracle evaluates the same program (cortex_oracle.cpp::run_program). */
    CXB_RULE_PROGRAM = 12
};
/* opcodes of CXB_RULE_PROGRAM (stack of 16, 8 temporaries) */
enum {
    CXB_OP_DEP = 1,    /* DEP i k   : push component k of dependency i (in add_dependency! order)      */
    CXB_OP_CONST = 2,  /* CONST j   : push consts[j]                                                      */
    CXB_OP_PARAM = 3,  /* PARAM     : push the factor's parameter                                         */
    CXB_OP_ADD = 4, CXB_OP_SUB = 5, CXB_OP_MUL = 6, CXB_OP_DIV = 7, /* a b -> a (op) b                    */
    CXB_OP_NEG = 8, CXB_OP_EXP = 9, CXB_OP_LOG = 10, CXB_OP_SQRT = 11,
    CXB_OP_STORE = 12, /* STORE k   : pop -> component k of the result                                    */
    CXB_OP_TSET = 13,  /* TSET j    : pop -> temporary j                                                  */
    CXB_OP_TGET = 14,  /* TGET j    : push temporary j                                                    */
    CXB_OP_NDEPS = 15  /* NDEPS     : push the number of dependencies                                     */
};

/* ---- dependency resolvers: src/dependencies.jl -------------------------------------------- */
enum {
    CXB_RESOLVER_NONE = 0,       /* resolve_dependencies = false, src/inference_engine.jl:65,84     */
    CXB_RESOLVER_DEFAULT_BP = 1, /* DefaultDependencyResolver, src/dependencies.jl:3-173            */
    CXB_RESOLVER_MEAN_FIELD = 2  /* MeanFieldResolver of test/inference_engine_tests.jl:597-621     */
};

/* ---- schedules of update_marginals! (cxb_set_schedule) ---------------------------------------
 * The reference loop (src/inference_engine.jl:559-632) is sequential and in place. The device has three ways to run it:
 *   LEVEL       the level-synchronous frontier schedule (SURVEY A.5) under its contract checks: equal to the reference
 *               order or CXB_ERR_OUT_OF_CONTRACT, and a refused request leaves the engine exactly as it was;
 *   SEQUENTIAL  the reference loop literally, statement by statement, by one warp on the device (exact by construction,
 *               any wiring; one signal at a time);
 *   AUTO        (default) hand-wired graphs (cxb_create_signal / cxb_add_dependency were used) run SEQUENTIAL; graphs
 *               wired by the built-in resolvers run LEVEL (through a memoised schedule or a closed-form plan when the
 *               request and the flag state were seen before) and fall back to SEQUENTIAL when LEVEL refuses.
 * So with AUTO the answer is always the reference's. */
enum { CXB_SCHEDULE_AUTO = 0, CXB_SCHEDULE_LEVEL = 1, CXB_SCHEDULE_SEQUENTIAL = 2 };
/* what answered the last cxb_update_marginals (cxb_last_schedule): LEVEL / SEQUENTIAL as above, or */
enum { CXB_RAN_REPLAY = 3, /* memoised level schedule replayed (same request, same flag state as a recorded run) */
       CXB_RAN_PLAN = 4    /* same, values by the closed-form kernel of a recognised structure (chains / grid / pairwise) */ };

/* statistics of one update_marginals! call */
typedef struct cxb_update_stats {
    int64_t levels;           /* level-synchronous loop levels that executed >= 1 signal           */
    int64_t updates;          /* total signal computations (= TracedInferenceExecution count)      */
    int64_t updates_by_kind[6];
    int64_t final_marginals;  /* marginals computed in the final phase                              */
    int64_t final_linked;     /* linked signals computed in the final phase                         */
    int64_t kernel_launches;  /* CUDA kernels launched by this call                                 */
} cxb_update_stats;

/* ===========================================================================================
 * Engine life cycle.   Replaces: InferenceEngine(...) constructor, src/inference_engine.jl:60-89
 * =========================================================================================== */
int32_t cxb_create(int32_t device, int32_t dtype, int32_t value_dim, int32_t family, cxb_engine** out);
void cxb_destroy(cxb_engine* h);
const char* cxb_last_error(cxb_engine* h);
const char* cxb_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py reports the delta as gpu_launches) */
uint64_t cxb_kernel_launches(void);

/* Graph ingestion. Replaces the 7 backend generics get_variable / get_factor / get_variable_ids /
 * get_factor_ids / get_connection / get_connected_variable_ids / get_connected_factor_ids
 * (src/model_engine.jl:329-391) + set_signals_variants! (src/inference_engine.jl:228-247):
 * the Julia glue walks them once and hands over flat arrays. */
int32_t cxb_graph_build(cxb_engine* h, int64_t n_ids, const uint8_t* is_factor, const int32_t* factor_type,
                        int64_t n_edges, const int64_t* edge_var, const int64_t* edge_fac);

/* Rule registration by factor type. Replaces methods of compute_message_to_variable!
 * (src/inference_engine.jl:351-361) switching on Factor.functional_form. */
int32_t cxb_register_rule(cxb_engine* h, int32_t factor_type, int32_t rule_kind, const double* params,
                          int64_t n_params);
/* per-factor scalar parameter (noise variance of that factor); default = params[0] of its rule */
int32_t cxb_set_factor_params(cxb_engine* h, int64_t n, const int64_t* factor_ids, const double* values);
/* Value family of the signals of a variable (its marginal, messages, ProductOfMessages nodes) when the model mixes
 * value types; default = the engine family given to cxb_create. In the reference the type is carried by the Julia
 * value itself (NormalMeanPrecision / Gamma / Float64, test/runtests.jl:52-99) and `product` dispatches on it. */
int32_t cxb_set_variable_families(cxb_engine* h, int64_t n, const int64_t* variable_ids, const int32_t* families);

/* create_inference_signal(), src/inference_signal.jl:140-142 -> sid */
int64_t cxb_create_signal(cxb_engine* h);
/* set_variant!(signal, variant), src/signal.jl:185-192, for signals made by cxb_create_signal: kind = CXB_KIND_*;
 * JointMarginal(factor_id, variable_ids): pass the factor (its registered rule computes the signal) and -1 as variable */
int32_t cxb_set_signal_variant(cxb_engine* h, int64_t signal, int32_t kind, int64_t variable_id, int64_t factor_id);
/* add_dependency!(signal, dependency; weak, listen, check_computed, intermediate), src/signal.jl:286-337 */
int32_t cxb_add_dependency(cxb_engine* h, int64_t signal, int64_t dependency, int32_t flags);
/* resolve_dependencies!(resolver, engine), src/dependencies.jl:5-15 */
int32_t cxb_resolve_dependencies(cxb_engine* h, int32_t resolver);
/* one call of resolve_factor_dependencies!(resolver, engine, factor_id) / resolve_variable_dependencies!(resolver,
 * engine, variable_id), src/dependencies.jl:17-126: lets a user resolver delegate to a built-in one per id, as
 * test/inference_engine_tests.jl:813-815 does */
int32_t cxb_resolve_factor_dependencies(cxb_engine* h, int32_t resolver, int64_t factor_id);
int32_t cxb_resolve_variable_dependencies(cxb_engine* h, int32_t resolver, int64_t variable_id);
/* link_signal_to_variable!(variable, signal), src/model_engine.jl:80-83 */
int32_t cxb_link_signal(cxb_engine* h, int64_t variable_id, int64_t signal);
/* bulk form of the above (protocol B links every pairwise m2f: 4e7 signals at config-5 size) */
int32_t cxb_link_signals(cxb_engine* h, int64_t n, const int64_t* variable_ids, const int64_t* signals);

/* ---- introspection (bit-exact parity of the wiring) ---------------------------------------- */
int64_t cxb_n_signals(cxb_engine* h);
/* get_variable_marginal / get_connection_message_to_variable / ..._to_factor,
 * src/model_engine.jl:60, src/inference_engine.jl:176-187; returns -1 if absent */
int64_t cxb_signal_id(cxb_engine* h, int32_t kind, int64_t variable_id, int64_t factor_id);
/* get_variant(signal), src/signal.jl:180: out[0]=kind, out[1]=variable_id, out[2]=factor_id,
 * out[3]=range first, out[4]=range last (ProductOfMessages; 0-based positions in the neighbour list) */
int32_t cxb_signal_info(cxb_engine* h, int64_t signal, int64_t out[5]);
/* get_dependencies(signal) + the 4-bit props, src/signal.jl:208, 507-526; returns count (may exceed cap) */
int64_t cxb_get_dependencies(cxb_engine* h, int64_t signal, int64_t* out_ids, uint8_t* out_nibbles, int64_t cap);
/* get_listeners(signal) + listenmask, src/signal.jl:217, 90 */
int64_t cxb_get_listeners(cxb_engine* h, int64_t signal, int64_t* out_ids, uint8_t* out_listen, int64_t cap);
/* engine warnings ("Variable has no connected factors", src/dependencies.jl:40-43): returns count, fills variable ids */
int64_t cxb_get_warnings(cxb_engine* h, int64_t* out_variable_ids, int64_t cap);

/* ---- data in / out -------------------------------------------------------------------------- */
/* set_value!(signal, v) with listener notification, src/signal.jl:232-253; values[n][stride] float64 */
int32_t cxb_set_values(cxb_engine* h, int64_t n, const int64_t* signals, const double* values, int64_t stride);
/* get_value(signal), src/signal.jl:171 */
int32_t cxb_get_values(cxb_engine* h, int64_t n, const int64_t* signals, double* out, int64_t stride);
/* is_pending(signal) (lazy, mutates the cache), is_computed(signal): src/signal.jl:141-164; return 0/1, <0 on error */
int32_t cxb_is_pending(cxb_engine* h, int64_t signal);
int32_t cxb_is_computed(cxb_engine* h, int64_t signal);
/* compute!(strategy, signal; force, skip_if_no_listeners) with the registered rule as strategy,
 * src/signal.jl:392-410: CXB_ERR_NOT_PENDING unless pending or force */
int32_t cxb_compute(cxb_engine* h, int64_t signal, int32_t force, int32_t skip_if_no_listeners);

/* ---- scheduler ------------------------------------------------------------------------------ */
/* request_inference_for(engine, ids), src/inference_engine.jl:298-323 */
int32_t cxb_request_inference(cxb_engine* h, int64_t n, const int64_t* variable_ids);
/* scan_inference_request(request), src/inference_engine.jl:540-546: pending signals reachable from
 * the requested marginals. Order: ascending signal id (the reference order is the DFS visit order;
 * the oracle reports both, parity is on the id-sorted list). Returns count (may exceed cap). */
int64_t cxb_scan(cxb_engine* h, int64_t* out_signals, int64_t cap);
/* update_marginals!(engine, ids), src/inference_engine.jl:559-632 — level-synchronous schedule
 * (SURVEY Appendix A.5). stats may be NULL. */
int32_t cxb_update_marginals(cxb_engine* h, int64_t n, const int64_t* variable_ids, cxb_update_stats* stats);
/* "Prepare once, run many" forms of the two bulk calls. cxb_set_values / cxb_update_marginals take host id arrays and
 * float64 values; at 10^6..10^7 signals per call that host work dwarfs the kernels. A prepared signal list / request
 * validates and uploads its ids ONCE (the reference's InferenceRequest object, src/inference_engine.jl:265-323, is the same
 * idea); values then come in the ENGINE dtype, [n][value_dim] contiguous, from host memory or (values_on_device != 0) from
 * device memory - in which case the call is asynchronous on the engine's stream (cxb_stream). The signals of a list must be
 * distinct and must not depend on each other (bulk set_value! of independent signals, e.g. all observations). Handles
 * (>= 0; -1 on error) stay valid until the structure changes. */
int64_t cxb_prepare_signals(cxb_engine* h, int64_t n, const int64_t* signals);
int32_t cxb_set_values_prepared(cxb_engine* h, int64_t list, const void* values, int32_t values_on_device);
int32_t cxb_get_values_prepared(cxb_engine* h, int64_t list, void* out, int32_t out_on_device);
int64_t cxb_prepare_request(cxb_engine* h, int64_t n, const int64_t* variable_ids);
int32_t cxb_update_marginals_prepared(cxb_engine* h, int64_t request, cxb_update_stats* stats);
/* the CUDA stream the engine launches on (cudaStream_t as void*) */
void* cxb_stream(cxb_engine* h);
/* schedule selection (see CXB_SCHEDULE_*) and which path answered the last request */
int32_t cxb_set_schedule(cxb_engine* h, int32_t schedule);
int32_t cxb_last_schedule(cxb_engine* h);
/* scan_inference_request in the reference's literal order: the DFS visit order of process_dependencies!, duplicates
 * included (src/inference_engine.jl:540-546, src/signal.jl:466-490), by the sequential device traversal */
int64_t cxb_scan_dfs(cxb_engine* h, int64_t* out_signals, int64_t cap);
/* process_dependencies!(f, signal; retry), src/signal.jl:466-490, run on the device in the reference's visit order.
 * The callback is a table: f(dep) = answers[dep] != 0 (one byte per signal); answers == NULL: f = is_pending (the
 * scanner's callback, with its caching side effect). Writes the visit sequence (every call of f, retries included),
 * returns the number of visits (may exceed cap, <0 on error); *processed_out = the function's return value. */
int64_t cxb_process_dependencies_table(cxb_engine* h, int64_t signal, int32_t retry, const uint8_t* answers,
                                       int64_t* out_visited, int64_t cap, int32_t* processed_out);
/* Execution trace of the last cxb_update_marginals (InferenceEngineTracer, src/inference_engine.jl:650-862):
 * enable with cxb_trace_enable(h, 1). out_level: 0-based loop level, -1 = final-phase marginals,
 * -2 = final-phase linked signals. Within a level signals are in ascending id order. */
int32_t cxb_trace_enable(cxb_engine* h, int32_t on);
int64_t cxb_trace_get(cxb_engine* h, int64_t* out_level, int64_t* out_signals, int64_t cap);
/* TracedInferenceExecution.total_time_in_ns (src/inference_engine.jl:650-657) of the same records: a level is one batch of
 * kernels, its device time (CUDA events around the rule and set_value! kernels) is shared evenly by its members */
int64_t cxb_trace_get_times(cxb_engine* h, int64_t* out_ns, int64_t cap);
/* TracedInferenceExecution.variable_id of the same records: under the SEQUENTIAL schedule the requested variable whose
 * traversal executed the signal (and out_level of cxb_trace_get is the reference's round number, executions in the
 * reference's order); under LEVEL the variable of the signal's variant (-1 if none) */
int64_t cxb_trace_get_variables(cxb_engine* h, int64_t* out_variable_ids, int64_t cap);

/* ===========================================================================================
 * Structured model engines: closed-form plans for the fixed-stencil graph families (SURVEY §8a,
 * "the device does not need to store the CSR/nibbles explicitly").  They build the SAME graph,
 * wiring and schedule as cxb_graph_build + DEFAULT_BP on the equivalent explicit graph; the
 * explicit path is what the parity tests compare them against.
 * =========================================================================================== */

/* ---- batch of independent linear-Gaussian random-walk chains (BASELINE configs 1-2) ---------
 * graph per chain: test/inference_engine_tests.jl:436-462 (x_t, y_t, likelihood_t, transition_t).
 * Layout: time-major [T][B]. One run = update_marginals!(engine, x[1:T]) of every chain:
 * B*(6T-4) message updates, all six message classes materialised. */
typedef struct cxb_chains cxb_chains;
int32_t cxb_chains_create(int32_t device, int32_t dtype, int64_t n_chains, int64_t n_steps, cxb_chains** out);
void cxb_chains_destroy(cxb_chains* c);
const char* cxb_chains_last_error(cxb_chains* c);
/* per-chain noise variances q[B] (transition) and r[B] (observation): cxb_set_factor_params analogue */
int32_t cxb_chains_set_noise(cxb_chains* c, const double* q, const double* r);
/* set_value!(m2f(y_t, likelihood_t), y_t) for all (t,b): host array [T][B] in the engine dtype; H2D copy */
int32_t cxb_chains_set_observations(cxb_chains* c, const void* y_host);
/* same, from a device pointer already resident (no copy when y_dev is the internal buffer) */
int32_t cxb_chains_set_observations_device(cxb_chains* c, const void* y_dev);
/* update_marginals!(engine, all state variables); n_updates_out = B*(6T-4) */
int32_t cxb_chains_update_marginals(cxb_chains* c, int64_t* n_updates_out);
/* marginals as canonical pairs [T][B][2] in the engine dtype; D2H copy */
int32_t cxb_chains_get_marginals(cxb_chains* c, void* out_host);
/* message class m in 0..5: 0 m2v(x_t,lik_t), 1 m2v(x_t,tr_{t-1}), 2 m2f(x_t,tr_t), 3 m2v(x_t,tr_t),
 * 4 m2f(x_t,tr_{t-1}), 5 marginal(x_t); [T][B][2] engine dtype */
int32_t cxb_chains_get_messages(cxb_chains* c, int32_t message_class, void* out_host);
/* device pointers for zero-copy interop (torch wraps them for NCCL); index as above, 6 = observations */
void* cxb_chains_device_ptr(cxb_chains* c, int32_t which);
/* host->device observations + update + device->host marginals in one call (the e2e path) */
int32_t cxb_chains_infer_host(cxb_chains* c, const void* y_host, void* marginals_out_host, int64_t* n_updates_out);
/* CUDA stream the handle launches on (cudaStream_t as void*) and last-run kernel time from CUDA events (ms) */
void* cxb_chains_stream(cxb_chains* c);
int32_t cxb_chains_last_kernel_ms(cxb_chains* c, float* ms_out);
int32_t cxb_chains_sync(cxb_chains* c);

/* ---- 2-D Potts grid, loopy BP by synchronous sweeps (BASELINE config 4) ---------------------
 * variables = pixels of an H x W grid (this rank's rows [row0, row0+H) of a global grid);
 * one unary (leaf) factor per pixel + pairwise factors on the 4-neighbourhood, K labels,
 * psi[a][b] = exp(beta*[a==b]).  One sweep = protocol B of SURVEY Appendix B: re-assert the unary
 * evidence, then update_marginals!(engine, all pixels): all m2v, then marginals, then linked m2f. */
typedef struct cxb_grid cxb_grid;
int32_t cxb_grid_create(int32_t device, int32_t dtype, int64_t rows, int64_t cols, int32_t n_labels, double beta,
                        int32_t has_upper_neighbour, int32_t has_lower_neighbour, cxb_grid** out);
void cxb_grid_destroy(cxb_grid* g);
const char* cxb_grid_last_error(cxb_grid* g);
/* set_value!(m2v(v, unary_v), u_v): host [rows][cols][K] engine dtype */
int32_t cxb_grid_set_unary(cxb_grid* g, const void* unary_host);
/* set every pairwise m2f to the uniform initial message (protocol B step 1) */
int32_t cxb_grid_reset_messages(cxb_grid* g);
/* one synchronous sweep on the local rows; halo rows must have been exchanged (cxb_grid_halo_*) */
int32_t cxb_grid_sweep(cxb_grid* g, int64_t* n_updates_out);
/* halo buffers (device pointers, cols*K elements each): the m2f messages this shard sends up/down
 * (direction 0 = to upper neighbour, 1 = to lower neighbour) and receives from them */
void* cxb_grid_halo_send_ptr(cxb_grid* g, int32_t direction);
void* cxb_grid_halo_recv_ptr(cxb_grid* g, int32_t direction);
int64_t cxb_grid_halo_elems(cxb_grid* g);
/* Fused halo exchange over peer memory (NVLink P2P): once a row neighbour is connected, cxb_grid_sweep itself delivers
 * the messages of the cut edges — the sweep kernel stores them straight into the neighbour GPU's halo buffer and a sweep
 * counter is published after the kernel; the next sweep waits (on the stream) for the neighbours' counters. No separate
 * exchange call is needed for a connected direction (0 = the shard above, 1 = the shard below). The reference has no
 * counterpart (single process, src/inference_engine.jl:559-632); SURVEY 8e.
 * cxb_grid_p2p_export writes 128 bytes (two cudaIpcMemHandle_t); cxb_grid_reset_messages requires every shard idle. */
int32_t cxb_grid_p2p_export(cxb_grid* g, void* handles_out);
int32_t cxb_grid_p2p_connect_ipc(cxb_grid* g, int32_t direction, const void* neighbour_handles);
int32_t cxb_grid_p2p_connect_local(cxb_grid* g, int32_t direction, cxb_grid* neighbour);
/* marginals [rows][cols][K] engine dtype, D2H */
int32_t cxb_grid_get_marginals(cxb_grid* g, void* out_host);
/* One JOB through host buffers (the e2e path of config 4): unary evidence [rows][cols][K] from (pinned) host memory, n_sweeps
 * synchronous sweeps, marginals back to (pinned) host memory. Asynchronous and pipelined over three streams: the call returns
 * when everything is enqueued; the evidence of the next job travels in and the marginals of the previous job travel out
 * while this job's sweeps run (two evidence and two marginal buffers). marginals_out_host is complete when cxb_grid_sync
 * returns. Messages carry over from the previous job (call cxb_grid_reset_messages, all shards idle, for a cold start). */
int32_t cxb_grid_infer_host(cxb_grid* g, const void* unary_host, void* marginals_out_host, int32_t n_sweeps, int64_t* n_updates_out);
/* message planes for parity: which = 0..3 m2v from the (up,left,right,down) factor, 4..7 m2f to them; D2H.
 * A sweep computes every m2v but stores only those of its first and last rows; the first read of an m2v plane after a
 * sweep rebuilds the other rows, bit for bit, from the m2f messages that sweep read (one extra kernel on the grid's stream,
 * about 34 GB of traffic at 8192^2, K = 16 fp32; later reads of the same sweep's planes launch nothing).
 * CXB_GRID_EAGER_M2V=1 at cxb_grid_create stores every m2v every sweep instead. */
int32_t cxb_grid_get_messages(cxb_grid* g, int32_t which, void* out_host);
void* cxb_grid_stream(cxb_grid* g);
int32_t cxb_grid_last_kernel_ms(cxb_grid* g, float* ms_out);
int32_t cxb_grid_sync(cxb_grid* g);

/* ---- batch of discrete HMMs (BASELINE config 3) ----------------------------------------------
 * graph per chain as the SSM test with categorical states (SURVEY Appendix C): z_t, y_t, emission
 * and transition factors, uniform prior leaf on z_1. Scaled forward-backward, every message
 * normalised; materialises forward messages and marginals ([T][B][K]). */
typedef struct cxb_hmm cxb_hmm;
int32_t cxb_hmm_create(int32_t device, int32_t dtype, int64_t n_chains, int64_t n_steps, int32_t n_states,
                       int32_t n_symbols, cxb_hmm** out);
void cxb_hmm_destroy(cxb_hmm* m);
const char* cxb_hmm_last_error(cxb_hmm* m);
/* transition A[K][K] (row = from state), emission E[K][M]; float64 host arrays */
int32_t cxb_hmm_set_tables(cxb_hmm* m, const double* transition, const double* emission);
/* observations o[T][B] uint8, host. Every symbol must satisfy 0 <= o < n_symbols: otherwise CXB_ERR_BAD_ARG, and the
 * handle has no observations until a later call succeeds (cxb_hmm_update_marginals returns CXB_ERR_STATE). */
int32_t cxb_hmm_set_observations(cxb_hmm* m, const uint8_t* obs_host);
int32_t cxb_hmm_update_marginals(cxb_hmm* m, int64_t* n_updates_out);
/* marginals [T][B][K] engine dtype, D2H (t0..t1 slice to bound the copy) */
int32_t cxb_hmm_get_marginals(cxb_hmm* m, int64_t t0, int64_t t1, void* out_host);
int32_t cxb_hmm_get_forward(cxb_hmm* m, int64_t t0, int64_t t1, void* out_host);
void* cxb_hmm_stream(cxb_hmm* m);
int32_t cxb_hmm_last_kernel_ms(cxb_hmm* m, float* ms_out);
int32_t cxb_hmm_sync(cxb_hmm* m);

/* ---- arbitrary pairwise categorical graph, loopy BP by synchronous sweeps (BASELINE config 5) -------------------
 * variables 0..n-1, one unary (leaf) factor per variable, pairwise factor f = (u_f < v_f) with table
 * psi_{t_f}[x_u][x_v]; K states. Same graph, wiring and protocol B sweep as cxb_graph_build + DEFAULT_BP +
 * linked m2f on tests/models.py:make_powerlaw_model; a sweep stands for 4m + n + (#ProductOfMessages) updates. */
typedef struct cxb_pairwise cxb_pairwise;
int32_t cxb_pairwise_create(int32_t device, int32_t dtype, int64_t n_variables, int64_t n_factors, int32_t n_states,
                            int32_t n_tables, cxb_pairwise** out);
void cxb_pairwise_destroy(cxb_pairwise* g);
const char* cxb_pairwise_last_error(cxb_pairwise* g);
/* factor endpoints (u < v) and table index per factor, in ascending factor id */
int32_t cxb_pairwise_set_graph(cxb_pairwise* g, const int64_t* fac_u, const int64_t* fac_v, const int32_t* fac_table);
/* tables [n_tables][K][K] float64, indexed [x_lower][x_higher] (CXB_RULE_CAT_TABLE convention) */
int32_t cxb_pairwise_set_tables(cxb_pairwise* g, const double* tables);
/* set_value!(m2v(v, unary_v), u_v): host [n][K] engine dtype */
int32_t cxb_pairwise_set_unary(cxb_pairwise* g, const void* unary_host);
int32_t cxb_pairwise_reset_messages(cxb_pairwise* g);
int32_t cxb_pairwise_sweep(cxb_pairwise* g, int64_t* n_updates_out);
int32_t cxb_pairwise_get_marginals(cxb_pairwise* g, void* out_host);
/* which = 0: m2v, 1: m2f; out[(2f + side)][K], side 0 = endpoint u, 1 = endpoint v; engine dtype */
int32_t cxb_pairwise_get_messages(cxb_pairwise* g, int32_t which, void* out_host);
int64_t cxb_pairwise_algorithmic_bytes(cxb_pairwise* g);
void* cxb_pairwise_stream(cxb_pairwise* g);
int32_t cxb_pairwise_last_kernel_ms(cxb_pairwise* g, float* ms_out);
int32_t cxb_pairwise_sync(cxb_pairwise* g);

#ifdef __cplusplus
}
#endif
#endif /* CORTEX_B200_H */
