// hmm_tc.cuh — tensor-core (tcgen05 + TMEM) path of the HMM engine for large state counts (BASELINE config 3, K = 512).
//
// At K >= 128 one time step of a batch of chains is a dense GEMM: pred[chain][j] = sum_i msg[chain][i] * Tbl[i][j]
// (Tbl = A forward, A^T backward), followed by the elementwise categorical rules (emission product, marginal product,
// normalisation).  One kernel launch = one time step of every chain (the launch boundary is the only grid-wide
// synchronisation the recursion needs):
//   * CTA (tile, slice) owns 128 chains (MMA M) x NT = 32 or 64 output states and the full reduction over K input states;
//   * operands are bf16 "split" pieces (x = p0 + p1 + p2, piece k = bf16 of what the earlier pieces left over); the product
//     is accumulated in fp32 in TMEM from the piece products p_a q_b with a + b < 3 (fp32-level accuracy, which sparse
//     tables need: see NP below). The table pieces of a chunk lie one after the other in the stage, so message piece a meets table
//     pieces 0 .. NP-1-a in ONE tcgen05.mma.kind::f16 of N = (NP - a) NT: NP instructions per 16 input states instead of
//     NP (NP + 1) / 2, into NP accumulator blocks that the epilogue adds small to large;
//   * both operands stream through a 3-stage shared-memory ring (~180 KB in flight per SM) by 1-D bulk async copies
//     (cp.async.bulk, completion on mbarriers), ONE copy per operand and stage, of images that are ALREADY in the canonical
//     K-major / no-swizzle UMMA layout: the table slices are formatted once on the host ([slice][chunk][piece]), the message
//     operand of step t+1 is written in that layout ([tile][chunk][piece]) by the epilogue of step t;
//   * warp roles: warps 0-3 epilogue (TMEM -> registers, rules, stores) and, while the MMAs run, the exact
//     normalisation of the PREVIOUS step's output; warp 4 bulk-copy producer; warps 5 and 6 MMA issuers (one elected
//     thread each, alternate chunks, separate accumulator sets): what a step waits on is the issue rate of a thread's
//     tcgen05.mma stream (~60-80 cycles per instruction at these small N; measured with the clock stamps of
//     CXB_HMM_TC_TRACE=1), not the tensor pipe (N = 32 .. 96: 16 .. 48 cycles) and not the ingest (~77 B/clk per SM);
//   * normalisation is deferred exactly as in the K = 64 kernel: the carried message is scaled by the power of two
//     2^-floor(log2 sum(prev)), each step writes its unnormalised result plus per-slice row sums, and the next launch
//     (or the finishing kernel) divides by the exact total.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace cxb {
namespace tc {

constexpr int M_TILE = 128;   // chains per CTA (MMA M)
// output states per CTA (MMA N) is a template parameter NT: 64 (64 CTAs at B = 1,024, K = 512) or 32 (128 CTAs: less
// operand ingest and half the epilogue per SM, more aggregate L2 traffic)
constexpr int K_CHUNK = 64;   // input states per operand chunk (4 MMA K-steps of 16)
// NP = bf16 pieces per operand: x = p0 + p1 + p2, p_k = bf16(residual), ~2^-25 per term (fp32-level). Two pieces keep
// ~2^-17 per term: enough for dense tables, where the 512 terms of a sum average it out, NOT for sparse ones (1e-4 on a
// banded matrix). Products p_a * q_b with a + b < NP: 6 per 16 input states.
constexpr int NP = 3;
template <int NT>
struct Cfg {
    static constexpr uint32_t B_CHUNK_BYTES = NT * 64 * 2;                    // table chunk, per piece
    static constexpr uint32_t STAGE_BYTES = NP * (128 * 64 * 2) + NP * B_CHUNK_BYTES;  // message pieces + table pieces
    static constexpr int STAGES = (int)((200u * 1024u) / STAGE_BYTES);        // ~200 KB of operands in flight
    // instruction descriptor: D = f32, A = B = bf16, both K-major, N = n, M = 128
    static constexpr uint32_t idesc(uint32_t n) { return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24); }
    // The table pieces of a chunk lie one after the other in the stage, which makes them ONE B operand of NP x NT rows:
    // message piece a is multiplied with table pieces 0 .. NP-1-a in a single tcgen05.mma of N = (NP - a) NT that
    // accumulates into TMEM columns [0, N): column block b ends up with sum_a msg_a tbl_b, the epilogue adds the blocks
    // (small to large). NP MMAs per 16 input states instead of NP (NP + 1) / 2 — the step was bound by the issue rate
    // of one thread's tcgen05.mma stream (~60 cycles per instruction at N = 32), not by the tensor pipe or the ingest.
    // TWO issuer threads take the chunks alternately, each into its own set of accumulator blocks (the epilogue adds the
    // sets): the issue streams overlap, the tensor pipe has room for both.
    static constexpr uint32_t SET_COLS = NP * NT;
    static constexpr uint32_t TMEM_COLS = 2 * SET_COLS <= 32 ? 32 : 2 * SET_COLS <= 64 ? 64 : 2 * SET_COLS <= 128 ? 128 : 2 * SET_COLS <= 256 ? 256 : 512;
    static_assert(NP * NT <= 256, "accumulator blocks must fit one MMA (N <= 256)");
};
constexpr int THREADS = 224;  // 4 epilogue warps + producer warp + 2 MMA issuer warps
constexpr int MAX_K = 2048;   // any multiple of 64 up to here (both operands stream through the ring)
constexpr uint32_t A_CHUNK_BYTES = M_TILE * K_CHUNK * 2;  // 16 KB per hi / lo
constexpr uint32_t LBO = 128;                             // bytes between core matrices adjacent in K
constexpr uint32_t SBO = (K_CHUNK / 8) * 128;             // bytes between 8-row groups

// element offset (in bf16 elements) of (row, k) inside one canonical chunk: [row/8][k/8][row%8][k%8]
__host__ __device__ inline uint32_t chunk_elem(uint32_t row, uint32_t k) {
    return ((row >> 3) * (K_CHUNK / 8) + (k >> 3)) * 64 + (row & 7) * 8 + (k & 7);
}

// ---- PTX wrappers ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {  // K-major, no swizzle, version 1 (Blackwell)
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(LBO >> 4) << 16) | ((uint64_t)(SBO >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {  // no wait: several loads in flight
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ float pow2_inv(float s) {
    unsigned e = (__float_as_uint(s) >> 23) & 0xffu;
    return __uint_as_float((254u - e) << 23);
}
__device__ __forceinline__ float rcp_nr(float x) {  // MUFU.RCP + one Newton step
    float q;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(q) : "f"(x));
    return fmaf(q, fmaf(-x, q, 1.0f), q);
}
// split 8 consecutive values into NP bf16 pieces (piece k = bf16 of what the earlier pieces left over), one 16-byte vector each
__device__ __forceinline__ void split_store8(const float* x, __nv_bfloat16* const (&dst)[NP]) {
    float res[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) res[i] = x[i];
#pragma unroll
    for (int pc = 0; pc < NP; ++pc) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __nv_bfloat16 p0 = __float2bfloat16_rn(res[2 * i]), p1 = __float2bfloat16_rn(res[2 * i + 1]);
            res[2 * i] -= __bfloat162float(p0);
            res[2 * i + 1] -= __bfloat162float(p1);
            w[i] = (uint32_t)__bfloat16_as_ushort(p0) | ((uint32_t)__bfloat16_as_ushort(p1) << 16);
        }
        *reinterpret_cast<uint4*>(dst[pc]) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

struct StepArgs {
    const __nv_bfloat16* op_in;   // [tiles][K / 64 chunks][NP pieces][8192] message operand of this step (previous step's result)
    __nv_bfloat16* op_out;        // same layout: message operand of the next step
    const __nv_bfloat16* tbl_img; // [K / NT slices][K / 64 chunks][NP pieces][NT x 64] table slices, rows = output states
    const float* emis_n;          // [M symbols][K]
    const uint8_t* obs_t;         // [B] symbols of this time step
    float* raw_out;               // [B][K] this step's unnormalised result (FWD: forward message, BWD: fwd * bwd)
    float* raw_prev;              // [B][K] previous step's unnormalised result, normalised in place by this launch (or null)
    const float* fwd_t;           // BWD: [B][K] normalised forward message of this time step
    const float* part_in;         // [2 (carried, result)][K / 64][Bpad] row sums of the previous step, per slice
    float* part_out;              // same, of this step
    int B, Bpad, K, n_sym;
    long long* trace;             // tuning aid (CXB_HMM_TC_TRACE=1): per-CTA clock64 stamps of the pipeline events, else null
};
__device__ __forceinline__ void stamp(const StepArgs& a, int slot) {
    if (a.trace) a.trace[(size_t)((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 16 + slot] = clock64();
}

// rows [m][n0 .. n0 + 63] of a [B][K] fp32 plane: 16 independent 128-bit accesses per thread (one round trip)
__device__ __forceinline__ void load_row64(const float* p, float4 (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = reinterpret_cast<const float4*>(p)[i];
}

template <bool FWD, int NT>
__device__ __forceinline__ void hmm_tc_step_body(const StepArgs& a) {
    constexpr int N_TILE = NT, STAGES = Cfg<NT>::STAGES;
    constexpr uint32_t B_CHUNK_BYTES = Cfg<NT>::B_CHUNK_BYTES, STAGE_BYTES = Cfg<NT>::STAGE_BYTES, TMEM_COLS = Cfg<NT>::TMEM_COLS;
    constexpr int LPR = N_TILE / 4, RPI = 32 / LPR, ITER = 32 / RPI;  // lanes per row, rows per instruction, iterations per warp
    extern __shared__ __align__(128) unsigned char smem[];
    const int n_chunks = a.K / K_CHUNK;
    unsigned char* ring = smem;  // [STAGES][message hi | message lo | table hi | table lo]
    float* s_em = reinterpret_cast<float*>(ring + (size_t)STAGES * STAGE_BYTES);  // [n_sym][64]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_em + (size_t)a.n_sym * N_TILE);
    uint64_t* full = bars;                      // [STAGES]
    uint64_t* empty = bars + STAGES;            // [STAGES]
    uint64_t* accum = bars + 2 * STAGES;        // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x, slice = blockIdx.y, n0 = slice * N_TILE;
    if (threadIdx.x == 0) stamp(a, 0);
    // programmatic dependent launch: the next step's grid may be scheduled now (its CTAs set up their barriers and TMEM on
    // idle SMs and then block in griddepcontrol.wait until THIS grid has completed and flushed)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(smem_u32(&full[s]), 1);
            mbar_init(smem_u32(&empty[s]), 1);
        }
        mbar_init(smem_u32(accum), 2);  // both issuers commit
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {  // TMEM: NP blocks of NT fp32 columns x 128 lanes for the accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    asm volatile("griddepcontrol.wait;" ::: "memory");  // everything below reads what the previous step's grid wrote
    if (threadIdx.x == 0) stamp(a, 1);

    if (warp == 4) {
        // ===== producer: bulk copies of the table slice and of the streamed message operand (ONE thread, chunks in order: a
        // waiter on an mbarrier may be at most one phase behind it, which two producers sharing three stages would not be) =====
        if (lane == 0) {
            const __nv_bfloat16* tb = a.tbl_img + (size_t)slice * NP * n_chunks * (B_CHUNK_BYTES / 2);
            const __nv_bfloat16* op = a.op_in + (size_t)tile * NP * n_chunks * (A_CHUNK_BYTES / 2);
            for (int c = 0; c < n_chunks; ++c) {
                const int s = c % STAGES;
                const uint32_t st = smem_u32(ring + (size_t)s * STAGE_BYTES), bar = smem_u32(&full[s]);
                mbar_wait(smem_u32(&empty[s]), ((c / STAGES) & 1) ^ 1);
                mbar_expect_tx(bar, STAGE_BYTES);
                // the NP pieces of a chunk are contiguous in global memory (message: [tile][chunk][piece], table: [slice][chunk][piece])
                // and in the stage: ONE bulk copy per operand and stage. The copy engine of an SM moves a 60 KB stage at
                // 98 B/clk as one copy but at 55 B/clk as six (profiles/r02_bulk_ingest.log) - the ingest is what a step waits on.
                bulk_g2s(st, op + (size_t)c * NP * (A_CHUNK_BYTES / 2), NP * A_CHUNK_BYTES, bar);
                bulk_g2s(st + NP * A_CHUNK_BYTES, tb + (size_t)c * NP * (B_CHUNK_BYTES / 2), NP * B_CHUNK_BYTES, bar);
            }
            stamp(a, 2);
        }
    } else if (warp == 5 || warp == 6) {
        // ===== MMA issuers: one thread each, its own accumulator set. A STAGE belongs to one issuer (even stages: issuer 0,
        // odd stages: issuer 1), so the only waiter of a stage's mbarrier sees every one of its phases (a parity wait cannot
        // tell phases two apart) =====
        if (lane == 0) {
            const int me = warp - 5;
            const uint32_t tmem_set = tmem_base + (uint32_t)me * Cfg<NT>::SET_COLS;
            bool first = true;
            for (int c = 0; c < n_chunks; ++c) {
                const int s = c % STAGES;
                if ((s & 1) != me) continue;
                mbar_wait(smem_u32(&full[s]), (c / STAGES) & 1);
                if (c == 0) stamp(a, 3);
                if (c == n_chunks - 1) stamp(a, 4);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_base = smem_u32(ring + (size_t)s * STAGE_BYTES), b_base = a_base + NP * A_CHUNK_BYTES;
#pragma unroll
                for (int ks = 0; ks < K_CHUNK / 16; ++ks) {
                    const uint32_t off = ks * 2 * LBO;  // 16 input states = 2 core matrices along K
#pragma unroll
                    for (int pa = 0; pa < NP; ++pa)  // message piece pa x table pieces 0 .. NP-1-pa (one operand of (NP - pa) NT rows)
                        umma_bf16(tmem_set, smem_desc(a_base + pa * A_CHUNK_BYTES + off), smem_desc(b_base + off),
                                  Cfg<NT>::idesc((uint32_t)((NP - pa) * NT)), !first || (ks != 0) || (pa != 0));
                }
                first = false;
                umma_commit(smem_u32(&empty[s]));  // frees the stage when these MMAs have read it
            }
            umma_commit(smem_u32(accum));
            if (me == 0) stamp(a, 5);
        }
    } else {
        // ===== epilogue warps =====
        // Arithmetic is done with thread = one chain (TMEM lane) x the 64 output states of the slice; every [B][K] fp32
        // plane is touched with HALF A WARP PER ROW (16 lanes x 16 bytes = the row's 256 contiguous bytes), per-row scalars
        // travel by shuffle and the tile goes through a shared-memory staging buffer (the operand ring, idle by then).
        const int row = warp * 32 + lane;            // TMEM lane / row of the tile
        const int m = tile * M_TILE + row;           // chain
        const bool live = m < a.B;
        const int hrow = lane / LPR, c4 = lane % LPR;  // cooperative phase: rows 32 warp + RPI it + hrow, float4 column c4
        for (int x = threadIdx.x; x < a.n_sym * N_TILE; x += 128)
            s_em[x] = a.emis_n[(size_t)(x / N_TILE) * a.K + n0 + (x % N_TILE)];
        const int n_slices = a.K / N_TILE;
        float tot_c = 0.0f, tot_r = 0.0f;
        for (int j = 0; j < n_slices; ++j) {
            tot_c += a.part_in[(size_t)(0 * n_slices + j) * a.Bpad + m];
            tot_r += a.part_in[(size_t)(1 * n_slices + j) * a.Bpad + m];
        }
        const float r = live ? pow2_inv(tot_c) : 0.0f;
        const float q_prev = rcp_nr(tot_r);
        // the previous step's rows leave exactly normalised (in place), while the MMAs of this step run
        if (a.raw_prev) {
            float4 pv[ITER];
#pragma unroll
            for (int it = 0; it < ITER; ++it) {
                const int mm = tile * M_TILE + warp * 32 + RPI * it + hrow;
                if (mm < a.B) pv[it] = reinterpret_cast<const float4*>(a.raw_prev + (size_t)mm * a.K + n0)[c4];
            }
#pragma unroll
            for (int it = 0; it < ITER; ++it) {
                const int mm = tile * M_TILE + warp * 32 + RPI * it + hrow;
                const float q = __shfl_sync(0xffffffffu, q_prev, RPI * it + hrow);
                if (mm < a.B)
                    reinterpret_cast<float4*>(a.raw_prev + (size_t)mm * a.K + n0)[c4] =
                        make_float4(pv[it].x * q, pv[it].y * q, pv[it].z * q, pv[it].w * q);
            }
        }
        // backward: this time step's forward message, requested now, used after the accumulator is ready
        float4 fw[ITER];
        if (!FWD) {
#pragma unroll
            for (int it = 0; it < ITER; ++it) {
                const int mm = tile * M_TILE + warp * 32 + RPI * it + hrow;
                fw[it] = !a.fwd_t  ? make_float4(1.f, 1.f, 1.f, 1.f)  // no forward message yet: the prediction itself is stored
                         : mm < a.B ? reinterpret_cast<const float4*>(a.fwd_t + (size_t)mm * a.K + n0)[c4]
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        if (threadIdx.x == 0) stamp(a, 6);
        asm volatile("bar.sync 1, 128;" ::: "memory");  // s_em visible to the 4 epilogue warps
        int o = live ? (int)a.obs_t[m] : 0;
        if (o >= a.n_sym) o = a.n_sym - 1;

        mbar_wait(smem_u32(accum), 0);
        if (threadIdx.x == 0) stamp(a, 7);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // every MMA has completed (accum barrier), so the ring is free: stage[row][0..63] (row stride 68 floats) takes the
        // accumulator rows (thread = TMEM lane), everything else happens half a warp per row
        constexpr int SROW = N_TILE + 4;
        constexpr int PSTR = LPR + 4;  // row stride of the partial sums: 128-bit reads of 8 consecutive rows hit 8 different bank groups
        float* stage = reinterpret_cast<float*>(ring);
        float* s_sum = stage + (size_t)M_TILE * SROW;  // [2 (carried, result)][128 rows][PSTR]
#pragma unroll
        for (int half = 0; half < N_TILE / 32; ++half) {
            float pred[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) pred[i] = 0.0f;
#pragma unroll
            for (int set = 0; set < 2; ++set) {  // the accumulator blocks of one issuer's set are requested together
                uint32_t blkv[NP][32];
#pragma unroll
                for (int blk = 0; blk < NP; ++blk)
                    tmem_ld32_issue(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)set * Cfg<NT>::SET_COLS + (uint32_t)(blk * N_TILE + half * 32), blkv[blk]);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float acc = __uint_as_float(blkv[NP - 1][i]);  // small to large
#pragma unroll
                    for (int blk = NP - 2; blk >= 0; --blk) acc += __uint_as_float(blkv[blk][i]);
                    pred[i] += acc;
                }
            }
            float4* srow = reinterpret_cast<float4*>(stage + (size_t)row * SROW + half * 32);
#pragma unroll
            for (int i = 0; i < 8; ++i) srow[i] = make_float4(pred[4 * i], pred[4 * i + 1], pred[4 * i + 2], pred[4 * i + 3]);
        }
        __syncwarp();  // a warp only re-reads the 32 staging rows it wrote itself
        // this slice is columns [n0, n0 + NT) of K: chunk n0 / 64 of the next step's message operand, offset n0 % 64 inside it
        __nv_bfloat16* op_pc[NP];
#pragma unroll
        for (int pc = 0; pc < NP; ++pc)
            op_pc[pc] = a.op_out + ((size_t)tile * NP * n_chunks + (size_t)(n0 / K_CHUNK) * NP + pc) * (A_CHUNK_BYTES / 2);
#pragma unroll
        for (int it = 0; it < ITER; ++it) {
            const int src = RPI * it + hrow, rr = warp * 32 + src, mm = tile * M_TILE + rr;
            const int o_r = __shfl_sync(0xffffffffu, o, src);
            const float r_r = __shfl_sync(0xffffffffu, r, src);  // 0 for the padding rows of the last tile
            const float4 pd = *reinterpret_cast<const float4*>(stage + (size_t)rr * SROW + c4 * 4);
            const float4 e4 = *reinterpret_cast<const float4*>(s_em + o_r * N_TILE + c4 * 4);
            const float4 cr = make_float4(e4.x * pd.x * r_r, e4.y * pd.y * r_r, e4.z * pd.z * r_r, e4.w * pd.w * r_r);  // carried message
            float4 res = cr;  // forward: the result IS the carried message; backward: fwd * pred
            if (!FWD) res = make_float4(pd.x * fw[it].x, pd.y * fw[it].y, pd.z * fw[it].z, pd.w * fw[it].w);
            // row sums: the lane's 4-column partials go to shared memory and ONE lane per row adds them up after the loop
            // (no shuffle chain per row on the path of the stores; the sums leave as one coalesced line per warp)
            s_sum[(size_t)rr * PSTR + c4] = (cr.x + cr.y) + (cr.z + cr.w);
            if (!FWD) s_sum[(size_t)(M_TILE + rr) * PSTR + c4] = (res.x + res.y) + (res.z + res.w);
            if (mm < a.B) reinterpret_cast<float4*>(a.raw_out + (size_t)mm * a.K + n0)[c4] = res;
            // next step's message operand in the canonical UMMA layout (this slice = chunk `slice` of K): 4 states = 8 bytes
            // per lane; two rows x two lanes fill whole 32-byte sectors
            float res4[4] = {cr.x, cr.y, cr.z, cr.w};  // residuals: piece k = bf16(what pieces 0 .. k-1 left over)
            const uint32_t e = chunk_elem((uint32_t)rr, (uint32_t)(n0 % K_CHUNK + c4 * 4));
#pragma unroll
            for (int pc = 0; pc < NP; ++pc) {
                uint32_t w[2];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const __nv_bfloat16 p0 = __float2bfloat16_rn(res4[2 * i]), p1 = __float2bfloat16_rn(res4[2 * i + 1]);
                    res4[2 * i] -= __bfloat162float(p0);
                    res4[2 * i + 1] -= __bfloat162float(p1);
                    w[i] = (uint32_t)__bfloat16_as_ushort(p0) | ((uint32_t)__bfloat16_as_ushort(p1) << 16);
                }
                *reinterpret_cast<uint2*>(op_pc[pc] + e) = make_uint2(w[0], w[1]);
            }
        }
        __syncwarp();  // a warp only sums the 32 rows it wrote itself
        {
            float sc = 0.0f, sr = 0.0f;
#pragma unroll
            for (int q = 0; q < LPR / 4; ++q) {
                const float4 x = *reinterpret_cast<const float4*>(s_sum + (size_t)row * PSTR + 4 * q);
                sc += (x.x + x.y) + (x.z + x.w);
                if (!FWD) {
                    const float4 y = *reinterpret_cast<const float4*>(s_sum + (size_t)(M_TILE + row) * PSTR + 4 * q);
                    sr += (y.x + y.y) + (y.z + y.w);
                }
            }
            if (FWD) sr = sc;
            a.part_out[(size_t)(0 * n_slices + slice) * a.Bpad + m] = sc;
            a.part_out[(size_t)(1 * n_slices + slice) * a.Bpad + m] = live ? sr : 0.0f;
        }
        if (threadIdx.x == 0) stamp(a, 8);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) stamp(a, 9);
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
}
// Both passes in ONE launch per step: blockIdx.z = 0 runs step s of the forward pass (time s), blockIdx.z = 1 step s of the
// backward pass (time T-1-s). The two recursions are independent, so a launch holds twice the CTAs (2 x 64 at B = 1,024,
// K = 512, NT = 64: every SM busy) and the set-up, launch gap and epilogue of one pass hide under the operand ingest of
// the other. The backward half needs the forward message of its time step only for the MARGINAL (fwd * bwd): while the
// forward pass has not reached that time yet (first half of the launches) it is given fwd_t = nullptr, stores the
// normalised backward prediction instead, and k_hmm_tc_combine multiplies the forward message in afterwards.
struct StepArgs2 {
    StepArgs d[2];
};
template <int NT>
__global__ void __launch_bounds__(THREADS, 1) k_hmm_tc_step_pair(const StepArgs2 p) {
    if (blockIdx.z == 0)
        hmm_tc_step_body<true, NT>(p.d[0]);
    else
        hmm_tc_step_body<false, NT>(p.d[1]);
}
// marginal rows the backward half left as normalised predictions: marg = normalise(fwd * marg), one warp per (time, chain) row
__global__ void k_hmm_tc_combine(const float* __restrict__ fwd, float* __restrict__ marg, long long n_rows, int K) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const int lane = threadIdx.x & 31;
    const float4* f = reinterpret_cast<const float4*>(fwd + (size_t)row * K);
    float4* g = reinterpret_cast<float4*>(marg + (size_t)row * K);
    float sum = 0.0f;
    for (int i = lane; i < K / 4; i += 32) {
        const float4 a = __ldcs(f + i), b = g[i];
        const float4 r = make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w);
        g[i] = r;
        sum += (r.x + r.y) + (r.z + r.w);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
    const float q = rcp_nr(sum);
    for (int i = lane; i < K / 4; i += 32) {
        const float4 r = g[i];
        __stcs(g + i, make_float4(r.x * q, r.y * q, r.z * q, r.w * q));
    }
}

// first step of a pass: carried message = emission message; result = emission (FWD) / forward message (BWD)
template <bool FWD, int NT>
__global__ void k_hmm_tc_init(StepArgs a) {
    constexpr int N_TILE = NT;
    const int m = blockIdx.x * blockDim.x + threadIdx.x;  // chain (padded)
    const int slice = blockIdx.y, n0 = slice * N_TILE, n_chunks = a.K / K_CHUNK, n_slices = a.K / N_TILE;
    if (m >= a.Bpad) return;
    const bool live = m < a.B;
    const int tile = m / M_TILE, row = m % M_TILE;
    int o = live ? (int)a.obs_t[m] : 0;
    if (o >= a.n_sym) o = a.n_sym - 1;
    float sum_c = 0.0f, sum_r = 0.0f;
    for (int k0 = 0; k0 < N_TILE; k0 += 8) {
        float c[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            c[i] = live ? a.emis_n[(size_t)o * a.K + n0 + k0 + i] : 0.0f;
            sum_c += c[i];
            if (live) {
                const float res = FWD ? c[i] : a.fwd_t ? a.fwd_t[(size_t)m * a.K + n0 + k0 + i] : 1.0f;
                a.raw_out[(size_t)m * a.K + n0 + k0 + i] = res;
                sum_r += res;
            }
        }
        const uint32_t e = chunk_elem((uint32_t)row, (uint32_t)(n0 % K_CHUNK + k0));
        __nv_bfloat16* dst[NP];
#pragma unroll
        for (int pc = 0; pc < NP; ++pc)
            dst[pc] = a.op_out + ((size_t)tile * NP * n_chunks + (size_t)(n0 / K_CHUNK) * NP + pc) * (A_CHUNK_BYTES / 2) + e;
        split_store8(c, dst);
    }
    a.part_out[(size_t)(0 * n_slices + slice) * a.Bpad + m] = sum_c;
    a.part_out[(size_t)(1 * n_slices + slice) * a.Bpad + m] = sum_r;
}
// last step of a pass: nothing follows, so its result is normalised here
__global__ void k_hmm_tc_finish(float* raw, const float* part, int B, int Bpad, int K, int n_slices) {
    const int m = blockIdx.x;
    if (m >= B) return;
    float tot = 0.0f;
    for (int j = 0; j < n_slices; ++j) tot += part[(size_t)(1 * n_slices + j) * Bpad + m];
    const float q = rcp_nr(tot);
    for (int n = threadIdx.x; n < K; n += blockDim.x) raw[(size_t)m * K + n] *= q;
}

template <int NT>
inline size_t step_smem_bytes(int n_sym) {
    return (size_t)Cfg<NT>::STAGES * Cfg<NT>::STAGE_BYTES + (size_t)n_sym * NT * sizeof(float) +
           (2 * Cfg<NT>::STAGES + 1) * sizeof(uint64_t) + 16;
}

// host: bf16 round-to-nearest-even of a float
inline uint16_t bf16_rn_host(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);  // NaN
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
inline float bf16_to_float_host(uint16_t h) {
    uint32_t u = (uint32_t)h << 16;
    float x;
    memcpy(&x, &u, 4);
    return x;
}
// table image: rows[n][k] (n = output state, k = input state), fp32 -> [slice][chunk][piece][NT x 64] in the canonical layout
inline void build_table_image(const float* rows, int K, int N_TILE, std::vector<uint16_t>& img) {
    const int n_chunks = K / K_CHUNK, n_slices = K / N_TILE;
    const size_t B_CHUNK_BYTES = (size_t)N_TILE * K_CHUNK * 2;
    img.assign((size_t)n_slices * NP * n_chunks * (B_CHUNK_BYTES / 2), 0);
    for (int n = 0; n < K; ++n)
        for (int k = 0; k < K; ++k) {
            float res = rows[(size_t)n * K + k];
            const int slice = n / N_TILE, r = n % N_TILE, c = k / K_CHUNK, kk = k % K_CHUNK;
            const size_t base = (size_t)slice * NP * n_chunks * (B_CHUNK_BYTES / 2);
            for (int pc = 0; pc < NP; ++pc) {
                const uint16_t piece = bf16_rn_host(res);
                res -= bf16_to_float_host(piece);
                img[base + (size_t)(c * NP + pc) * (B_CHUNK_BYTES / 2) + chunk_elem(r, kk)] = piece;
            }
        }
}

}  // namespace tc
}  // namespace cxb
