// hmm.cu — structured engine for a batch of discrete HMMs (BASELINE config 3).
//
// Graph per chain (SURVEY Appendix C): hidden z_t, observed y_t, emission factor (z_t, y_t), transition factor
// (z_t, z_{t+1}), uniform prior leaf on z_1; data enter as set_value!(m2f(y_t, em_t), o_t).  One call =
// update_marginals!(engine, z[1:T]) of every chain = 6T-4 message updates per chain (categorical sum-product,
// every message normalised to sum 1).  Materialised in HBM: the forward message m2f(z_t, tr_t) and the marginal
// ("forward message + marginal" contract of SURVEY §8d: 12K+2 bytes per (chain, step)).
//
// Kernel shape: the recursion over t is strictly sequential, the batch is small (1,024 chains), so the unit of
// parallelism is ONE WARP PER CHAIN with lane l owning states l, l+32, ...:
//   out[j] = sum_i Tbl[i][j] * v[i]        (Tbl = A forward, A^T backward)
// For K <= 64 (fp32) the lane's columns of Tbl live in REGISTERS (2 x 64 values), v is staged in a per-warp
// shared-memory line and read back with broadcast 128-bit loads, so a step is K*K/32 FFMAs + K/4 LDS per warp
// and no block-level barrier.  Larger K stream Tbl through shared memory in row tiles shared by the 8 chains of
// the CTA.
// Which kernel runs (Hmm::launch_t; tests/test_hmm_widths.py keeps a copy of the rule):
//   * fp32, K = 64 -> k_hmm64_pass, the emission table in shared memory for M <= 128, else read from global memory;
//   * fp32, K >= 128 a multiple of 64, M <= 64 -> the tcgen05 path of hmm_tc.cuh (k_hmm_tc_step_pair<NT>, NT = 32 or 64);
//   * K = 32 -> k_hmm_pass with the table in registers;
//   * every other (K, dtype, M), and CXB_HMM_NO_TC=1 -> k_hmm_pass with the table in shared memory: whole when it fits,
//     else streamed in row tiles; the emission table sits in shared memory when it and one table row fit in 200 KiB next
//     to the staging, else in global memory.  Every shape cxb_hmm_create accepts (2 <= K <= 1024, 1 <= M <= 256) runs.
// cxb_hmm_set_observations refuses a symbol >= M, so the kernels' clamp of o to M - 1 never changes a value.
#include <algorithm>
#include <cmath>
#include <type_traits>

#include <cstring>

#include "common.cuh"
#include "hmm_tc.cuh"

namespace cxb {

constexpr int HMM_WARPS = 8;  // chains per CTA

template <class T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One pass over time. FWD: t ascending, writes fwd[t] = m2f(z_t, tr_t) = normalise(em_t * pred_t).
// BWD: t descending, reads fwd[t], writes marg[t] = normalise(fwd[t] * bwd_t), carries
// m2f(z_t, tr_{t-1}) = normalise(em_t * bwd_t).  tbl is A (FWD) or A^T (BWD), row-major [K][K];
// emis_n is the column-normalised emission table transposed to [M][K] (m2v(z_t, em_t) = emis_n[o_t]), staged in
// shared memory (EM_SMEM) or, when it does not fit next to a table row, read from global memory (<= 2 MB, L2-resident).
// Nothing on the per-step critical path waits on global memory: observations are fetched 32 steps at a
// time (one per lane, broadcast by shuffle, double buffered), the forward message of the next step is already in
// registers and the one 8 steps ahead is being pulled into L2 (prefetch.global.L2).
template <class T, int K, bool REGA, bool FWD, bool EM_SMEM>
__global__ void __launch_bounds__(HMM_WARPS * 32)
k_hmm_pass(const T* __restrict__ tbl, const T* __restrict__ emis_n, const uint8_t* __restrict__ obs, T* __restrict__ fwd,
           T* __restrict__ marg, long long B, long long Tn, int Kdyn, int n_sym, int tile_rows) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int Kk = REGA ? K : Kdyn;
    constexpr int CPL_MAX = REGA ? K / 32 : 32;  // states per lane (<= 1024 states in the streamed path)
    const int cpl = (Kk + 31) / 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long b = (long long)blockIdx.x * HMM_WARPS + warp;
    const bool live = b < B;
    const long long bb = live ? b : 0;
    T* sh_v = reinterpret_cast<T*>(smem_raw) + (size_t)warp * Kk;            // per-warp staging of v
    T* sh_em = reinterpret_cast<T*>(smem_raw) + (size_t)HMM_WARPS * Kk;        // [M][K] emission messages (EM_SMEM)
    T* sh_tbl = sh_em + (EM_SMEM ? (size_t)n_sym * Kk : 0);                    // streamed path: row tile of tbl

    T areg[REGA ? K : 1][REGA ? K / 32 : 1];
    if (REGA) {
#pragma unroll
        for (int i = 0; i < K; ++i)
#pragma unroll
            for (int c = 0; c < K / 32; ++c) areg[i][c] = tbl[(size_t)i * K + lane + 32 * c];
    }
    if (EM_SMEM)
        for (int x = threadIdx.x; x < n_sym * Kk; x += blockDim.x) sh_em[x] = emis_n[x];
    const bool whole_table = !REGA && tile_rows >= Kk;
    if (whole_table)
        for (int x = threadIdx.x; x < Kk * Kk; x += blockDim.x) sh_tbl[x] = tbl[x];
    __syncthreads();

    auto time_of = [&](long long step) { return FWD ? step : Tn - 1 - step; };
    auto load_obs_block = [&](long long step0) -> int {  // lane l fetches the symbol of step0 + l
        long long st = step0 + lane;
        return (st < Tn) ? (int)obs[(size_t)time_of(st) * B + bb] : 0;
    };
    int obs_cur = 0, obs_next = load_obs_block(0);

    T v[CPL_MAX];  // carried message (lane's states)
#pragma unroll
    for (int c = 0; c < CPL_MAX; ++c) v[c] = T(0);
    T a_next[CPL_MAX];  // BWD: forward message of the upcoming step
#pragma unroll
    for (int c = 0; c < CPL_MAX; ++c) {
        int j = lane + 32 * c;
        a_next[c] = (!FWD && c < cpl && j < Kk) ? __ldcs(&fwd[((size_t)time_of(0) * B + bb) * Kk + j]) : T(0);
    }

    for (long long step = 0; step < Tn; ++step) {
        const long long t = time_of(step);
        if ((step & 31) == 0) {
            obs_cur = obs_next;
            obs_next = load_obs_block(step + 32);
        }
        int o = __shfl_sync(0xffffffffu, obs_cur, (int)(step & 31));
        if (o >= n_sym) o = n_sym - 1;
        T a[CPL_MAX];
        if (!FWD) {
#pragma unroll
            for (int c = 0; c < CPL_MAX; ++c) a[c] = a_next[c];
            if (step + 1 < Tn) {
                const T* nx = &fwd[((size_t)time_of(step + 1) * B + bb) * Kk];
#pragma unroll
                for (int c = 0; c < CPL_MAX; ++c) {
                    int j = lane + 32 * c;
                    if (c < cpl && j < Kk) a_next[c] = __ldcs(nx + j);
                }
            }
            if (step + 8 < Tn) {
                const T* far = &fwd[((size_t)time_of(step + 8) * B + bb) * Kk];
                if (lane * 32 < Kk * (int)sizeof(T)) asm volatile("prefetch.global.L2 [%0];" ::"l"(far + lane * (32 / sizeof(T))));
            }
        }
        T out[CPL_MAX];
#pragma unroll
        for (int c = 0; c < CPL_MAX; ++c) out[c] = T(0);
        const bool has_prev = step > 0;
        if (has_prev) {
            // stage v, then out[j] = sum_i tbl[i][j] v[i]
            __syncwarp();
#pragma unroll
            for (int c = 0; c < CPL_MAX; ++c)
                if (c < cpl && lane + 32 * c < Kk) sh_v[lane + 32 * c] = v[c];
            __syncwarp();
            if (REGA) {
                T acc[REGA ? K / 32 : 1][4];  // 4 independent FMA chains per column
#pragma unroll
                for (int c = 0; c < K / 32; ++c)
#pragma unroll
                    for (int u = 0; u < 4; ++u) acc[c][u] = T(0);
#pragma unroll
                for (int i = 0; i < K; i += 4) {
                    T vi[4];
                    if (sizeof(T) == 4) {
                        float4 q = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(sh_v) + i);
                        vi[0] = q.x; vi[1] = q.y; vi[2] = q.z; vi[3] = q.w;
                    } else {
#pragma unroll
                        for (int u = 0; u < 4; ++u) vi[u] = sh_v[i + u];
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int c = 0; c < K / 32; ++c) acc[c][u] = fma(areg[i + u][c], vi[u], acc[c][u]);
                }
#pragma unroll
                for (int c = 0; c < K / 32; ++c) out[c] = (acc[c][0] + acc[c][1]) + (acc[c][2] + acc[c][3]);
            } else if (whole_table) {
                for (int i = 0; i < Kk; ++i) {
                    T vi = sh_v[i];
#pragma unroll 4
                    for (int c = 0; c < cpl; ++c) {
                        int j = lane + 32 * c;
                        if (j < Kk) out[c] = fma(sh_tbl[(size_t)i * Kk + j], vi, out[c]);
                    }
                }
            } else {
                for (int r0 = 0; r0 < Kk; r0 += tile_rows) {
                    int nr = min(tile_rows, Kk - r0);
                    __syncthreads();
                    for (int x = threadIdx.x; x < nr * Kk; x += blockDim.x) sh_tbl[x] = tbl[(size_t)r0 * Kk + x];
                    __syncthreads();
                    for (int i = 0; i < nr; ++i) {
                        T vi = sh_v[r0 + i];
#pragma unroll 4
                        for (int c = 0; c < cpl; ++c) {
                            int j = lane + 32 * c;
                            if (j < Kk) out[c] = fma(sh_tbl[(size_t)i * Kk + j], vi, out[c]);
                        }
                    }
                }
            }
        }
        // emission message of this step
        T em[CPL_MAX];
#pragma unroll
        for (int c = 0; c < CPL_MAX; ++c) {
            int j = lane + 32 * c;
            em[c] = (c < cpl && j < Kk) ? (EM_SMEM ? sh_em[(size_t)o * Kk + j] : __ldg(&emis_n[(size_t)o * Kk + j])) : T(0);
        }
        const size_t base = ((size_t)t * B + bb) * Kk;
        if (FWD) {
            // m2f(z_t, tr_t) = normalise(em * pred); at t = 0 the uniform prior leaves normalise(em)
            T part = T(0);
#pragma unroll
            for (int c = 0; c < CPL_MAX; ++c) {
                v[c] = has_prev ? em[c] * out[c] : em[c];
                part += v[c];
            }
            T tot = warp_sum(part);
#pragma unroll
            for (int c = 0; c < CPL_MAX; ++c) {
                v[c] = v[c] / tot;
                int j = lane + 32 * c;
                if (live && c < cpl && j < Kk) __stcs(&fwd[base + j], v[c]);
            }
        } else {
            T part = T(0), part2 = T(0);
#pragma unroll
            for (int c = 0; c < CPL_MAX; ++c) {
                T g = has_prev ? a[c] * out[c] : a[c];    // marginal = fwd * bwd
                T m = has_prev ? em[c] * out[c] : em[c];  // m2f(z_t, tr_{t-1}) = em * bwd
                a[c] = g;
                v[c] = m;
                part += g;
                part2 += m;
            }
            T tot = warp_sum(part), tot2 = warp_sum(part2);
#pragma unroll
            for (int c = 0; c < CPL_MAX; ++c) {
                int j = lane + 32 * c;
                v[c] = v[c] / tot2;
                if (live && c < cpl && j < Kk) __stcs(&marg[base + j], a[c] / tot);
            }
        }
    }
}

// ---- K = 64, fp32: one warp per chain, one warp per CTA (1,024 CTAs = 6.9 per SM for config 3) ------------------------------
// The 64 x 64 table lives in registers: lane (jg = lane / 2, ig = lane % 2) owns the 4 x 32 tile
// tbl[32 ig .. 32 ig + 31][4 jg .. 4 jg + 3] as 64 packed pairs and does 64 FFMA2 (fma.rn.f32x2) per step; the carried
// message is read back with eight conflict-free 128-bit shared loads; the two i-halves are combined by a 2-shuffle
// transpose-reduce that leaves output states (2 lane, 2 lane + 1) in the lane, so messages move as one float2 per lane
// (256 contiguous bytes per warp).  Nothing but the matvec is on the per-step critical path: the carried message is NOT
// normalised exactly, it is scaled by the power of two 2^-floor(log2 sum(u_{s-1})) (exact, keeps sum(u_s) within
// [n_s, 2 n_s), n_s = the true normaliser), and the exactly normalised message / marginal of step s-1
// (u_{s-1} / sum(u_{s-1})) is written one step late, while the matvec of step s is in flight.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}
// branch-free reciprocal (MUFU.RCP + one Newton step, <= 1 ulp for the normal, positive sums it is used on): __frcp_rn
// carries a slow-path call that would split the step into basic blocks and serialise the shuffle chain with the matvec
__device__ __forceinline__ float hmm_rcp(float x) {
    float q;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(q) : "f"(x));
    return fmaf(q, fmaf(-x, q, 1.0f), q);
}
__device__ __forceinline__ float hmm_pow2_inv(float s) {
    unsigned e = (__float_as_uint(s) >> 23) & 0xffu;
    return __uint_as_float((254u - e) << 23);
}
template <bool FWD, bool EM_SMEM>
__global__ void __launch_bounds__(256)
k_hmm64_pass(const float* __restrict__ tbl, const float* __restrict__ emis_n, const uint8_t* __restrict__ obs,
             float* __restrict__ fwd, float* __restrict__ marg, long long B, long long Tn, int n_sym) {
    constexpr int K = 64, LOOK = 4, VS = 72;  // VS: the second half of the message is shifted by 4 banks
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    float* sh_v = reinterpret_cast<float*>(smem_raw) + warp * 2 * VS;  // [2][VS] carried message, double buffered
    float* sh_em = reinterpret_cast<float*>(smem_raw) + n_warps * 2 * VS;  // [M][64] emission messages (if they fit)
    const int lane = threadIdx.x & 31, jg = lane >> 1, ig = lane & 1;
    const long long b = (long long)blockIdx.x * n_warps + warp;
    float2 a2[4][16];  // a2[jj][ip] = (tbl[32 ig + 2 ip][4 jg + jj], tbl[32 ig + 2 ip + 1][4 jg + jj])
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
        for (int ip = 0; ip < 16; ++ip) {
            const int j = 4 * jg + jj, i = 32 * ig + 2 * ip;
            a2[jj][ip] = make_float2(tbl[(size_t)i * K + j], tbl[(size_t)(i + 1) * K + j]);
        }
    if (EM_SMEM) {
        for (int x = threadIdx.x; x < n_sym * K; x += blockDim.x) sh_em[x] = emis_n[x];
        __syncthreads();
    }
    if (b >= B) return;  // whole warps leave; nothing below synchronises across warps
    const int my_slot = 2 * lane + 4 * (lane >> 4);  // where states (2 lane, 2 lane + 1) live in sh_v

    auto time_of = [&](long long step) { return FWD ? step : Tn - 1 - step; };
    auto load_obs_block = [&](long long step0) -> int {  // lane l fetches the symbol of step0 + l
        long long st = step0 + lane;
        return (st < Tn) ? (int)obs[(size_t)time_of(st) * B + b] : 0;
    };
    auto fwd_at = [&](long long step) -> float2 {  // BWD: forward message of `step` for this lane's two states
        return (step < Tn) ? __ldcs(reinterpret_cast<const float2*>(&fwd[((size_t)time_of(step) * B + b) * K]) + lane)
                           : make_float2(0.0f, 0.0f);
    };
    int obs_cur = 0, obs_next = load_obs_block(0);
    float2 a_cur[LOOK], a_nxt[LOOK];
#pragma unroll
    for (int u = 0; u < LOOK; ++u) {
        a_cur[u] = make_float2(0.0f, 0.0f);
        a_nxt[u] = FWD ? make_float2(0.0f, 0.0f) : fwd_at(u);
    }
    float2 u1 = make_float2(0.0f, 0.0f);  // carried message of the previous step (scaled, not normalised)
    float2 ring[LOOK];                      // what steps s-1 .. s-4 leave behind (FWD: the message, BWD: fwd * bwd)
#pragma unroll
    for (int u = 0; u < LOOK; ++u) ring[u] = make_float2(0.0f, 0.0f);
    float p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;  // butterfly partial sums in flight (one level per step)

    // One step. GEN = false is the steady state (4 <= s < Tn): straight-line code.
    //  * scale: r = 2^-floor(log2 max(u_{s-1})) from ONE warp-wide redux.sync.max.f32 (exact scaling, bounded range);
    //  * exact sums for the write-out are a software-pipelined butterfly: every step issues the five shuffles of five
    //    different ages (no dependent shuffle chain inside a step), so the value of step s-4 leaves, exactly
    //    normalised, during step s.
    auto step = [&](auto gen_tag, long long s, int slot, float2 a_now) {
        constexpr bool GEN = decltype(gen_tag)::value;
        int o = __shfl_sync(0xffffffffu, obs_cur, (int)(s & 31));
        if (o >= n_sym) o = n_sym - 1;
        const float2 em = EM_SMEM ? *reinterpret_cast<const float2*>(sh_em + o * K + 2 * lane)
                                  : __ldg(reinterpret_cast<const float2*>(emis_n + (size_t)o * K) + lane);
        float mx;
        {
            const float lm = fmaxf(u1.x, u1.y);
            asm("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(mx) : "f"(lm));
        }
        const float r = hmm_pow2_inv(mx);
        {   // pipelined butterfly: ring[(s-1)&3] entered at level 1, ring[s&3] (step s-4) completes now
            const float2 x1 = ring[(slot + LOOK - 1) % LOOK];
            const float q1 = x1.x + x1.y;
            const float n1 = q1 + __shfl_xor_sync(0xffffffffu, q1, 16);
            const float n2 = p1 + __shfl_xor_sync(0xffffffffu, p1, 8);
            const float n3 = p2 + __shfl_xor_sync(0xffffffffu, p2, 4);
            const float m4 = p3 + __shfl_xor_sync(0xffffffffu, p3, 2);
            const float tot = m4 + __shfl_xor_sync(0xffffffffu, m4, 1);
            p1 = n1;
            p2 = n2;
            p3 = n3;
            if (!GEN || (s >= LOOK && s - LOOK < Tn)) {
                const float q = hmm_rcp(tot);
                const float2 x4 = ring[slot];
                float* dst = FWD ? fwd : marg;
                __stcs(reinterpret_cast<float2*>(&dst[((size_t)time_of(s - LOOK) * B + b) * K]) + lane,
                       make_float2(x4.x * q, x4.y * q));
            }
        }
        if (!GEN || s < Tn) {
            float2 val = make_float2(1.0f, 1.0f);
            if (!GEN || s > 0) {
                const float4* vp = reinterpret_cast<const float4*>(sh_v + (s & 1) * VS + 36 * ig);
                float4 v4[8];  // the whole half-message first: 8 independent 128-bit shared loads in flight
#pragma unroll
                for (int q = 0; q < 8; ++q) v4[q] = vp[q];
                float2 c[4], e[4];  // 8 independent FFMA2 chains
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) c[jj] = e[jj] = make_float2(0.0f, 0.0f);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float2 lo = make_float2(v4[q].x, v4[q].y), hi = make_float2(v4[q].z, v4[q].w);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) c[jj] = ffma2(a2[jj][2 * q], lo, c[jj]);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) e[jj] = ffma2(a2[jj][2 * q + 1], hi, e[jj]);
                }
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) c[jj] = make_float2(c[jj].x + e[jj].x, c[jj].y + e[jj].y);
                // transpose-reduce over the two i-halves: lane ig keeps states 2 ig, 2 ig + 1 of its j-group
                const float acc0 = c[0].x + c[0].y, acc1 = c[1].x + c[1].y, acc2 = c[2].x + c[2].y, acc3 = c[3].x + c[3].y;
                const float keep0 = ig ? acc2 : acc0, keep1 = ig ? acc3 : acc1;
                const float send0 = ig ? acc0 : acc2, send1 = ig ? acc1 : acc3;
                val.x = keep0 + __shfl_xor_sync(0xffffffffu, send0, 1);
                val.y = keep1 + __shfl_xor_sync(0xffffffffu, send1, 1);
            }
            const float2 unew = (!GEN || s > 0) ? make_float2(em.x * val.x * r, em.y * val.y * r) : em;
            ring[slot] = FWD ? unew : make_float2(a_now.x * val.x, a_now.y * val.y);
            *reinterpret_cast<float2*>(sh_v + ((s + 1) & 1) * VS + my_slot) = unew;
            u1 = unew;
            __syncwarp();
        }
    };

    for (long long s0 = 0; s0 < Tn + LOOK; s0 += LOOK) {
        if ((s0 & 31) == 0) {
            obs_cur = obs_next;
            obs_next = load_obs_block(s0 + 32);
        }
        if (!FWD) {
#pragma unroll
            for (int u = 0; u < LOOK; ++u) {
                a_cur[u] = a_nxt[u];
                a_nxt[u] = fwd_at(s0 + LOOK + u);
            }
            if (s0 + 16 < Tn && lane < 2)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(&fwd[((size_t)time_of(s0 + 16) * B + b) * K + 32 * lane]));
        }
        if (s0 >= LOOK && s0 + LOOK <= Tn) {
#pragma unroll
            for (int uu = 0; uu < LOOK; ++uu) step(std::false_type{}, s0 + uu, uu, a_cur[uu]);
        } else {
#pragma unroll
            for (int uu = 0; uu < LOOK; ++uu) step(std::true_type{}, s0 + uu, uu, a_cur[uu]);
        }
    }
}

// cxb_hmm_set_observations' range check: *bad = 1 if any of the n bytes is >= n_sym (< 256). Four bytes per compare
// (__vcmpgeu4), 16 per load; cudaMalloc'd obs is 16-byte aligned, the last n % 16 bytes are read one by one.
__global__ void __launch_bounds__(256) k_hmm_check_obs(const uint8_t* __restrict__ obs, size_t n, int n_sym, int* __restrict__ bad) {
    const unsigned lim = 0x01010101u * (unsigned)n_sym;
    const size_t n16 = n / 16, stride = (size_t)gridDim.x * blockDim.x, tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned any = 0;
    for (size_t i = tid; i < n16; i += stride) {
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(obs) + i);
        any |= __vcmpgeu4(w.x, lim) | __vcmpgeu4(w.y, lim) | __vcmpgeu4(w.z, lim) | __vcmpgeu4(w.w, lim);
    }
    for (size_t i = n16 * 16 + tid; i < n; i += stride) any |= obs[i] >= n_sym;
    if (__syncthreads_or(any != 0) && threadIdx.x == 0) *bad = 1;
}

struct Hmm {
    int device = 0, dtype = CXB_F32, K = 0, M = 0;
    long long B = 0, T = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    DBuf<unsigned char> A, At, En, fwd, marg;
    DBuf<uint8_t> obs;
    DBuf<int> obs_bad;  // flag of k_hmm_check_obs
    // tensor-core path (hmm_tc.cuh): table images (forward: rows of A^T, backward: rows of A), message operands, row sums
    DBuf<uint16_t> tc_img_f, tc_img_b, tc_op[2], tc_op_b[2];  // _b: the backward pass's own ping-pong
    DBuf<float> tc_part[2], tc_part_b[2];
    bool tc_ready = false;
    int tc_nt = 64;  // output states per CTA of the tensor-core step kernel (32 or 64)
    bool tc_eligible() const {
        if (const char* e = getenv("CXB_HMM_NO_TC"))
            if (atoi(e)) return false;
        return dtype == CXB_F32 && K % 64 == 0 && K >= 128 && K <= tc::MAX_K && M <= 64;
    }
    long long tc_bpad() const { return (B + tc::M_TILE - 1) / tc::M_TILE * tc::M_TILE; }
    bool have_tables = false, have_obs = false, ran = false;
    size_t esz() const { return dtype == CXB_F32 ? 4 : 8; }
    ~Hmm() {
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }
    int32_t init() {
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
            err = "no CUDA device available (cortex_b200 has no CPU fallback)";
            return CXB_ERR_CUDA;
        }
        if (device < 0 || device >= count || B <= 0 || T <= 0 || K < 2 || K > 1024 || M < 1 || M > 256) {
            err = "bad device / shape (2 <= states <= 1024, 1 <= symbols <= 256)";
            return CXB_ERR_BAD_ARG;
        }
        CXB_CUDA(cudaSetDevice(device));
        CXB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        CXB_CUDA(cudaEventCreate(&ev0));
        CXB_CUDA(cudaEventCreate(&ev1));
        CXB_CUDA(A.reserve((size_t)K * K * esz()));
        CXB_CUDA(At.reserve((size_t)K * K * esz()));
        CXB_CUDA(En.reserve((size_t)M * K * esz()));
        CXB_CUDA(obs.reserve((size_t)T * B));
        CXB_CUDA(obs_bad.reserve(1));
        CXB_CUDA(fwd.reserve((size_t)T * B * K * esz()));
        CXB_CUDA(marg.reserve((size_t)T * B * K * esz()));
        return CXB_OK;
    }
    void put(std::vector<unsigned char>& raw, size_t i, double v) {
        if (dtype == CXB_F32)
            ((float*)raw.data())[i] = (float)v;
        else
            ((double*)raw.data())[i] = v;
    }
    int32_t set_tables(const double* trans, const double* emis) {
        CXB_CUDA(cudaSetDevice(device));
        std::vector<unsigned char> a((size_t)K * K * esz()), at((size_t)K * K * esz()), en((size_t)M * K * esz());
        for (int i = 0; i < K; ++i)
            for (int j = 0; j < K; ++j) {
                put(a, (size_t)i * K + j, trans[(size_t)i * K + j]);
                put(at, (size_t)j * K + i, trans[(size_t)i * K + j]);
            }
        for (int o = 0; o < M; ++o) {  // m2v(z, em) = normalise(E[:, o]) (HMM_EMIT rule)
            double s = 0;
            for (int j = 0; j < K; ++j) s += emis[(size_t)j * M + o];
            if (!(s > 0)) {
                err = "emission column sums must be positive";
                return CXB_ERR_BAD_ARG;
            }
            for (int j = 0; j < K; ++j) put(en, (size_t)o * K + j, emis[(size_t)j * M + o] / s);
        }
        CXB_CUDA(cudaMemcpyAsync(A.p, a.data(), a.size(), cudaMemcpyHostToDevice, stream));
        CXB_CUDA(cudaMemcpyAsync(At.p, at.data(), at.size(), cudaMemcpyHostToDevice, stream));
        CXB_CUDA(cudaMemcpyAsync(En.p, en.data(), en.size(), cudaMemcpyHostToDevice, stream));
        if (tc_eligible()) {
            // slices of 32 output states when 64-state slices would leave most SMs idle
            int n_sm = 148;
            cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
            // the widest grid that is still resident at once: (chain tiles) x (K / NT slices) x (2 passes) CTAs, one per SM
            tc_nt = (tc_bpad() / tc::M_TILE) * (K / 32) * 2 <= n_sm ? 32 : 64;
            std::vector<uint16_t> img;
            tc::build_table_image((const float*)at.data(), K, tc_nt, img);  // forward: pred[j] = sum_i msg[i] A[i][j] -> rows of A^T
            CXB_CUDA(tc_img_f.reserve(img.size()));
            CXB_CUDA(cudaMemcpyAsync(tc_img_f.p, img.data(), img.size() * 2, cudaMemcpyHostToDevice, stream));
            CXB_CUDA(cudaStreamSynchronize(stream));
            tc::build_table_image((const float*)a.data(), K, tc_nt, img);   // backward: pred[j] = sum_i A[j][i] msg[i] -> rows of A
            CXB_CUDA(tc_img_b.reserve(img.size()));
            CXB_CUDA(cudaMemcpyAsync(tc_img_b.p, img.data(), img.size() * 2, cudaMemcpyHostToDevice, stream));
            const long long bpad = tc_bpad();
            const size_t op_elems = (size_t)(bpad / tc::M_TILE) * tc::NP * (K / tc::K_CHUNK) * (tc::A_CHUNK_BYTES / 2);
            for (int i = 0; i < 2; ++i) {
                CXB_CUDA(tc_op[i].reserve(op_elems));
                CXB_CUDA(tc_part[i].reserve((size_t)2 * (K / tc_nt) * bpad));
                CXB_CUDA(cudaMemsetAsync(tc_op[i].p, 0, op_elems * 2, stream));
                CXB_CUDA(cudaMemsetAsync(tc_part[i].p, 0, (size_t)2 * (K / tc_nt) * bpad * sizeof(float), stream));
                CXB_CUDA(tc_op_b[i].reserve(op_elems));
                CXB_CUDA(tc_part_b[i].reserve((size_t)2 * (K / tc_nt) * bpad));
                CXB_CUDA(cudaMemsetAsync(tc_op_b[i].p, 0, op_elems * 2, stream));
                CXB_CUDA(cudaMemsetAsync(tc_part_b[i].p, 0, (size_t)2 * (K / tc_nt) * bpad * sizeof(float), stream));
            }
            tc_ready = true;
        }
        CXB_CUDA(cudaStreamSynchronize(stream));
        have_tables = true;
        return CXB_OK;
    }
    template <class T, int KK, bool REGA, bool EM_SMEM>
    int32_t launch_pair(int tile_rows, size_t smem) {
        unsigned grid = cdiv((size_t)B, HMM_WARPS);
        if (smem > 48 * 1024) {
            CXB_CUDA(cudaFuncSetAttribute(k_hmm_pass<T, KK, REGA, true, EM_SMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CXB_CUDA(cudaFuncSetAttribute(k_hmm_pass<T, KK, REGA, false, EM_SMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        }
        CXB_LAUNCH((k_hmm_pass<T, KK, REGA, true, EM_SMEM>), grid, HMM_WARPS * 32, smem, stream, (const T*)A.p, (const T*)En.p, obs.p,
                   (T*)fwd.p, (T*)marg.p, B, this->T, K, M, tile_rows);
        CXB_LAUNCH((k_hmm_pass<T, KK, REGA, false, EM_SMEM>), grid, HMM_WARPS * 32, smem, stream, (const T*)At.p, (const T*)En.p, obs.p,
                   (T*)fwd.p, (T*)marg.p, B, this->T, K, M, tile_rows);
        return CXB_OK;
    }
    int32_t launch_tc() { return tc_nt == 32 ? launch_tc_pair_nt<32>() : launch_tc_pair_nt<64>(); }
    // One launch per time step (hmm_tc.cuh): launch s runs step s of BOTH passes (forward at time s, backward at time
    // T-1-s): T + 4 launches. The backward half writes the marginal directly once the forward message of its time step is
    // final (normalised in place by forward launch t+1, i.e. for T-1-s <= s-2); before that it stores the normalised
    // backward prediction and k_hmm_tc_combine multiplies the forward messages in at the end (times >= T - s_direct).
    template <int NT>
    int32_t launch_tc_pair_nt() {
        const int bpad = (int)tc_bpad(), tiles = bpad / tc::M_TILE, n_slices = K / NT;
        const size_t smem = tc::step_smem_bytes<NT>(M), row = (size_t)B * K;
        CXB_CUDA(cudaFuncSetAttribute(tc::k_hmm_tc_step_pair<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        float *fw = (float*)fwd.p, *mg = (float*)marg.p;
        tc::StepArgs2 p{};
        for (int z = 0; z < 2; ++z) {
            p.d[z].emis_n = (const float*)En.p;
            p.d[z].B = (int)B;
            p.d[z].Bpad = bpad;
            p.d[z].K = K;
            p.d[z].n_sym = M;
        }
        p.d[0].tbl_img = (const __nv_bfloat16*)tc_img_f.p;
        p.d[1].tbl_img = (const __nv_bfloat16*)tc_img_b.p;
        const dim3 grid(tiles, n_slices, 2), igrid(bpad / 128, n_slices);
        const long long Tn = this->T, s_direct = (Tn + 2) / 2;  // first launch whose backward half sees a final forward message
        DBuf<long long> trace;
        const bool tracing = getenv("CXB_HMM_TC_TRACE") && atoi(getenv("CXB_HMM_TC_TRACE"));
        const size_t n_cta = (size_t)tiles * n_slices * 2;
        if (tracing) {
            CXB_CUDA(trace.reserve(n_cta * 16));
            CXB_CUDA(cudaMemsetAsync(trace.p, 0, n_cta * 16 * sizeof(long long), stream));
            p.d[0].trace = p.d[1].trace = trace.p;
        }
        for (long long s = 0; s < Tn; ++s) {
            const long long tf = s, tb = Tn - 1 - s;
            tc::StepArgs& f = p.d[0];
            tc::StepArgs& b = p.d[1];
            f.op_in = (const __nv_bfloat16*)tc_op[(s + 1) & 1].p;
            f.op_out = (__nv_bfloat16*)tc_op[s & 1].p;
            f.part_in = tc_part[(s + 1) & 1].p;
            f.part_out = tc_part[s & 1].p;
            f.obs_t = obs.p + (size_t)tf * B;
            f.raw_out = fw + (size_t)tf * row;
            f.raw_prev = s ? fw + (size_t)(tf - 1) * row : nullptr;
            f.fwd_t = nullptr;
            b.op_in = (const __nv_bfloat16*)tc_op_b[(s + 1) & 1].p;
            b.op_out = (__nv_bfloat16*)tc_op_b[s & 1].p;
            b.part_in = tc_part_b[(s + 1) & 1].p;
            b.part_out = tc_part_b[s & 1].p;
            b.obs_t = obs.p + (size_t)tb * B;
            b.raw_out = mg + (size_t)tb * row;
            b.raw_prev = s ? mg + (size_t)(tb + 1) * row : nullptr;
            b.fwd_t = s >= s_direct ? fw + (size_t)tb * row : nullptr;
            if (s == 0) {
                CXB_LAUNCH((tc::k_hmm_tc_init<true, NT>), igrid, 128, 0, stream, f);
                CXB_LAUNCH((tc::k_hmm_tc_init<false, NT>), igrid, 128, 0, stream, b);
            } else {
                cudaLaunchConfig_t cfg{};
                cfg.gridDim = grid;
                cfg.blockDim = dim3(tc::THREADS);
                cfg.dynamicSmemBytes = smem;
                cfg.stream = stream;
                cudaLaunchAttribute attr[1];
                attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                attr[0].val.programmaticStreamSerializationAllowed = s > 1 ? 1 : 0;  // launch 1 follows the two init kernels
                cfg.attrs = attr;
                cfg.numAttrs = 1;
                CXB_CUDA(cudaLaunchKernelEx(&cfg, tc::k_hmm_tc_step_pair<NT>, p));
                ++::cxb::g_kernel_launches;
            }
        }
        CXB_LAUNCH(tc::k_hmm_tc_finish, (unsigned)B, 128, 0, stream, fw + (size_t)(Tn - 1) * row, tc_part[(Tn - 1) & 1].p, (int)B, bpad, K,
                   n_slices);
        CXB_LAUNCH(tc::k_hmm_tc_finish, (unsigned)B, 128, 0, stream, mg, tc_part_b[(Tn - 1) & 1].p, (int)B, bpad, K, n_slices);
        const long long t0 = Tn - std::min(s_direct, Tn), n_rows = (Tn - t0) * B;  // times the backward half ran ahead of the forward pass
        if (n_rows > 0)
            CXB_LAUNCH(tc::k_hmm_tc_combine, (unsigned)((n_rows + 7) / 8), 256, 0, stream, fw + (size_t)t0 * row, mg + (size_t)t0 * row, n_rows, K);
        if (tracing) {  // stamps of the LAST paired launch, averaged over the CTAs of each half, relative to the earliest CTA start
            std::vector<long long> h(n_cta * 16);
            CXB_CUDA(cudaStreamSynchronize(stream));
            CXB_CUDA(cudaMemcpy(h.data(), trace.p, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
            static const char* names[10] = {"start", "init+alloc done", "producer issued all", "mma: first chunk landed", "mma: last chunk landed",
                                            "mma: all issued", "epi: prev normalised", "epi: accumulator ready", "epi: done", "exit"};
            for (int z = 0; z < 2; ++z)
                for (int k = 0; k < 10; ++k) {
                    double acc = 0;
                    const size_t c0 = (size_t)z * tiles * n_slices, c1 = c0 + (size_t)tiles * n_slices;
                    for (size_t c = c0; c < c1; ++c) acc += (double)(h[c * 16 + k] - h[c * 16]);
                    fprintf(stderr, "cxb_hmm tc trace (%s half): %-26s %8.0f cycles after the CTA's own start\n", z ? "backward" : "forward", names[k],
                            acc / (tiles * n_slices));
                }
        }
        return CXB_OK;
    }
    int32_t launch_k64() {
        // one warp per chain; warps per CTA chosen so that one CTA per SM holds the whole batch when it can (its warps
        // then spread evenly over the 4 schedulers): 1,024 chains -> 147 CTAs of 7 warps
        int n_sm = 148;
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
        const int wpc = (int)std::min<long long>(8, std::max<long long>(1, (B + n_sm - 1) / n_sm));
        const unsigned grid = (unsigned)((B + wpc - 1) / wpc), threads = 32u * (unsigned)wpc;
        const bool em_smem = M <= 128;
        size_t smem = (size_t)wpc * 2 * 72 * sizeof(float) + (em_smem ? (size_t)M * 64 * sizeof(float) : 0);
        const float *a = (const float*)A.p, *at = (const float*)At.p, *en = (const float*)En.p;
        if (em_smem) {
            CXB_LAUNCH((k_hmm64_pass<true, true>), grid, threads, smem, stream, a, en, obs.p, (float*)fwd.p, (float*)marg.p, B, this->T, M);
            CXB_LAUNCH((k_hmm64_pass<false, true>), grid, threads, smem, stream, at, en, obs.p, (float*)fwd.p, (float*)marg.p, B, this->T, M);
        } else {
            CXB_LAUNCH((k_hmm64_pass<true, false>), grid, threads, smem, stream, a, en, obs.p, (float*)fwd.p, (float*)marg.p, B, this->T, M);
            CXB_LAUNCH((k_hmm64_pass<false, false>), grid, threads, smem, stream, at, en, obs.p, (float*)fwd.p, (float*)marg.p, B, this->T, M);
        }
        return CXB_OK;
    }
    template <class T>
    int32_t launch_t() {
        const long long stage = (long long)HMM_WARPS * K * sizeof(T), em = (long long)M * K * sizeof(T),  // per-warp staging, emission messages
            row = (long long)K * sizeof(T), budget = 200 * 1024;
        if (sizeof(T) == 4 && K == 64) return launch_k64();
        if (sizeof(T) == 4 && tc_ready && tc_eligible()) return launch_tc();
        if (K == 32) return launch_pair<T, 32, true, true>(0, (size_t)(stage + em));  // at most 66 KB (fp64, M = 256)
        // the emission table stays in shared memory while it and one table row fit; else it is read from global memory (L2)
        // and the row tiles get all but the staging: at K = 1024 fp64 that is 17 rows
        const bool em_smem = stage + em + row <= budget;
        const long long rest = budget - stage - (em_smem ? em : 0);
        const int tile_rows = (int)std::min<long long>(K, rest / row);
        const size_t smem = (size_t)(budget - rest + tile_rows * row);
        return em_smem ? launch_pair<T, 0, false, true>(tile_rows, smem) : launch_pair<T, 0, false, false>(tile_rows, smem);
    }
    int32_t launch() {
        if (!have_tables || !have_obs) {
            err = "set the tables and the observations first";
            return CXB_ERR_STATE;
        }
        CXB_CUDA(cudaSetDevice(device));
        CXB_CUDA(cudaEventRecord(ev0, stream));
        int32_t st = dtype == CXB_F32 ? launch_t<float>() : launch_t<double>();
        if (st) return st;
        CXB_CUDA(cudaEventRecord(ev1, stream));
        CXB_CUDA(cudaGetLastError());
        ran = true;
        return CXB_OK;
    }
};

}  // namespace cxb

using cxb::Hmm;
static inline Hmm* HM(cxb_hmm* m) { return reinterpret_cast<Hmm*>(m); }
#define HM_CUDA(m, expr)                                        \
    do {                                                        \
        cudaError_t e__ = (expr);                               \
        if (e__ != cudaSuccess) {                               \
            HM(m)->err = ::cxb::cuda_msg(e__, #expr);           \
            return CXB_ERR_CUDA;                                \
        }                                                       \
    } while (0)

extern "C" {

int32_t cxb_hmm_create(int32_t device, int32_t dtype, int64_t n_chains, int64_t n_steps, int32_t n_states, int32_t n_symbols,
                       cxb_hmm** out) try {
    if (!out || (dtype != CXB_F32 && dtype != CXB_F64)) return CXB_ERR_BAD_ARG;
    *out = nullptr;
    Hmm* m = new Hmm();
    m->device = device;
    m->dtype = dtype;
    m->B = n_chains;
    m->T = n_steps;
    m->K = n_states;
    m->M = n_symbols;
    int32_t st = m->init();
    if (st) {
        fprintf(stderr, "cxb_hmm_create: %s\n", m->err.c_str());
        delete m;
        return st;
    }
    *out = reinterpret_cast<cxb_hmm*>(m);
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
void cxb_hmm_destroy(cxb_hmm* m) {
    if (m) {
        cudaSetDevice(HM(m)->device);
        delete HM(m);
    }
}
const char* cxb_hmm_last_error(cxb_hmm* m) { return m ? HM(m)->err.c_str() : "null handle"; }
int32_t cxb_hmm_set_tables(cxb_hmm* m, const double* transition, const double* emission) try {
    return HM(m)->set_tables(transition, emission);
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_hmm_set_observations(cxb_hmm* m, const uint8_t* obs_host) try {
    Hmm* h = HM(m);
    const size_t n = (size_t)h->T * h->B;
    HM_CUDA(m, cudaSetDevice(h->device));
    h->have_obs = false;
    HM_CUDA(m, cudaMemcpyAsync(h->obs.p, obs_host, n, cudaMemcpyHostToDevice, h->stream));
    int bad = 0;
    if (h->M < 256) {  // with 256 symbols every byte is one
        HM_CUDA(m, cudaMemsetAsync(h->obs_bad.p, 0, sizeof(int), h->stream));
        CXB_LAUNCH(cxb::k_hmm_check_obs, std::min(cxb::cdiv(n, 16 * 256), 1024u), 256, 0, h->stream, h->obs.p, n, h->M, h->obs_bad.p);
        HM_CUDA(m, cudaGetLastError());
        HM_CUDA(m, cudaMemcpyAsync(&bad, h->obs_bad.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    }
    HM_CUDA(m, cudaStreamSynchronize(h->stream));
    if (bad) {
        h->err = "observation symbol out of range (0 <= o < n_symbols)";
        return CXB_ERR_BAD_ARG;
    }
    h->have_obs = true;
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_hmm_update_marginals(cxb_hmm* m, int64_t* n_updates_out) try {
    Hmm* h = HM(m);
    int32_t st = h->launch();
    if (st) return st;
    if (n_updates_out) *n_updates_out = h->B * (6 * h->T - 4);
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
static int32_t hmm_get(cxb_hmm* m, const unsigned char* src, int64_t t0, int64_t t1, void* out_host) {
    Hmm* h = HM(m);
    if (!h->ran || t0 < 0 || t1 > h->T || t0 >= t1) {
        h->err = "bad time slice or no update has run yet";
        return CXB_ERR_BAD_ARG;
    }
    size_t step = (size_t)h->B * h->K * h->esz();
    HM_CUDA(m, cudaSetDevice(h->device));
    HM_CUDA(m, cudaMemcpyAsync(out_host, src + (size_t)t0 * step, (size_t)(t1 - t0) * step, cudaMemcpyDeviceToHost, h->stream));
    HM_CUDA(m, cudaStreamSynchronize(h->stream));
    return CXB_OK;
}
int32_t cxb_hmm_get_marginals(cxb_hmm* m, int64_t t0, int64_t t1, void* out_host) try { return hmm_get(m, HM(m)->marg.p, t0, t1, out_host); } CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_hmm_get_forward(cxb_hmm* m, int64_t t0, int64_t t1, void* out_host) try { return hmm_get(m, HM(m)->fwd.p, t0, t1, out_host); } CXB_ABI_CATCH(CXB_ERR_INTERNAL)
void* cxb_hmm_stream(cxb_hmm* m) { return (void*)HM(m)->stream; }
int32_t cxb_hmm_last_kernel_ms(cxb_hmm* m, float* ms_out) try {
    Hmm* h = HM(m);
    if (!h->ran) {
        h->err = "no update has run yet";
        return CXB_ERR_STATE;
    }
    HM_CUDA(m, cudaEventSynchronize(h->ev1));
    HM_CUDA(m, cudaEventElapsedTime(ms_out, h->ev0, h->ev1));
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_hmm_sync(cxb_hmm* m) try {
    HM_CUDA(m, cudaStreamSynchronize(HM(m)->stream));
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)

}  // extern "C"
