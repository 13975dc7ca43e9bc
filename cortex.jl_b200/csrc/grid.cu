// grid.cu — structured engine for loopy BP on a 2-D Potts grid by synchronous sweeps (BASELINE config 4).
//
// Graph (identical to tests/models.py:make_grid_model, ascending ids): pixels row-major; one unary (leaf)
// factor per pixel; pairwise factors on the 4-neighbourhood created per pixel as (right, down).  For a pixel
// the connected factors in ascending id order are therefore  unary < up < left < right < down, which is the
// multiplication order of every product below (DefaultDependencyResolver n<=5 path, src/dependencies.jl:60-88).
//
// One sweep = protocol B of SURVEY Appendix B = re-assert the unary evidence + update_marginals!(engine, all):
//   loop phase : every m2v(v,f)   = normalise(Potts(m2f(u,f)))          from the PREVIOUS sweep's m2f
//   final phase: marginal(v)      = normalise(unary * prod_f m2v(v,f))
//                linked m2f(v,f)  = normalise(unary * prod_{g != f} m2v(v,g))
// Potts table psi[a][b] = exp(beta [a==b])  =>  sum_b psi[a][b] m[b] = sum(m) + (e^beta - 1) m[a].
//
// Kernel: fused per-pixel pass, HBM-bound (576 B of traffic per interior pixel at K=16 fp32: read 4 m2f + unary, write
// 4 m2f).  Every m2v and every marginal is computed, but only rows 0 and H - 1 store theirs: the others are a function of
// this sweep's input m2f and unary, which stay intact until the next sweep (or until the host flushes them before a reset,
// set_unary or infer_host overwrites them), so k_potts_m2v rebuilds them bit for bit on the first read of an m2v plane
// (cxb_grid_get_messages) or of the marginals (cxb_grid_get_marginals): interior-row marginals are computed only when read.
// No later sweep reads them; storing them would add 256 B (m2v) + 64 B (marginal) per pixel.  The last sweep of an
// infer_host job stores every marginal, so its download needs no rebuild.  CXB_GRID_EAGER_M2V=1 stores every m2v and every
// marginal every sweep (896 B per pixel).  LP = K / (16 B / sizeof(T)) lanes cooperate on one
// pixel, each lane moving 16-byte vectors, so a warp touches 32*16 = 512 contiguous bytes per plane per
// instruction; K-sums are 2-4 warp-shuffle steps.  m2f planes are double buffered (sweep reads `cur`, writes
// `nxt`), every value is read exactly once.  Row sharding: the up/down messages of the first/last local row
// are contiguous rows of the `up`/`down` planes and are exchanged with the neighbour ranks between sweeps
// (halo_send_ptr / halo_recv_ptr), see cortex.jl_b200/grid.py.
//
// Per-edge couplings (cxb_grid_set_couplings): factor e has its own beta_e; the closed form above holds per factor with
// w_e = e^beta_e - 1, converted on the host exactly as the uniform w is, so equal couplings give the uniform grid bit for
// bit. The kernels' PE instantiations load w_e from two planes in the engine dtype, w_h [H][W] and w_v [H + 1][W] (rows 0
// and H: the cut edges), +8 B per pixel at fp32; the PE = false instantiations are the uniform kernels unchanged. The lazy
// rebuilds read the same planes, so set_couplings first flushes whatever the last sweep left pending.
#include <cmath>

#include <cstring>

#include "common.cuh"

namespace cxb {

// direction index d: 0 = up, 1 = left, 2 = right, 3 = down (ascending factor id); opposite(d) = 3 - d
template <class T, int E>
struct VecE;
template <>
struct VecE<float, 4> {
    using type = float4;
};
template <>
struct VecE<double, 2> {
    using type = double2;
};

template <class T, int E>
__device__ __forceinline__ void load_vec(const T* p, T (&v)[E]) {
    using V = typename VecE<T, E>::type;
    V x = __ldcs(reinterpret_cast<const V*>(p));
    const T* s = reinterpret_cast<const T*>(&x);
#pragma unroll
    for (int k = 0; k < E; ++k) v[k] = s[k];
}
template <class T, int E>
__device__ __forceinline__ void store_vec(T* p, const T (&v)[E]) {
    using V = typename VecE<T, E>::type;
    V x;
    T* s = reinterpret_cast<T*>(&x);
#pragma unroll
    for (int k = 0; k < E; ++k) s[k] = v[k];
    __stcs(reinterpret_cast<V*>(p), x);
}
template <class T, int E, int LP>
__device__ __forceinline__ T group_sum(const T (&v)[E]) {
    T s = v[0];
#pragma unroll
    for (int k = 1; k < E; ++k) s += v[k];
#pragma unroll
    for (int o = LP / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, LP);
    return s;
}

// 1 / x for a positive normal x. fp32: MUFU.RCP + one Newton step (<= 1 ulp) instead of the IEEE division subroutine
// (a CALL with a slow path, nine times per pixel); fp64: exact.
template <class T>
__device__ __forceinline__ T rcp_pos(T x) {
    if constexpr (sizeof(T) == 4) {
        float q;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(q) : "f"(x));
        return fmaf(q, fmaf(-x, q, 1.0f), q);
    } else {
        return T(1) / x;
    }
}

// loop phase of one factor: m2v(v, f) = normalise(S + w * in), S = sum(in), stored at plane + o when `store`; an absent
// factor gives the neutral element and stores nothing. The sweep and k_potts_m2v both call this, so a rebuilt m2v is
// bit-identical to the one the sweep multiplied with. (The store sits inside the branch: computing its address outside it
// costs the fp32 sweep up to 9 registers.)
template <class T, int E, int LP>
__device__ __forceinline__ void potts_m2v(const T (&in)[E], bool ex, T w, T (&mv)[E], bool store, void* plane, size_t o) {
    const T S = group_sum<T, E, LP>(in);
#pragma unroll
    for (int k = 0; k < E; ++k) mv[k] = S + w * in[k];
    const T tot = group_sum<T, E, LP>(mv);  // every lane shuffles, present factor or not
    if (ex) {
        const T inv = rcp_pos<T>(tot);
#pragma unroll
        for (int k = 0; k < E; ++k) mv[k] = mv[k] * inv;
        if (store) store_vec<T, E>((T*)plane + o, mv);
    } else {
#pragma unroll
        for (int k = 0; k < E; ++k) mv[k] = T(1);
    }
}

// final phase, marginal(v) = normalise(unary * prod_f m2v(v, f)) in ascending factor order, absent factors skipped; stored at
// marg + o when `store`. Every lane shuffles whether it stores or not. The sweep and k_potts_m2v both call this, so a rebuilt
// marginal is bit-identical to the one the sweep would have stored.
template <class T, int E, int LP>
__device__ __forceinline__ void potts_marginal(const T (&un)[E], const T (&mv)[4][E], const bool (&ex)[4], bool store, void* marg, size_t o) {
    T acc[E];
#pragma unroll
    for (int k = 0; k < E; ++k) {
        T a = un[k];
        if (ex[0]) a = a * mv[0][k];
        if (ex[1]) a = a * mv[1][k];
        if (ex[2]) a = a * mv[2][k];
        if (ex[3]) a = a * mv[3][k];
        acc[k] = a;
    }
    const T inv_tot = rcp_pos<T>(group_sum<T, E, LP>(acc));
#pragma unroll
    for (int k = 0; k < E; ++k) acc[k] = acc[k] * inv_tot;
    if (store) store_vec<T, E>((T*)marg + o, acc);
}

struct GridView {
    long long H, W;
    int has_up, has_down;
    // The rows 1 .. H - 2 of the m2v planes / of the marginals. k_potts_sweep: 1 = store them; 0 = store only rows 0 and
    // H - 1, whose up / down inputs may come from a halo buffer that a neighbour can overwrite before they are read, and
    // leave the others to k_potts_m2v. k_potts_m2v: 1 = rebuild them.
    int inner_m2v, inner_marg;
    const void* unary;       // [H][W][K]
    const void* m2f_cur[4];  // [H][W][K] per direction (message from the pixel towards direction d)
    void* m2f_nxt[4];
    void* m2v[4];
    void* marg;
    const void* halo_up;    // m2f(down) of the row above the shard, [W][K]
    const void* halo_down;  // m2f(up) of the row below the shard
    // fused halo exchange over peer memory (NVLink P2P): where the row-neighbour shard wants this sweep's boundary
    // messages — its halo buffer of the NEXT sweep's parity — or null (no neighbour / exchange done by the caller)
    void* peer_up;          // upper neighbour's halo_down slot: receives row 0 of plane `up`
    void* peer_down;        // lower neighbour's halo_up slot: receives the last row of plane `down`
};

// Per-edge couplings (cxb_grid_set_couplings), w = e^beta - 1 of each of a pixel's four factors, from the planes wh[H][W]
// (factor to the right of pixel (i, j); last column unused) and wv[H + 1][W] (factor above local row i; rows 0 and H are the
// cut edges); pix = i * W + j. An absent factor's coupling is never used; the left one is not even loaded, as pix - 1 is
// outside the plane at pixel 0. Each weight is loaded by both of its pixels, the second load hits L1 or L2.
template <class T>
__device__ __forceinline__ void couplings(const T* __restrict__ wh, const T* __restrict__ wv, long long W, long long pix, bool has_left,
                                          T w, T (&wd)[4]) {
    wd[0] = __ldg(wv + pix);
    wd[1] = has_left ? __ldg(wh + pix - 1) : w;
    wd[2] = __ldg(wh + pix);
    wd[3] = __ldg(wv + pix + W);
}

// PE: every factor has its own coupling (couplings()); otherwise all have `w`, and wh / wv are unused. They follow `w`, and
// PE = false passes `w` itself to potts_m2v, so the uniform kernels compile to the instruction stream they had before
// per-edge couplings existed.
template <class T, int K, int E, bool PE>
__global__ void __launch_bounds__(256) k_potts_sweep(GridView g, T w, const T* __restrict__ wh, const T* __restrict__ wv) {
    constexpr int LP = K / E;  // lanes per pixel
    static_assert(LP >= 1 && LP <= 32 && (LP & (LP - 1)) == 0, "K / E must be a power of two <= 32");
    const long long npix = g.H * g.W;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long pix = gid / LP;
    const int lane = (int)(gid % LP);
    const bool valid = pix < npix;
    if (!valid) pix = npix - 1;  // keep the whole warp in the shuffles; results of clamped groups are dropped
    const long long i = pix / g.W, j = pix % g.W;
    const size_t o = (size_t)pix * K + (size_t)lane * E;

    bool ex[4];
    ex[0] = i > 0 || g.has_up;
    ex[1] = j > 0;
    ex[2] = j + 1 < g.W;
    ex[3] = i + 1 < g.H || g.has_down;

    T un[E];
    load_vec<T, E>((const T*)g.unary + o, un);

    T in[4][E];
    {
        // incoming m2f(u, f): the neighbour's message towards us = its plane opposite(d)
        const T* src[4];
        src[0] = (i > 0) ? (const T*)g.m2f_cur[3] + o - (size_t)g.W * K : (const T*)g.halo_up + (size_t)j * K + (size_t)lane * E;
        src[1] = (const T*)g.m2f_cur[2] + o - K;
        src[2] = (const T*)g.m2f_cur[1] + o + K;
        src[3] = (i + 1 < g.H) ? (const T*)g.m2f_cur[0] + o + (size_t)g.W * K
                               : (const T*)g.halo_down + (size_t)j * K + (size_t)lane * E;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            if (ex[d]) {
                load_vec<T, E>(src[d], in[d]);
            } else {
#pragma unroll
                for (int k = 0; k < E; ++k) in[d][k] = T(1);
            }
        }
    }
    // loop phase
    // rows 0 and H - 1 (every row when H <= 2) in one unsigned compare; i == 0 || i + 1 == g.H costs the fp32 sweep registers
    const bool edge_row = (unsigned long long)(pix - g.W) >= (unsigned long long)(npix - 2 * g.W);
    T wd[4];
    if constexpr (PE) couplings<T>(wh, wv, g.W, pix, ex[1], w, wd);
    T mv[4][E];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        potts_m2v<T, E, LP>(in[d], ex[d], PE ? wd[d] : w, mv[d], valid && (g.inner_m2v || edge_row), g.m2v[d], o);
    }
    // final phase: the linked m2f, then the marginal (products in ascending factor order, left to right; the marginal last
    // keeps the fp32 sweep at 48 registers)
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        T acc[E];
#pragma unroll
        for (int k = 0; k < E; ++k) {
            T a = un[k];
#pragma unroll
            for (int d2 = 0; d2 < 4; ++d2)
                if (d2 != d && ex[d2]) a = a * mv[d2][k];
            acc[k] = a;
        }
        const T inv_tot = rcp_pos<T>(group_sum<T, E, LP>(acc));
#pragma unroll
        for (int k = 0; k < E; ++k) acc[k] = acc[k] * inv_tot;
        if (valid && ex[d]) store_vec<T, E>((T*)g.m2f_nxt[d] + o, acc);
        // the cut edges: the same message goes straight into the neighbour GPU's halo buffer (peer store over NVLink),
        // overlapped with the rest of the sweep; cxb_grid_sweep publishes a sweep counter after the kernel
        if (d == 0 && valid && i == 0 && g.peer_up) store_vec<T, E>((T*)g.peer_up + (size_t)j * K + (size_t)lane * E, acc);
        if (d == 3 && valid && i + 1 == g.H && g.peer_down) store_vec<T, E>((T*)g.peer_down + (size_t)j * K + (size_t)lane * E, acc);
    }
    potts_marginal<T, E, LP>(un, mv, ex, valid && (g.inner_marg || edge_row), g.marg, o);
}

// Rows 1 .. H - 2 of the m2v planes (g.inner_m2v) and / or of the marginals (g.inner_marg), which a sweep with the same flag
// 0 does not store, rebuilt from the m2f planes that sweep read (g.m2f_cur) and, for the marginals, the unary plane it read
// (g.unary): both stay intact until the next sweep, whose own values supersede these, or until the host flushes (reset,
// set_unary, infer_host). Rows 1 .. H - 2 take their up and down inputs from this shard's planes, never from a halo buffer.
// Lane layout as in k_potts_sweep; no m2v store where the factor is absent, so those slots keep the zeros of init.
template <class T, int K, int E, bool PE>
__global__ void __launch_bounds__(256) k_potts_m2v(GridView g, T w, const T* __restrict__ wh, const T* __restrict__ wv) {
    constexpr int LP = K / E;
    const long long npix = (g.H - 2) * g.W;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long q = gid / LP;
    const int lane = (int)(gid % LP);
    const bool valid = q < npix;
    if (!valid) q = npix - 1;  // keep the whole warp in the shuffles
    const long long pix = q + g.W;
    const long long j = pix % g.W;
    const size_t o = (size_t)pix * K + (size_t)lane * E;
    const bool ex[4] = {true, j > 0, j + 1 < g.W, true};
    const T* src[4];
    src[0] = (const T*)g.m2f_cur[3] + o - (size_t)g.W * K;
    src[1] = (const T*)g.m2f_cur[2] + o - K;
    src[2] = (const T*)g.m2f_cur[1] + o + K;
    src[3] = (const T*)g.m2f_cur[0] + o + (size_t)g.W * K;
    T in[4][E], un[E];  // all loads in flight before the first store
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        if (ex[d]) {
            load_vec<T, E>(src[d], in[d]);
        } else {
#pragma unroll
            for (int k = 0; k < E; ++k) in[d][k] = T(1);
        }
    }
    if (g.inner_marg) load_vec<T, E>((const T*)g.unary + o, un);
    T wd[4];
    if constexpr (PE) couplings<T>(wh, wv, g.W, pix, ex[1], w, wd);
    T mv[4][E];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        potts_m2v<T, E, LP>(in[d], ex[d], PE ? wd[d] : w, mv[d], valid && g.inner_m2v, g.m2v[d], o);
    }
    if (g.inner_marg) potts_marginal<T, E, LP>(un, mv, ex, valid, g.marg, o);
}

// stream-ordered hand-shake of the fused halo exchange: sweeps completed by the neighbours are counted in flags that
// live in THIS shard's memory and are written by the neighbours' k_halo_signal
// The spin is BOUNDED (a row neighbour that died or never enqueued its sweep must not hang the stream for ever): after
// `timeout_ns` of waiting the kernel records which neighbour is missing in *timed_out and returns; the host finds the flag at
// the next cxb_grid_sync / cxb_grid_get_* and reports CXB_ERR_STATE (the shard's messages are then not to be trusted).
__global__ void k_halo_wait(const volatile unsigned* flag_a, const volatile unsigned* flag_b, unsigned expected, unsigned long long timeout_ns,
                            unsigned* timed_out) {
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    auto wait = [&](const volatile unsigned* f, unsigned bit) {
        while (*f < expected) {
            __nanosleep(64);
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > timeout_ns) {
                atomicOr(timed_out, bit);
                return;
            }
        }
    };
    if (flag_a) wait(flag_a, 1u);
    if (flag_b) wait(flag_b, 2u);
    __threadfence_system();
}
__global__ void k_halo_signal(unsigned* peer_flag_a, unsigned* peer_flag_b, unsigned value) {
    __threadfence_system();  // the sweep kernel's peer stores (previous kernel of this stream) are visible before the flag
    if (peer_flag_a) *(volatile unsigned*)peer_flag_a = value;
    if (peer_flag_b) *(volatile unsigned*)peer_flag_b = value;
    __threadfence_system();
}

template <class T>
__global__ void k_fill(T* p, size_t n, T v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

struct Grid {
    int device = 0, dtype = CXB_F32, K = 0, has_up = 0, has_down = 0, cur = 0;
    long long H = 0, W = 0;
    double beta = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    DBuf<unsigned char> unary, m2f[2], m2v, marg, halo_recv;  // m2f[b]: 4 planes; m2v: 4 planes; halo_recv: [2 parities][2 rows]
    DBuf<unsigned> flags;                       // [0] sweeps completed by the upper neighbour, [1] by the lower neighbour
    // pipelined host entry point (infer_host): job j uses unary buffer j & 1 and marginal buffer j & 1, so that the evidence of
    // job j + 1 travels host -> device and the marginals of job j - 1 device -> host while the sweeps of job j run
    DBuf<unsigned char> unary_alt, marg_alt;
    unsigned char *cur_unary = nullptr, *cur_marg = nullptr;  // what sweep() reads / writes (default: unary.p / marg.p)
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_sw[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    unsigned long long job_no = 0;
    unsigned sweep_no = 0;                      // sweeps since the last reset (parity of the halo buffers)
    unsigned long long halo_timeout_ns = 20ull * 1000000000ull;  // CXB_GRID_HALO_TIMEOUT_MS overrides (tests)
    // m2v planes and marginals: a sweep stores only their first and last rows unless eager_m2v (CXB_GRID_EAGER_M2V=1), or,
    // for the marginals, the sweep is the last of an infer_host job; m2v_pending / marg_pending = the other rows of the last
    // sweep are not yet rebuilt (flush). pend_unary / pend_marg: the evidence that sweep read and the marginal buffer it
    // wrote, which infer_host may since have switched away from
    bool eager_m2v = false, m2v_pending = false, marg_pending = false;
    const unsigned char* pend_unary = nullptr;
    unsigned char* pend_marg = nullptr;
    cudaEvent_t ev_fl = nullptr;  // infer_host: the evidence upload waits for a marginal rebuild that reads its buffer
    // per-edge couplings (cxb_grid_set_couplings), w = e^beta - 1 in the engine dtype: w_h [H][W], w_v [H + 1][W]; reserved on
    // first use. coupled = the kernels read them instead of the create-time beta
    DBuf<unsigned char> w_h, w_v;
    bool coupled = false;
    // after a stream sync: did a halo wait give up on a neighbour?
    int32_t check_halo() {
        if (!peer_halo[0] && !peer_halo[1]) return CXB_OK;
        unsigned t = 0;
        if (cudaMemcpy(&t, flags.p + 2, sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) return CXB_ERR_CUDA;
        if (!t) return CXB_OK;
        err = std::string("fused halo exchange: the row neighbour ") + ((t & 1) ? "above" : "below") +
              " did not deliver its boundary messages in time (its sweep was never enqueued, or the process is gone)";
        return CXB_ERR_STATE;
    }
    unsigned char* peer_halo[2] = {nullptr, nullptr};  // the neighbours' halo_recv (direction 0 = above, 1 = below)
    unsigned* peer_flags[2] = {nullptr, nullptr};      // the neighbours' flags
    void* ipc_opened[4] = {nullptr, nullptr, nullptr, nullptr};
    bool have_unary = false, have_msgs = false, ran = false;
    size_t esz() const { return dtype == CXB_F32 ? 4 : 8; }
    size_t plane() const { return (size_t)H * W * K * esz(); }
    size_t row() const { return (size_t)W * K * esz(); }
    ~Grid() {
        for (void* q : ipc_opened)
            if (q) cudaIpcCloseMemHandle(q);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (ev_fl) cudaEventDestroy(ev_fl);
        for (int i = 0; i < 2; ++i) {
            if (ev_in[i]) cudaEventDestroy(ev_in[i]);
            if (ev_sw[i]) cudaEventDestroy(ev_sw[i]);
            if (ev_out[i]) cudaEventDestroy(ev_out[i]);
        }
        if (s_in) cudaStreamDestroy(s_in);
        if (s_out) cudaStreamDestroy(s_out);
        if (stream) cudaStreamDestroy(stream);
    }
    int32_t init() {
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
            err = "no CUDA device available (cortex_b200 has no CPU fallback)";
            return CXB_ERR_CUDA;
        }
        int E = dtype == CXB_F32 ? 4 : 2;
        int LP = K / E;
        if (device < 0 || device >= count || H <= 0 || W <= 0 || K < E || K % E || LP > 32 || (LP & (LP - 1))) {
            err = "bad device / shape (labels must be 4,8,...,128 for fp32 and 2,4,...,64 for fp64, a power of two)";
            return CXB_ERR_BAD_ARG;
        }
        CXB_CUDA(cudaSetDevice(device));
        CXB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        if (const char* e = getenv("CXB_GRID_HALO_TIMEOUT_MS")) halo_timeout_ns = (unsigned long long)std::max(1, atoi(e)) * 1000000ull;
        if (const char* e = getenv("CXB_GRID_EAGER_M2V")) eager_m2v = atoi(e) != 0;
        CXB_CUDA(cudaEventCreate(&ev0));
        CXB_CUDA(cudaEventCreate(&ev1));
        CXB_CUDA(unary.reserve(plane()));
        CXB_CUDA(m2f[0].reserve(4 * plane()));
        CXB_CUDA(m2f[1].reserve(4 * plane()));
        CXB_CUDA(m2v.reserve(4 * plane()));
        CXB_CUDA(marg.reserve(plane()));
        CXB_CUDA(halo_recv.reserve(4 * row()));
        CXB_CUDA(flags.reserve(4));  // [0], [1] sweep counters written by the neighbours; [2] halo wait timed out (bit 0 above, bit 1 below)
        CXB_CUDA(cudaMemsetAsync(flags.p, 0, 4 * sizeof(unsigned), stream));
        CXB_CUDA(cudaMemsetAsync(m2v.p, 0, 4 * plane(), stream));
        CXB_CUDA(cudaMemsetAsync(marg.p, 0, plane(), stream));
        return CXB_OK;
    }
    template <class T>
    int32_t fill(void* p, size_t n, double v) {
        CXB_LAUNCH(k_fill<T>, cdiv(n, 256), 256, 0, stream, (T*)p, n, (T)v);
        return CXB_OK;
    }
    int32_t reset() {
        CXB_CUDA(cudaSetDevice(device));
        if (int32_t st = flush(true, true)) return st;  // before the fill below overwrites the m2f planes it reads
        size_t n = (size_t)4 * H * W * K, nh = (size_t)4 * W * K;
        double u = 1.0 / K;
        for (int b = 0; b < 2; ++b) dtype == CXB_F32 ? fill<float>(m2f[b].p, n, u) : fill<double>(m2f[b].p, n, u);
        dtype == CXB_F32 ? fill<float>(halo_recv.p, nh, u) : fill<double>(halo_recv.p, nh, u);
        // with a fused (peer-memory) exchange every shard of the grid must be idle here: the neighbours' counters restart
        CXB_CUDA(cudaMemsetAsync(flags.p, 0, 4 * sizeof(unsigned), stream));
        CXB_CUDA(cudaGetLastError());
        // synchronous: a neighbour shard that starts sweeping right after ITS reset stores its boundary messages into this
        // shard's halo buffer; were this fill still queued behind the large message planes it would overwrite them with the
        // uniform message (found at 1024^2 and larger by tests/test_fullsize_parity.py; the small grids never showed it)
        CXB_CUDA(cudaStreamSynchronize(stream));
        cur = 0;
        sweep_no = 0;
        have_msgs = true;
        return CXB_OK;
    }
    // the views of both kernels: m2f planes of buffer `in` are read, those of in ^ 1 written
    GridView view(int in) const {
        GridView g{};
        g.H = H;
        g.W = W;
        g.has_up = has_up;
        g.has_down = has_down;
        g.inner_m2v = g.inner_marg = eager_m2v;
        for (int d = 0; d < 4; ++d) {
            g.m2f_cur[d] = m2f[in].p + (size_t)d * plane();
            g.m2f_nxt[d] = m2f[in ^ 1].p + (size_t)d * plane();
            g.m2v[d] = m2v.p + (size_t)d * plane();
        }
        return g;
    }
    // k_potts_sweep over every pixel, or k_potts_m2v over rows 1 .. H - 2
    template <class T, int E>
    int32_t launch_k(const GridView& g, bool m2v_only) {
        const T w = (T)(std::exp(beta) - 1.0);
        const T* wh = coupled ? (const T*)w_h.p : nullptr;
        const T* wv = coupled ? (const T*)w_v.p : nullptr;
        long long threads = (m2v_only ? H - 2 : H) * W * (K / E);
        unsigned grid = cdiv((size_t)threads, 256);
        switch (K / E) {
#define LAUNCH(KERNEL, LPV, PE) CXB_LAUNCH((KERNEL<T, LPV * E, E, PE>), grid, 256, 0, stream, g, w, wh, wv)
#define CASE(LPV)                                                                                      \
    case LPV:                                                                                          \
        if (m2v_only && coupled)                                                                       \
            LAUNCH(k_potts_m2v, LPV, true);                                                            \
        else if (m2v_only)                                                                             \
            LAUNCH(k_potts_m2v, LPV, false);                                                           \
        else if (coupled)                                                                              \
            LAUNCH(k_potts_sweep, LPV, true);                                                          \
        else                                                                                           \
            LAUNCH(k_potts_sweep, LPV, false);                                                         \
        break;
            CASE(1)
            CASE(2)
            CASE(4)
            CASE(8)
            CASE(16)
            CASE(32)
#undef CASE
#undef LAUNCH
        }
        return CXB_OK;
    }
    // cxb_grid_set_couplings: every value is checked before any device state changes; both null = back to the uniform beta
    template <class T>
    int32_t set_couplings(const double* hz, const double* vt) {
        if (!hz != !vt) {
            err = "set_couplings: give both coupling arrays, or neither (back to the uniform beta)";
            return CXB_ERR_BAD_ARG;
        }
        std::vector<T> h, v;
        if (hz) {
            h.assign((size_t)H * W, T(0));
            v.assign((size_t)(H + 1) * W, T(0));
            auto conv = [&](double beta, T& out) {
                const T w = (T)(std::exp(beta) - 1.0);  // the expression of launch_k: equal couplings give the uniform grid
                if (!std::isfinite(beta) || !std::isfinite(w)) {
                    err = "set_couplings: beta " + std::to_string(beta) + " is not finite, or exp(beta) - 1 overflows the engine dtype";
                    return false;
                }
                out = w;
                return true;
            };
            for (long long i = 0; i < H; ++i)
                for (long long j = 0; j + 1 < W; ++j)
                    if (!conv(hz[i * (W - 1) + j], h[i * W + j])) return CXB_ERR_BAD_ARG;
            for (long long i = has_up ? 0 : 1; i <= (has_down ? H : H - 1); ++i)  // rows 0 and H only with a neighbour
                for (long long j = 0; j < W; ++j)
                    if (!conv(vt[i * W + j], v[i * W + j])) return CXB_ERR_BAD_ARG;
        }
        CXB_CUDA(cudaSetDevice(device));
        // the pending m2v / marginal rows of the last sweep are rebuilt with the couplings it read
        if (int32_t st = flush(true, true)) return st;
        if (hz) {
            CXB_CUDA(w_h.reserve(h.size() * sizeof(T)));
            CXB_CUDA(w_v.reserve(v.size() * sizeof(T)));
            CXB_CUDA(cudaMemcpyAsync(w_h.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, stream));
            CXB_CUDA(cudaMemcpyAsync(w_v.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, stream));
        }
        CXB_CUDA(cudaStreamSynchronize(stream));
        coupled = hz != nullptr;
        return CXB_OK;
    }
    // all_marg: store every marginal whatever the mode (the last sweep of an infer_host job)
    int32_t sweep(int64_t* n_updates, bool all_marg = false) {
        if (!have_unary || !have_msgs) {
            err = "set the unary evidence and reset the messages first";
            return CXB_ERR_STATE;
        }
        CXB_CUDA(cudaSetDevice(device));
        GridView g = view(cur);
        g.unary = cur_unary ? cur_unary : unary.p;
        g.marg = cur_marg ? cur_marg : marg.p;
        g.inner_marg |= all_marg;
        // halo buffers are double buffered by sweep parity: sweep s reads parity s & 1 (written by the neighbours' sweep
        // s - 1, or by the caller's exchange) and pushes its own boundary rows into the neighbours' parity (s + 1) & 1
        const size_t par = (size_t)(sweep_no & 1) * 2 * row(), nxt_par = (size_t)((sweep_no + 1) & 1) * 2 * row();
        g.halo_up = halo_recv.p + par;
        g.halo_down = halo_recv.p + par + row();
        g.peer_up = peer_halo[0] ? peer_halo[0] + nxt_par + row() : nullptr;   // the upper neighbour's halo_down
        g.peer_down = peer_halo[1] ? peer_halo[1] + nxt_par : nullptr;         // the lower neighbour's halo_up
        const bool fused = peer_halo[0] || peer_halo[1];
        if (fused && sweep_no > 0)  // the neighbours have finished sweep sweep_no - 1 (their boundary rows have landed here)
            CXB_LAUNCH(k_halo_wait, 1, 1, 0, stream, peer_halo[0] ? flags.p + 0 : nullptr, peer_halo[1] ? flags.p + 1 : nullptr, sweep_no,
                       halo_timeout_ns, flags.p + 2);
        CXB_CUDA(cudaEventRecord(ev0, stream));
        int32_t st = dtype == CXB_F32 ? launch_k<float, 4>(g, false) : launch_k<double, 2>(g, false);
        if (st) return st;
        CXB_CUDA(cudaEventRecord(ev1, stream));
        m2v_pending = !g.inner_m2v;
        marg_pending = !g.inner_marg;
        pend_unary = (const unsigned char*)g.unary;
        pend_marg = (unsigned char*)g.marg;
        if (fused)  // tell the neighbours: my sweep sweep_no is complete (I am their lower / upper neighbour)
            CXB_LAUNCH(k_halo_signal, 1, 1, 0, stream, peer_flags[0] ? peer_flags[0] + 1 : nullptr, peer_flags[1] ? peer_flags[1] + 0 : nullptr,
                       sweep_no + 1);
        CXB_CUDA(cudaGetLastError());
        cur ^= 1;
        ++sweep_no;
        ran = true;
        if (n_updates) {
            // existing (pixel, direction) pairs: vertical incl. the cut edges, horizontal inside rows
            long long vert = (H - 1) * W * 2 + (has_up ? W : 0) + (has_down ? W : 0);
            long long horz = H * (W - 1) * 2;
            *n_updates = 2 * (vert + horz) + H * W;  // m2v + m2f + marginals
        }
        return CXB_OK;
    }
    // rebuild the m2v rows (m2v) and / or the marginal rows (marg) the last sweep did not store, from the m2f planes it read
    // (m2f[cur ^ 1] once it has run) and the evidence it read, in one k_potts_m2v launch; enqueued on `stream` after the sweep
    // and outside ev0 / ev1
    int32_t flush(bool m2v, bool marg) {
        m2v = m2v && m2v_pending;
        marg = marg && marg_pending;
        if (!m2v && !marg) return CXB_OK;
        CXB_CUDA(cudaSetDevice(device));
        if (H > 2) {
            GridView g = view(cur ^ 1);
            g.inner_m2v = m2v;
            g.inner_marg = marg;
            g.unary = pend_unary;
            g.marg = pend_marg;
            int32_t st = dtype == CXB_F32 ? launch_k<float, 4>(g, true) : launch_k<double, 2>(g, true);
            if (st) return st;
            CXB_CUDA(cudaGetLastError());
        }
        if (m2v) m2v_pending = false;
        if (marg) marg_pending = false;
        return CXB_OK;
    }
    // Host entry point of one JOB: evidence from (pinned) host memory, n_sweeps synchronous sweeps, marginals back to host
    // memory - asynchronous and pipelined over three streams: the call returns once everything is enqueued; the host -> device
    // copy of the NEXT job's evidence and the device -> host copy of the PREVIOUS job's marginals overlap this job's sweeps.
    // marginals_out_host of job j is complete when cxb_grid_sync returns (or after two further jobs). The messages carry
    // over from the previous job (no reset: with a fused halo a reset needs every shard idle).
    int32_t infer_host(const void* unary_host, void* marg_out_host, int n_sweeps, int64_t* n_updates) {
        if (!have_msgs) {
            err = "reset the messages first";
            return CXB_ERR_STATE;
        }
        CXB_CUDA(cudaSetDevice(device));
        // marginals a plain sweep() left pending are rebuilt now: their evidence buffer may be the one this job uploads into
        const bool flushed = marg_pending;
        if (int32_t st = flush(false, true)) return st;
        if (!s_in) {
            CXB_CUDA(unary_alt.reserve(plane()));
            CXB_CUDA(marg_alt.reserve(plane()));
            CXB_CUDA(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
            CXB_CUDA(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
            CXB_CUDA(cudaEventCreateWithFlags(&ev_fl, cudaEventDisableTiming));
            for (int i = 0; i < 2; ++i) {
                CXB_CUDA(cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming));
                CXB_CUDA(cudaEventCreateWithFlags(&ev_sw[i], cudaEventDisableTiming));
                CXB_CUDA(cudaEventCreateWithFlags(&ev_out[i], cudaEventDisableTiming));
            }
            CXB_CUDA(cudaStreamSynchronize(stream));  // earlier set_unary / sweeps on the compute stream are done
        }
        const int b = (int)(job_no & 1);
        unsigned char* U = b ? unary_alt.p : unary.p;
        unsigned char* M = b ? marg_alt.p : marg.p;
        if (flushed) {
            CXB_CUDA(cudaEventRecord(ev_fl, stream));
            CXB_CUDA(cudaStreamWaitEvent(s_in, ev_fl, 0));
        }
        if (job_no >= 2) CXB_CUDA(cudaStreamWaitEvent(s_in, ev_sw[b], 0));  // the sweeps of job j - 2 have read this evidence buffer
        CXB_CUDA(cudaMemcpyAsync(U, unary_host, plane(), cudaMemcpyHostToDevice, s_in));
        CXB_CUDA(cudaEventRecord(ev_in[b], s_in));
        CXB_CUDA(cudaStreamWaitEvent(stream, ev_in[b], 0));
        if (job_no >= 2) CXB_CUDA(cudaStreamWaitEvent(stream, ev_out[b], 0));  // job j - 2's marginals have left this buffer
        cur_unary = U;
        cur_marg = M;
        have_unary = true;
        int64_t upd = 0;
        for (int k = 0; k < n_sweeps; ++k) {  // the last sweep stores every marginal: the download below needs no rebuild
            int32_t st = sweep(&upd, k + 1 == n_sweeps);
            if (st) return st;
        }
        CXB_CUDA(cudaEventRecord(ev_sw[b], stream));
        CXB_CUDA(cudaStreamWaitEvent(s_out, ev_sw[b], 0));
        CXB_CUDA(cudaMemcpyAsync(marg_out_host, M, plane(), cudaMemcpyDeviceToHost, s_out));
        CXB_CUDA(cudaEventRecord(ev_out[b], s_out));
        ++job_no;
        if (n_updates) *n_updates = upd * n_sweeps;
        return CXB_OK;
    }
    int32_t sync_all() {
        CXB_CUDA(cudaSetDevice(device));
        CXB_CUDA(cudaStreamSynchronize(stream));
        if (s_in) CXB_CUDA(cudaStreamSynchronize(s_in));
        if (s_out) CXB_CUDA(cudaStreamSynchronize(s_out));
        return check_halo();
    }
};

}  // namespace cxb

using cxb::Grid;
static inline Grid* GR(cxb_grid* g) { return reinterpret_cast<Grid*>(g); }
#define GR_CUDA(g, expr)                                        \
    do {                                                        \
        cudaError_t e__ = (expr);                               \
        if (e__ != cudaSuccess) {                               \
            GR(g)->err = ::cxb::cuda_msg(e__, #expr);           \
            return CXB_ERR_CUDA;                                \
        }                                                       \
    } while (0)

extern "C" {

int32_t cxb_grid_create(int32_t device, int32_t dtype, int64_t rows, int64_t cols, int32_t n_labels, double beta,
                        int32_t has_upper, int32_t has_lower, cxb_grid** out) try {
    if (!out || (dtype != CXB_F32 && dtype != CXB_F64)) return CXB_ERR_BAD_ARG;
    *out = nullptr;
    Grid* g = new Grid();
    g->device = device;
    g->dtype = dtype;
    g->H = rows;
    g->W = cols;
    g->K = n_labels;
    g->beta = beta;
    g->has_up = has_upper ? 1 : 0;
    g->has_down = has_lower ? 1 : 0;
    int32_t st = g->init();
    if (st) {
        fprintf(stderr, "cxb_grid_create: %s\n", g->err.c_str());
        delete g;
        return st;
    }
    *out = reinterpret_cast<cxb_grid*>(g);
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
void cxb_grid_destroy(cxb_grid* g) {
    if (g) {
        cudaSetDevice(GR(g)->device);
        delete GR(g);
    }
}
const char* cxb_grid_last_error(cxb_grid* g) { return g ? GR(g)->err.c_str() : "null handle"; }
int32_t cxb_grid_set_unary(cxb_grid* g, const void* unary_host) try {
    Grid* h = GR(g);
    GR_CUDA(g, cudaSetDevice(h->device));
    if (int32_t st = h->flush(false, true)) return st;  // the pending marginals are those of the evidence about to be replaced
    GR_CUDA(g, cudaMemcpyAsync(h->cur_unary ? h->cur_unary : h->unary.p, unary_host, h->plane(), cudaMemcpyHostToDevice, h->stream));
    GR_CUDA(g, cudaStreamSynchronize(h->stream));
    h->have_unary = true;
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_grid_set_couplings(cxb_grid* g, const double* horizontal, const double* vertical) try {
    Grid* h = GR(g);
    return h->dtype == CXB_F32 ? h->set_couplings<float>(horizontal, vertical) : h->set_couplings<double>(horizontal, vertical);
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_grid_reset_messages(cxb_grid* g) try { return GR(g)->reset(); } CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_grid_sweep(cxb_grid* g, int64_t* n_updates_out) try { return GR(g)->sweep(n_updates_out); } CXB_ABI_CATCH(CXB_ERR_INTERNAL)
// the messages computed by the LAST sweep that the neighbour shard needs: row 0 of plane `up` (direction 0),
// last row of plane `down` (direction 1) of the current buffer
void* cxb_grid_halo_send_ptr(cxb_grid* g, int32_t direction) {
    Grid* h = GR(g);
    unsigned char* base = h->m2f[h->cur].p;
    if (direction == 0) return base + 0 * h->plane();
    if (direction == 1) return base + 3 * h->plane() + (size_t)(h->H - 1) * h->row();
    return nullptr;
}
void* cxb_grid_halo_recv_ptr(cxb_grid* g, int32_t direction) {
    Grid* h = GR(g);
    unsigned char* base = h->halo_recv.p + (size_t)(h->sweep_no & 1) * 2 * h->row();  // the parity the NEXT sweep reads
    if (direction == 0) return base;             // from the upper neighbour (its `down` row)
    if (direction == 1) return base + h->row();  // from the lower neighbour (its `up` row)
    return nullptr;
}
// ---- fused halo exchange over peer memory ---------------------------------------------------------------------------------
// export: 2 x 64 bytes = cudaIpcMemHandle_t of the halo buffer and of the sweep counters of THIS shard
int32_t cxb_grid_p2p_export(cxb_grid* g, void* handles_out) try {
    Grid* h = GR(g);
    GR_CUDA(g, cudaSetDevice(h->device));
    cudaIpcMemHandle_t hh[2];
    GR_CUDA(g, cudaIpcGetMemHandle(&hh[0], h->halo_recv.p));
    GR_CUDA(g, cudaIpcGetMemHandle(&hh[1], h->flags.p));
    memcpy(handles_out, hh, sizeof(hh));
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
// connect the row neighbour in `direction` (0 = above, 1 = below) that lives in ANOTHER process, by its exported handles
int32_t cxb_grid_p2p_connect_ipc(cxb_grid* g, int32_t direction, const void* neighbour_handles) try {
    Grid* h = GR(g);
    if (direction != 0 && direction != 1) return CXB_ERR_BAD_ARG;
    GR_CUDA(g, cudaSetDevice(h->device));
    cudaIpcMemHandle_t hh[2];
    memcpy(hh, neighbour_handles, sizeof(hh));
    void *halo = nullptr, *fl = nullptr;
    GR_CUDA(g, cudaIpcOpenMemHandle(&halo, hh[0], cudaIpcMemLazyEnablePeerAccess));
    GR_CUDA(g, cudaIpcOpenMemHandle(&fl, hh[1], cudaIpcMemLazyEnablePeerAccess));
    h->ipc_opened[2 * direction] = halo;
    h->ipc_opened[2 * direction + 1] = fl;
    h->peer_halo[direction] = (unsigned char*)halo;
    h->peer_flags[direction] = (unsigned*)fl;
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
// same, for a neighbour shard owned by THIS process (several shards per process; single-GPU tests)
int32_t cxb_grid_p2p_connect_local(cxb_grid* g, int32_t direction, cxb_grid* neighbour) try {
    Grid *h = GR(g), *nb = GR(neighbour);
    if ((direction != 0 && direction != 1) || !nb || nb->W != h->W || nb->K != h->K || nb->dtype != h->dtype) return CXB_ERR_BAD_ARG;
    if (nb->device != h->device) {
        int can = 0;
        GR_CUDA(g, cudaDeviceCanAccessPeer(&can, h->device, nb->device));
        if (!can) {
            h->err = "no peer access between the two devices";
            return CXB_ERR_CUDA;
        }
        GR_CUDA(g, cudaSetDevice(h->device));
        cudaError_t e = cudaDeviceEnablePeerAccess(nb->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) GR_CUDA(g, e);
        (void)cudaGetLastError();
    }
    h->peer_halo[direction] = nb->halo_recv.p;
    h->peer_flags[direction] = nb->flags.p;
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int64_t cxb_grid_halo_elems(cxb_grid* g) try { return GR(g)->W * GR(g)->K; } CXB_ABI_CATCH(-1)
int32_t cxb_grid_get_marginals(cxb_grid* g, void* out_host) try {
    Grid* h = GR(g);
    GR_CUDA(g, cudaSetDevice(h->device));
    if (int32_t st = h->flush(false, true)) return st;
    GR_CUDA(g, cudaMemcpyAsync(out_host, h->cur_marg ? h->cur_marg : h->marg.p, h->plane(), cudaMemcpyDeviceToHost, h->stream));
    GR_CUDA(g, cudaStreamSynchronize(h->stream));
    return h->check_halo();
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
// which: 0..3 = m2v from the (up, left, right, down) factor; 4..7 = m2f towards them (current buffer)
int32_t cxb_grid_get_messages(cxb_grid* g, int32_t which, void* out_host) try {
    Grid* h = GR(g);
    if (which < 0 || which > 7) {
        h->err = "message plane must be 0..7";
        return CXB_ERR_BAD_ARG;
    }
    const unsigned char* src = which < 4 ? h->m2v.p + (size_t)which * h->plane() : h->m2f[h->cur].p + (size_t)(which - 4) * h->plane();
    GR_CUDA(g, cudaSetDevice(h->device));
    if (which < 4)
        if (int32_t st = h->flush(true, false)) return st;
    GR_CUDA(g, cudaMemcpyAsync(out_host, src, h->plane(), cudaMemcpyDeviceToHost, h->stream));
    GR_CUDA(g, cudaStreamSynchronize(h->stream));
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
void* cxb_grid_stream(cxb_grid* g) { return (void*)GR(g)->stream; }
int32_t cxb_grid_last_kernel_ms(cxb_grid* g, float* ms_out) try {
    Grid* h = GR(g);
    if (!h->ran) {
        h->err = "no sweep has run yet";
        return CXB_ERR_STATE;
    }
    GR_CUDA(g, cudaEventSynchronize(h->ev1));
    GR_CUDA(g, cudaEventElapsedTime(ms_out, h->ev0, h->ev1));
    return CXB_OK;
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_grid_infer_host(cxb_grid* g, const void* unary_host, void* marginals_out_host, int32_t n_sweeps, int64_t* n_updates_out) try {
    return GR(g)->infer_host(unary_host, marginals_out_host, n_sweeps, n_updates_out);
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)
int32_t cxb_grid_sync(cxb_grid* g) try {
    return GR(g)->sync_all();
} CXB_ABI_CATCH(CXB_ERR_INTERNAL)

}  // extern "C"
