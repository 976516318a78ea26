// b200lasso.cu -- libb200lasso.so: sm_100a implementation of the lasso block
// proximal-gradient hot path (C ABI declared in include/b200lasso.h).
//
// Reference being replaced (kingold5/convex_optimization, file:line under the
// reference tree):
//   * iteration              lasso.py:102-157 (CPU), :228-278 (GPU mat-vecs), :508-599 (cuBLAS)
//   * A_m^T r  / A_m d       gpu_calculation.py:20-55 / :58-91 (hand kernels), lasso.py:350-353
//   * diag(A^T A)            gpu_calculation.py:116-137, cpu_calculation.py:35-42
//   * prox / error           cpu_calculation.py:5-20
//
// Design (see DESIGN.md): one persistent cooperative kernel runs whole solves.  Each CTA
// owns a fixed slab of rows of A for every column block, so its slice of the residual r
// and of q = A_m D never leaves shared memory.  A producer warp streams the slab tile by
// tile with TMA bulk copies (cp.async.bulk -> UBLKCP) into an mbarrier ring; 16 consumer
// warps use each tile for the block gradient (pass 1) and for A_m D (pass 2).  Only the
// partial block gradients (w values per CTA), the step D (w values) and four scalars per
// CTA cross CTAs, through L2, with two grid barriers per block step.  The step size of
// block t is resolved lazily at the first barrier of block t+1
// (g_{t+1} = A^T r + gamma A^T q), which removes the third barrier.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <type_traits>
#include <vector>

#include "b200lasso.h"

// ------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------
static thread_local char g_err[768] = "";

static int fail(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}

#define CK(call)                                                                   \
    do {                                                                           \
        cudaError_t e_ = (call);                                                   \
        if (e_ != cudaSuccess)                                                     \
            return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
                        __FILE__, __LINE__);                                       \
    } while (0)

// ------------------------------------------------------------------------------------
// constants / small device helpers
// ------------------------------------------------------------------------------------
constexpr int NW = 8;                  // consumer warps
constexpr int NTC = NW * 32;           // consumer threads
// + one helper warpgroup: warp 8 = TMA producer, multi-GPU: warp 9 sends my partial rows, warp 10
// collects the peers'; warp 11 idles.  Twelve warps are launched with 168 registers each (what a
// 384-thread CTA can have); the helper warpgroup then hands most of its share to the consumers
// (setmaxnreg), whose inner loops want many loads in flight.
constexpr int NTHREADS = NTC + 128;
constexpr int HELPER_REGS = 56, CONSUMER_REGS = 224;            // 256 * 224 + 128 * 56 = 64512 = 384 * 168
// (the collector warp keeps up to 21 words per lane in flight.  Measured with other splits, 2 GPUs, C2 shards:
// consumers 192 / helpers 120: 1037 shard sweeps/s, 208 / 88: 899, 224 / 56: 771 against 1202 -- the spills of the
// helper warps sit on the critical path of every step)
constexpr int HELPER_REGS_MG = 152, CONSUMER_REGS_MG = 176;
constexpr int MAX_CS = 64;             // max stage-2 slice width (columns per CTA)

template <typename T> struct VT;
template <> struct VT<float> { using type = float4; static constexpr int V = 4; };
template <> struct VT<double> { using type = double2; static constexpr int V = 2; };

__device__ __forceinline__ float vdot(const float4 a, const float4 b) {
    return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
}
__device__ __forceinline__ double vdot(const double2 a, const double2 b) {
    return a.x * b.x + a.y * b.y;
}
__device__ __forceinline__ void vfma(float (&acc)[4], const float4 v, const float s) {
    acc[0] += v.x * s; acc[1] += v.y * s; acc[2] += v.z * s; acc[3] += v.w * s;
}
__device__ __forceinline__ void vfma(double (&acc)[2], const double2 v, const double s) {
    acc[0] += v.x * s; acc[1] += v.y * s;
}
__device__ __forceinline__ float4 vpack(const float (&a)[4]) { return make_float4(a[0], a[1], a[2], a[3]); }
__device__ __forceinline__ double2 vpack(const double (&a)[2]) { return make_double2(a[0], a[1]); }
__device__ __forceinline__ float4 vadd(const float4 a, const float4 b) {
    return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ double2 vadd(const double2 a, const double2 b) {
    return make_double2(a.x + b.x, a.y + b.y);
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// TMA 1-D bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes,
                                             uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// TMA 2-D tiled copy global -> shared through a tensor map (SASS: UTMALDG), and its L2 prefetch
__device__ __forceinline__ void tma_load_2d(void *dst_smem, const CUtensorMap *tmap, int x, int y,
                                            uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
            "r"(smem_u32(dst_smem)),
        "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap *tmap, int x, int y) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(tmap), "r"(x), "r"(y)
                 : "memory");
}
// TMA prefetch of a contiguous range into L2 (no shared memory involved; SASS: UBLKPF)
__device__ __forceinline__ void tma_prefetch_l2(const void *src_gmem, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cbar() {  // barrier over the consumer threads only
    asm volatile("bar.sync 1, %0;" ::"n"(NTC) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// phase / tile stamps of the traced runs: the SM's cycle counter (reading %globaltimer costs
// ~0.2 us a time, which distorts a 12 us step; the trace carries a (globaltimer, clock) pair per
// CTA at both ends of the launch to convert cycles to time)
__device__ __forceinline__ unsigned long long tstamp() { return (unsigned long long)clock64(); }
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ------------------------------------------------------------------------------------
// cross-CTA exchange: self-validating "LL" words
// ------------------------------------------------------------------------------------
// Every 8-byte half of a 16-byte word carries 32 bits of payload and a 32-bit tag (the
// context-wide step number, never 0).  A reader polls the word itself until both tags
// match, so the exchange needs no separate flag, fence or atomic: naturally aligned 64-bit
// accesses are single-copy atomic and each half validates itself.  One store latency plus
// one load latency per exchange, instead of store / fence / atomic / poll / load.
// Polling loads are plain L2 (.cg) loads on purpose: a batch of them is issued back to back
// and waited on once.  (ld.volatile makes ptxas interleave each tag check with the next
// load, which serialises the round trips.)  L1 is bypassed, so a re-read after the opaque
// Waiter::again() call observes the writer's store.
__device__ __forceinline__ ulonglong2 ll_ld(const ulonglong2 *p) { return __ldcg(p); }
__device__ __forceinline__ void ll_st(ulonglong2 *p, unsigned long long a, unsigned long long b) {
    asm volatile("st.volatile.global.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ unsigned long long ll_ld1(const unsigned long long *p) { return __ldcg(p); }
__device__ __forceinline__ void ll_st1(unsigned long long *p, unsigned long long a) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(a) : "memory");
}
// two adjacent words with one 256-bit store (whole 32-byte sectors; p 32-byte aligned)
__device__ __forceinline__ void ll_st2(ulonglong2 *p, unsigned long long a, unsigned long long b,
                                       unsigned long long c, unsigned long long d) {
    asm volatile("st.global.v4.u64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}
__device__ __forceinline__ unsigned long long ll_pack(uint32_t payload, uint32_t tag) {
    return ((unsigned long long)tag << 32) | (unsigned long long)payload;
}
__device__ __forceinline__ bool ll_ok(const ulonglong2 v, uint32_t tag) {
    return (uint32_t)(v.x >> 32) == tag && (uint32_t)(v.y >> 32) == tag;
}
__device__ __forceinline__ double ll_dbl(const ulonglong2 v) {
    return __hiloint2double((int)(uint32_t)v.y, (int)(uint32_t)v.x);
}
__device__ __forceinline__ void ll_st_dbl(ulonglong2 *p, double a, uint32_t tag) {
    ll_st(p, ll_pack((uint32_t)__double2loint(a), tag), ll_pack((uint32_t)__double2hiint(a), tag));
}
// the same word through a multicast (NVLS) mapping: ONE store, delivered by the switch to the
// replica of every GPU bound to the multicast object (SASS: a multimem store)
__device__ __forceinline__ void mm_st_dbl(ulonglong2 *p, double a, uint32_t tag) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p),
                 "f"(__int_as_float(__double2loint(a))), "f"(__uint_as_float(tag)),
                 "f"(__int_as_float(__double2hiint(a))), "f"(__uint_as_float(tag))
                 : "memory");
}

// per-type encoding of the exchanged values: (g_r, g_q) of a column as two floats in one
// word or one word per double; the step D as one 8-byte word per float or one 16-byte word
// per double
template <typename T> struct LLW;
template <> struct LLW<float> {
    static constexpr int WPC = 1;
    __device__ static __forceinline__ void put(ulonglong2 *p, float a, float b, uint32_t tag) {
        ll_st(p, ll_pack(__float_as_uint(a), tag), ll_pack(__float_as_uint(b), tag));
    }
    __device__ static __forceinline__ void get(const ulonglong2 (&v)[1], double &a, double &b) {
        a = (double)__uint_as_float((uint32_t)v[0].x);
        b = (double)__uint_as_float((uint32_t)v[0].y);
    }
    // the step D: one 16-byte word per column (dpw = 1: payload in the first half) or two columns
    // per word (dpw = 2: one 8-byte half each)
    __device__ static __forceinline__ void dwords(float v, uint32_t tag, unsigned long long &w0, unsigned long long &w1) {
        w0 = ll_pack(__float_as_uint(v), tag);
        w1 = ll_pack(0u, tag);
    }
    __device__ static __forceinline__ void dget(const ulonglong2 v, int dpw, float *out) {
        out[0] = __uint_as_float((uint32_t)v.x);
        if (dpw == 2) out[1] = __uint_as_float((uint32_t)v.y);
    }
    // the four columns of one column group: words p[0..3] = (g_r, g_q) pairs
    __device__ static __forceinline__ void put_group(ulonglong2 *p, const float4 r, const float4 q, uint32_t tag) {
        ll_st2(p, ll_pack(__float_as_uint(r.x), tag), ll_pack(__float_as_uint(q.x), tag),
               ll_pack(__float_as_uint(r.y), tag), ll_pack(__float_as_uint(q.y), tag));
        ll_st2(p + 2, ll_pack(__float_as_uint(r.z), tag), ll_pack(__float_as_uint(q.z), tag),
               ll_pack(__float_as_uint(r.w), tag), ll_pack(__float_as_uint(q.w), tag));
    }
};
template <> struct LLW<double> {
    static constexpr int WPC = 2;
    __device__ static __forceinline__ void put(ulonglong2 *p, double a, double b, uint32_t tag) {
        // one 32-byte sector, one store (p is an even word of a 256-byte aligned array)
        ll_st2(p, ll_pack((uint32_t)__double2loint(a), tag), ll_pack((uint32_t)__double2hiint(a), tag),
               ll_pack((uint32_t)__double2loint(b), tag), ll_pack((uint32_t)__double2hiint(b), tag));
    }
    __device__ static __forceinline__ void get(const ulonglong2 (&v)[2], double &a, double &b) {
        a = ll_dbl(v[0]);
        b = ll_dbl(v[1]);
    }
    __device__ static __forceinline__ void dwords(double v, uint32_t tag, unsigned long long &w0, unsigned long long &w1) {
        w0 = ll_pack((uint32_t)__double2loint(v), tag);
        w1 = ll_pack((uint32_t)__double2hiint(v), tag);
    }
    __device__ static __forceinline__ void dget(const ulonglong2 v, int, double *out) { out[0] = ll_dbl(v); }
    // the two columns of one column group: words p[0..3] = g_r, g_q, g_r, g_q
    __device__ static __forceinline__ void put_group(ulonglong2 *p, const double2 r, const double2 q, uint32_t tag) {
        ll_st2(p, ll_pack((uint32_t)__double2loint(r.x), tag), ll_pack((uint32_t)__double2hiint(r.x), tag),
               ll_pack((uint32_t)__double2loint(q.x), tag), ll_pack((uint32_t)__double2hiint(q.x), tag));
        ll_st2(p + 2, ll_pack((uint32_t)__double2loint(r.y), tag), ll_pack((uint32_t)__double2hiint(r.y), tag),
               ll_pack((uint32_t)__double2loint(q.y), tag), ll_pack((uint32_t)__double2hiint(q.y), tag));
    }
};

constexpr int NTTRACE = 96;        // per-tile stamps: 6 groups of 16 (see b200lasso.h)
constexpr int NTRACE = 16;         // time stamps per CTA and step of b200l_run_traced
// b200l_debug_flags: bits 0-2 switch parts of the fused kernel off to time the rest (1 exchange waits,
// 2 pass-1 math, 4 pass-2 math; the diagnostic instantiation, results meaningless), bit 18 keeps the
// step-wise mat-vecs on the load-batch kernels (results valid)
constexpr int32_t DBG_KNOCKOUTS = 7, DBG_LOAD_BATCH = 262144;
constexpr int NB = 8;              // exchange words a thread keeps in flight per round trip
constexpr int GMAX = 160;          // largest grid (sizes the acknowledgement words of the step-D exchange)

// ------------------------------------------------------------------------------------
// fused kernel parameters
// ------------------------------------------------------------------------------------
struct Ctl {
    double sp[4];                    // this CTA's line-search scalars of the pending step
    unsigned long long kc, k_issued;
    int stop;
    int abort;
    long long gate;                  // steps whose pass-2 copies the producer may issue
    long long gate2;                 // steps whose step-D gather is complete (pass-2 tiles past the first gate2_tiles)
    long long sc_go, sc_done;        // steps whose scalars are final in sp / whose totals are in tot (scalar warp)
    double tot[4];                   // line-search scalars of the pending step summed over all CTAs
    long long qready;                // multi-GPU: (step + 1) << 32 | rows of A_m D summed over the ranks
    long long p2start, p2done;       // multi-GPU: steps whose pass 2 (my partial rows) has begun / is complete
    long long own_rows;              // multi-GPU: (step + 1) << 32 | my rows that are final (and sent)
    double qsc[2];                   // multi-GPU: l1 / err terms summed over the ranks (until the step is complete)
    int hstop;                       // multi-GPU: the consumers are done, the collector warp exits
    unsigned long long t_start;      // time base of the phase trace
};

struct RunParams {
    const void *A;
    int64_t N;
    int64_t blk_stride;  // elements between consecutive blocks
    int32_t w, ld, nblocks;
    double *x;           // [nblocks][ld]
    const double *d;     // [nblocks][ld]
    const double *drec;  // [nblocks][ld]
    double *r;           // [N]
    ulonglong2 *gLL;     // [G readers][G writers][mw]  partial block gradients
    ulonglong2 *sLL;     // [G writers][4]              line-search scalars of the pending step
    ulonglong2 *dLL;     // [ld + acks]                 the step D
    int *abort_flag;
    const int32_t *order;
    int64_t nsteps, step0;
    double mu, err_bound;
    int32_t bounded;
    double *err_hist;
    unsigned long long *time_hist;
    long long *state;     // [0] steps_done [1] stopped [2] block_cnt [3] aborted
    double *gamma_state;  // [0] last gamma
    unsigned long long *trace;  // optional [G][nsteps][NTRACE] phase time stamps (ns since start)
    unsigned long long *ttrace; // optional [G][nsteps][NTTRACE] per-tile time stamps (absolute ns)
    uint32_t tag_base;
    unsigned long long wait_limit_ns;
    // geometry
    int32_t TR, S, slot_bytes, cs, cs_shift, nrg, ncg, rows_pad, rows_max_, l2_ahead;
    // multi-GPU: rank `rank` of `world` holds column slice `rank` of every block; peer[r] is the
    // q-inbox of rank r: [2 parities][G CTAs][world sources][qw] words (peer[rank] is local)
    int32_t tile_sends;       // multi-GPU send side: 1 the sender warp sends finished pass-2 tiles, 0 the lane that finishes a row sends it
    int32_t world, rank, qw;  // qw: words per rank in a cell
    ulonglong2 *peer[B200L_MAX_WORLD];
    ulonglong2 *mc;           // multicast mapping of all ranks' inboxes (NVLS) or NULL
    int32_t direct_pub;       // partial gradients are published from registers (one row group)
    int32_t dbg;              // diagnostics only: 1 skip exchange waits, 2 skip pass-1 math, 4 skip pass-2 math
    int32_t gate2_tiles;      // > 0: only this many pass-2 tiles are staged before the step-D gather is complete
    // transposed layout: a tile is TJ block columns x BX residual entries of this CTA
    // (BX/V odd: conflict-free 16-byte reads with lanes on consecutive columns)
    // A CTA's BX entries come as NBX boxes of BXb = BXVb * V entries each (TMA boxes hold at most 256 elements per
    // dimension); P1 threads share a column in pass 1 (TJ * P1 = consumer threads), BXVb = P1 * odd keeps their
    // 16-byte reads conflict-free.
    int32_t BX, BXV, TJ, nparts, nt_t, off_red2;
    int32_t NBX, BXb, BXVb, P1;
    int32_t mw, mw_shift, nown;     // message words (a power of two), owner CTAs
    int32_t dpw, dsec, ackbase;     // step D: columns per 16-byte word, published by whole sectors, first acknowledgement word
    // shared-memory offsets
    int32_t off_bar, off_ctl, off_rloc, off_qloc, off_rT, off_qT, off_delta, off_redT, off_red,
        off_small, off_qpart, off_tilecnt, ring_bytes;
};

// bounded spinning: returns false when the wait has to be abandoned (a peer timed out or
// this wait exceeded the limit) so that a lost CTA can never hang the device
struct Waiter {
    volatile int *gabort;
    volatile int *sabort;
    unsigned long long limit_ns;
    unsigned spins;
    unsigned long long t0;
    long long *diag;              // state[4..7]: where the first abandoned wait happened
    long long info;
    __device__ __forceinline__ void begin(long long where = 0) { spins = 0; t0 = 0; info = where; }
    __device__ __noinline__ bool again() {
        ++spins;
        if (spins > 8u) __nanosleep(20);
        if ((spins & 63u) == 0u && *sabort) return false;
        if ((spins & 1023u) == 0u) {
            if (*gabort) { *sabort = 1; return false; }
            const unsigned long long now = globaltimer_ns();
            if (t0 == 0) {
                t0 = now;
            } else if (now - t0 > limit_ns) {
                if (atomicExch((int *)gabort, 1) == 0) {
                    diag[0] = blockIdx.x;
                    diag[1] = threadIdx.x;
                    diag[2] = info;
                }
                *sabort = 1;
                return false;
            }
        }
        return true;
    }
};

// load 4 consecutive entries of a T vector in shared memory (16-byte aligned for float)
__device__ __forceinline__ void load4(const float *p, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4 *>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void load4(const double *p, double (&v)[4]) {
    const double2 a = *reinterpret_cast<const double2 *>(p);
    const double2 b = *reinterpret_cast<const double2 *>(p + 2);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ float4 vzero(float4) { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ double2 vzero(double2) { return make_double2(0.0, 0.0); }
__device__ __forceinline__ void vunpack(const float4 v, float (&a)[4]) { a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w; }
__device__ __forceinline__ void vunpack(const double2 v, double (&a)[2]) { a[0] = v.x; a[1] = v.y; }

// ring cursor: slot index and phase parity advance without divisions
struct Cursor {
    int slot;
    uint32_t phase;
    __device__ __forceinline__ void advance(int S) {
        if (++slot == S) { slot = 0; phase ^= 1u; }
    }
};

// ------------------------------------------------------------------------------------
// the fused persistent kernel, row-major blocks (nblocks, N, ld)
// ------------------------------------------------------------------------------------
// 8 consumer warps + 1 producer warp per CTA, one CTA per SM.  Few fat warps on purpose: the
// passes are bound by instruction issue unless every thread does enough work per tile to
// amortise the ring handshake (DESIGN.md "why 8 warps").  The per-step code is kept small
// (rolled loops, one copy of every phase): it runs once per block step and has to stay
// resident in the instruction cache.
//
// per-type arithmetic on one 16-byte column group
template <typename T> struct Ops;
template <> struct Ops<float> {
    struct Acc { float2 lo, hi; };
    __device__ static __forceinline__ unsigned long long u(const float2 v) {
        return *reinterpret_cast<const unsigned long long *>(&v);
    }
    __device__ static __forceinline__ float2 fma2(const float2 a, const float2 b, const float2 c) {
        unsigned long long d;   // packed FFMA2: two fp32 fused multiply-adds per instruction
        asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(u(a)), "l"(u(b)), "l"(u(c)));
        return *reinterpret_cast<float2 *>(&d);
    }
    __device__ static __forceinline__ void zero(Acc &a) { a.lo = make_float2(0.f, 0.f); a.hi = a.lo; }
    // a += v * s  (four columns of one row)
    __device__ static __forceinline__ void axpy(Acc &a, const float4 v, const float s) {
        const float2 ss = make_float2(s, s);
        a.lo = fma2(make_float2(v.x, v.y), ss, a.lo);
        a.hi = fma2(make_float2(v.z, v.w), ss, a.hi);
    }
    // a += v * d elementwise (partial dot product of one row)
    __device__ static __forceinline__ void mac(Acc &a, const float4 v, const float4 d) {
        a.lo = fma2(make_float2(v.x, v.y), make_float2(d.x, d.y), a.lo);
        a.hi = fma2(make_float2(v.z, v.w), make_float2(d.z, d.w), a.hi);
    }
    __device__ static __forceinline__ float hsum(const Acc &a) { return (a.lo.x + a.lo.y) + (a.hi.x + a.hi.y); }
    __device__ static __forceinline__ float4 pack(const Acc &a) { return make_float4(a.lo.x, a.lo.y, a.hi.x, a.hi.y); }
};
template <> struct Ops<double> {
    struct Acc { double x, y; };
    __device__ static __forceinline__ void zero(Acc &a) { a.x = 0.0; a.y = 0.0; }
    __device__ static __forceinline__ void axpy(Acc &a, const double2 v, const double s) {
        a.x = fma(v.x, s, a.x);
        a.y = fma(v.y, s, a.y);
    }
    __device__ static __forceinline__ void mac(Acc &a, const double2 v, const double2 d) {
        a.x = fma(v.x, d.x, a.x);
        a.y = fma(v.y, d.y, a.y);
    }
    __device__ static __forceinline__ double hsum(const Acc &a) { return a.x + a.y; }
    __device__ static __forceinline__ double2 pack(const Acc &a) { return make_double2(a.x, a.y); }
};

// sums of two values over the warp with 5+1 shuffles: returns the sum of `a` in lanes 0..15
// and the sum of `b` in lanes 16..31
template <typename T>
__device__ __forceinline__ T warp_sum_pair(const T a, const T b, const int lane) {
    const bool up = lane >= 16;
    T mine = up ? b : a;
    const T give = up ? a : b;
    mine += __shfl_xor_sync(0xffffffffu, give, 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    return mine;
}

// CPT : column groups (16-byte vectors) per thread in pass 1 (ld/V <= CPT*NTC).  CPT == 1 also
//       means at most 8 column groups per lane in pass 2, whose slice of the step D then lives
//       in registers; wider blocks read D from shared memory.
// TRANS: blocks are stored pre-transposed, (w, ldT >= N) row-major per block; a CTA's share of a
//       block is then a 2-D box (all columns x its residual entries), fetched tile by tile
//       through a tensor map.  Pass 1 is a row-dot per column (thread = column), pass 2 an
//       axpy over columns (thread = (16-byte group of residual entries, column part)).
// MODE : 0 = the plain single-GPU solve, 1 = with the multi-GPU exchange (sender / collector warps),
//       2 = 1 + the phase / tile tracing and the diagnostic switches.  Three instantiations because
//       the per-step code has to stay resident in the instruction cache and every rarely used
//       branch costs footprint (and registers in the inner loops).
template <typename T, int CPT, bool TRANS, int MODE>
__global__ void __launch_bounds__(NTHREADS, 1) lasso_fused(const RunParams p, const __grid_constant__ CUtensorMap tmap) {
    using VecT = typename VT<T>::type;
    using LL = LLW<T>;
    using OP = Ops<T>;
    using Acc = typename OP::Acc;
    constexpr int V = VT<T>::V;
    constexpr int WPC = LL::WPC;
    constexpr int DK = CPT == 1 ? NTC / 32 : 0;
    constexpr bool MG = MODE >= 1, DIAG = MODE == 2;
    // pre-transposed layout: CPT selects the tile shape -- 1: one thread and one TMA box per column (N / #SM <= 252
    // entries, C2), 2: the general shape (P1 threads per column, NBX boxes); a runtime switch cost 2.7 % on C2
    constexpr bool TGEN = TRANS && CPT > 1;
    const int WORLD = MG ? p.world : 1, DBG = DIAG ? p.dbg : 0;
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char *ring = smem;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + p.off_bar);
    uint64_t *empty = full + p.S;
    Ctl *ctl = reinterpret_cast<Ctl *>(smem + p.off_ctl);
    double *r_loc = reinterpret_cast<double *>(smem + p.off_rloc);
    double *q_loc = reinterpret_cast<double *>(smem + p.off_qloc);
    T *rT = reinterpret_cast<T *>(smem + p.off_rT);
    T *qT = reinterpret_cast<T *>(smem + p.off_qT);
    T *delta_s = reinterpret_cast<T *>(smem + p.off_delta);
    T *redT = reinterpret_cast<T *>(smem + p.off_redT);
    double2 *red = reinterpret_cast<double2 *>(smem + p.off_red);         // [NTC] gather partials per thread
    double *l1s = reinterpret_cast<double *>(smem + p.off_small);
    double *es = l1s + MAX_CS;
    double *lsred = l1s + 2 * MAX_CS;     // [2][NW] line-search partials of the warps
    double *qpart = reinterpret_cast<double *>(smem + p.off_qpart);       // [rows] A_m D
    int *tilecnt = reinterpret_cast<int *>(smem + p.off_tilecnt);         // warps done with a pass-2 tile

    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    const int c = blockIdx.x, G = gridDim.x;
    // rows of this CTA: an even split of N (TRANS: of the 16-byte groups of N, because the inner
    // coordinate of a tensor-map box has to be 16-byte aligned)
    const int64_t nunits = TRANS ? (p.N + V - 1) / V : p.N;
    const int64_t base = nunits / G;
    const int rem = (int)(nunits % G);
    const int64_t unit0 = (int64_t)c * base + (c < rem ? c : rem);
    const int64_t row0 = TRANS ? unit0 * V : unit0;
    const int rows_c = TRANS ? (int)max((int64_t)0, min((base + (c < rem ? 1 : 0)) * V, p.N - row0))
                             : (int)base + (c < rem ? 1 : 0);
    const int TR = p.TR, S = p.S, ld = p.ld, ncg = p.ncg;
    const int nt = TRANS ? (rows_c > 0 ? p.nt_t : 0) : (rows_c + TR - 1) / TR;
    const T *Aall = reinterpret_cast<const T *>(p.A);

    // the ring starts zero-filled (defined contents for the parts of a slot no copy writes)
    for (int i = tid; i < p.ring_bytes / 16; i += (int)blockDim.x)
        reinterpret_cast<uint4 *>(ring)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, NW);
        }
        ctl->sp[0] = ctl->sp[1] = ctl->sp[2] = ctl->sp[3] = 0.0;
        ctl->stop = 0;
        ctl->abort = 0;
        ctl->gate = 0;
        ctl->gate2 = 0;
        ctl->sc_go = 0;
        ctl->sc_done = 0;
        ctl->qready = 0;
        ctl->p2done = 0;
        ctl->p2start = 0;
        ctl->own_rows = 0;
        ctl->hstop = 0;
        for (int i = 0; i < 128; ++i) tilecnt[i] = 0;
        ctl->kc = 0;
        ctl->k_issued = 0;
        fence_mbar_init();
    }
    // order the generic-proxy zero fill before the async-proxy (TMA) writes into the ring
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    // register re-balancing between the warpgroups: every warp of a warpgroup executes it, first
    // thing in its role branch (the allocator sizes each branch by the limit set inside it)
    if (wid >= NW) {
        if (MG) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(HELPER_REGS_MG));
        else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(HELPER_REGS));
    if (wid == NW) {
        // ============================ producer warp ================================
        if (lane == 0) {
            unsigned long long k = 0;   // tiles issued
            Cursor cur{0, 1u};   // waits on "empty" with the inverted parity
            volatile int *stopf = &ctl->stop;
            bool live = true;
            int mc = (int)(p.step0 % p.nblocks);
            const uint32_t tile_bytes = (uint32_t)TR * (uint32_t)ld * (uint32_t)sizeof(T);
            const uint32_t last_bytes = (uint32_t)(rows_c - (nt - 1) * TR) * (uint32_t)ld * (uint32_t)sizeof(T);
            for (int64_t step = 0; step < p.nsteps && live; ++step) {
                const int m = p.order ? p.order[step] : mc;
                if (++mc == p.nblocks) mc = 0;
                const unsigned char *Ab =
                    reinterpret_cast<const unsigned char *>(Aall + (int64_t)m * p.blk_stride + row0 * (int64_t)ld);
                const unsigned char *An = nullptr;   // slab of the next step, prefetched into L2
                if (p.l2_ahead && step + 1 < p.nsteps) {
                    const int mn = p.order ? p.order[step + 1] : mc;
                    An = reinterpret_cast<const unsigned char *>(Aall + (int64_t)mn * p.blk_stride + row0 * (int64_t)ld);
                }
                const int ym = m * p.w, yn = (p.order ? (step + 1 < p.nsteps ? p.order[step + 1] : 0) : mc) * p.w;
                for (int pass = 0; pass < 2 && live; ++pass) {
                    // the re-stream for pass 2 waits (gate) until this CTA's gather is complete: issued
                    // earlier, the tiles queue the gather's loads behind them on the L2 link
                    if (pass == 1) {
                        while (*(volatile long long *)&ctl->gate <= step) {
                            if (*stopf) { live = false; break; }
                            __nanosleep(64);
                        }
                        if (!live) break;
                    }
                    for (int t = 0; t < nt; ++t) {
                        if (pass == 1 && p.gate2_tiles && t >= p.gate2_tiles) {
                            while (*(volatile long long *)&ctl->gate2 <= step) {
                                if (*stopf) { live = false; break; }
                            }
                            if (!live) break;
                        }
                        while (!mbar_try_wait(empty + cur.slot, cur.phase)) {
                            if (*stopf) { live = false; break; }
                        }
                        if (!live) break;
                        if (TRANS) {
                            mbar_expect_tx(full + cur.slot, (uint32_t)(p.TJ * p.BX) * (uint32_t)sizeof(T));
                            for (int bx = 0; bx < (TGEN ? p.NBX : 1); ++bx) {
                                tma_load_2d(ring + (size_t)cur.slot * p.slot_bytes + (size_t)bx * p.TJ * p.BXb * sizeof(T),
                                            &tmap, (int)row0 + bx * p.BXb, ym + t * p.TJ, full + cur.slot);
                                if (pass == 1 && An) tma_prefetch_2d(&tmap, (int)row0 + bx * p.BXb, yn + t * p.TJ);
                            }
                        } else {
                            const uint32_t bytes = t == nt - 1 ? last_bytes : tile_bytes;
                            mbar_expect_tx(full + cur.slot, bytes);
                            tma_bulk_g2s(ring + (size_t)cur.slot * p.slot_bytes, Ab + (size_t)t * tile_bytes, bytes,
                                         full + cur.slot);
                            // HBM runs one block ahead of the passes: while this step streams its slab
                            // (from L2), pull the slab of the next step into L2
                            if (pass == 1 && An) tma_prefetch_l2(An + (size_t)t * tile_bytes, bytes);
                        }
                        if (DIAG && p.ttrace && t < 16 && WORLD == 1)
                            p.ttrace[((size_t)c * p.nsteps + step) * NTTRACE + 64 + pass * 16 + t] = tstamp();
                        cur.advance(S);
                        ++k;
                    }
                }
            }
            ctl->k_issued = k;
        }
        __syncwarp();
    } else if (wid == NW + 1) {
        // ============== multi-GPU: sender of my partial A_m D ======================
        // My partial rows go to the peers tile by tile, as soon as the 8 consumer warps are done
        // with a pass-2 tile: consecutive lanes = consecutive words (whole NVLink packets), and
        // the peer stores stay out of the inner loop of pass 2.  (TRANS, or more tiles than
        // counters: the consumers send their rows themselves.)
        if (WORLD > 1 && p.tile_sends) {
            Waiter hw{p.abort_flag, &ctl->abort, p.wait_limit_ns, 0u, 0ull, p.state + 4, 0};
            bool live = true;
            for (long long hs = 0; live; ++hs) {
                const uint32_t tag = p.tag_base + (uint32_t)hs + 1u;
                unsigned spin = 0;
                while (!__all_sync(0xffffffffu, *(volatile long long *)&ctl->p2start > hs)) {
                    if (__any_sync(0xffffffffu, *(volatile int *)&ctl->hstop != 0)) {
                        live = false;
                        break;
                    }
                    __nanosleep(64);
                }
                if (!live) break;
                hw.begin((hs << 32) | (3LL << 30));
                const size_t mine = (((size_t)(tag & 1u) * G + c) * WORLD + p.rank) * p.qw;
                __threadfence_block();
                if (lane < 2) {                // l1 and err terms of my columns (set before pass 2)
                    const double v = ctl->sp[2 + lane];
                    if (p.mc) {
                        mm_st_dbl(p.mc + mine + rows_c + lane, v, tag);
                    } else {
#pragma unroll 1
                        for (int pr = 0; pr < WORLD; ++pr)
                            if (pr != p.rank) ll_st_dbl(p.peer[pr] + mine + rows_c + lane, v, tag);
                    }
                }
#pragma unroll 1
                for (int t = 0; t < nt; ++t) {
                    // (naps: this warp shares its scheduler with two consumer warps)
                    while (!__all_sync(0xffffffffu, *(volatile int *)&tilecnt[t & 127] >= NW)) {
                        __nanosleep(100);
                        if ((++spin & 63u) == 0u && !__all_sync(0xffffffffu, hw.again())) break;
                    }
                    __threadfence_block();
                    const int rows_t = min(TR, rows_c - t * TR);
#pragma unroll 1
                    for (int i = lane; i < rows_t; i += 32) {
                        const double v = qpart[t * TR + i];
                        if (p.mc) {            // one store, the switch delivers it to every rank
                            mm_st_dbl(p.mc + mine + t * TR + i, v, tag);
                        } else {
#pragma unroll 1
                            for (int pr = 0; pr < WORLD; ++pr)
                                if (pr != p.rank) ll_st_dbl(p.peer[pr] + mine + t * TR + i, v, tag);
                        }
                    }
                    __syncwarp();
                    if (DIAG && p.ttrace && lane == 0 && t < 16)
                        p.ttrace[((size_t)c * p.nsteps + hs) * NTTRACE + 64 + t] = tstamp();
                    if (lane == 0) {
                        tilecnt[t & 127] = 0;
                        // my rows of this tile are final: the collector may add them up
                        *(volatile long long *)&ctl->own_rows = ((hs + 1) << 32) | (long long)min((t + 1) * TR, rows_c);
                    }
                }
            }
        }
    } else if (wid == NW + 2) {
        // ============== multi-GPU: collector of the peers' partial A_m D ===========
        // (the reduce of lasso.py:126 over the reference's P column slices).  CTA c of every
        // rank owns the same rows; during pass 2 each rank stores its finished rows (and its
        // l1 / err terms) as tagged words straight into the inbox of CTA c on every peer
        // (NVLink peer stores).  This warp polls them from the start of pass 2 and, while the
        // consumers already run pass 1 of the next step -- which needs the summed rows tile by
        // tile, in the order they were sent --, releases every row as soon as all ranks' parts
        // are there: the NVLink latency hides behind the streaming.  Sums in rank order: every
        // rank holds bitwise the same q, gamma and r.  Cells are double-buffered by step parity:
        // a rank can be at most one exchange ahead.
        if (WORLD > 1) {
            Waiter hw{p.abort_flag, &ctl->abort, p.wait_limit_ns, 0u, 0ull, p.state + 4, 0};
            const int nq = rows_c + 2;                       // rows, then the l1 and err terms
            constexpr int CH = 3;                            // C2 shard: 68 rows + 2 scalars = one batch
            bool live = true;
            for (long long hs = 0; live; ++hs) {
                const uint32_t tag = p.tag_base + (uint32_t)hs + 1u;
                const ulonglong2 *mycell = p.peer[p.rank] + (((size_t)(tag & 1u) * G + c) * WORLD) * p.qw;
                double trq = 0.0, tqq = 0.0;
                int own_rows = 0;                            // my own rows below this index are final
                int rel_t = 0;                               // (trace) tiles whose rows have been released
                int last_ready = -1;
                unsigned spin = 0;
                // nothing can arrive before the ranks are in pass 2 of this step: nap until mine
                // begins (shared-memory flag, no L2 traffic)
                while (!__all_sync(0xffffffffu, *(volatile long long *)&ctl->p2start > hs)) {
                    if (__any_sync(0xffffffffu, *(volatile int *)&ctl->hstop != 0)) {
                        live = false;
                        break;
                    }
                    __nanosleep(64);
                }
                if (!live) break;
                hw.begin((hs << 32) | (2LL << 30));
#pragma unroll 1
                for (int i0 = 0; i0 < nq && live; i0 += 32 * CH) {   // CH x 32 words x (world-1) sources in flight
                    ulonglong2 w[CH][B200L_MAX_WORLD - 1];
                    bool done[CH];
#pragma unroll
                    for (int h = 0; h < CH; ++h) {
                        const int i = i0 + 32 * h + lane;
                        done[h] = i >= nq;
#pragma unroll
                        for (int k = 0; k < B200L_MAX_WORLD - 1; ++k)
                            if (k < WORLD - 1)
                                w[h][k] = ll_ld(mycell + (size_t)(k < p.rank ? k : k + 1) * p.qw + min(i, nq - 1));
                    }
                    for (;;) {
                        if (own_rows < rows_c) {
                            // final rows of my own partial product: what the sender warp has sent (so
                            // the consumers, who wait for this warp, can never overwrite rows the sender
                            // still has to read), or all of them once pass 2 is complete when the
                            // consumers send their rows themselves
                            const long long pd = *(volatile long long *)&ctl->p2done;
                            const long long orw = *(volatile long long *)&ctl->own_rows;
                            int mine_n = p.tile_sends ? ((orw >> 32) == hs + 1 ? (int)(orw & 0x7fffffff) : 0)
                                                   : (pd > hs ? rows_c : 0);
                            mine_n = __reduce_min_sync(0xffffffffu, mine_n);
                            if (mine_n > own_rows) {
                                own_rows = mine_n;
                                __threadfence_block();
                            } else if (mine_n == 0 && __any_sync(0xffffffffu, *(volatile int *)&ctl->hstop != 0)) {
                                live = false;                // the consumers are gone: no step hs
                                break;
                            }
                        }
#pragma unroll
                        for (int h = 0; h < CH; ++h) {
                            if (!done[h]) {
                                const int i = i0 + 32 * h + lane;
                                bool ok = true;
#pragma unroll
                                for (int k = 0; k < B200L_MAX_WORLD - 1; ++k) {
                                    if (k < WORLD - 1 && !ll_ok(w[h][k], tag)) {
                                        ok = false;
                                        w[h][k] = ll_ld(mycell + (size_t)(k < p.rank ? k : k + 1) * p.qw + i);
                                    }
                                }
                                if (ok && (i < own_rows || i >= rows_c)) {
                                    const double own = i < rows_c ? qpart[i] : ctl->sp[2 + (i - rows_c)];
                                    const bool is_max = i == rows_c + 1;
                                    double acc = 0.0;
#pragma unroll
                                    for (int k = 0; k < B200L_MAX_WORLD; ++k) {
                                        if (k == p.rank) acc = is_max ? fmax(acc, own) : acc + own;
                                        if (k < B200L_MAX_WORLD - 1 && k < WORLD - 1) {
                                            const double v = ll_dbl(w[h][k]);
                                            acc = is_max ? fmax(acc, v) : acc + v;
                                        }
                                    }
                                    if (i < rows_c) {
                                        q_loc[i] = acc;
                                        qT[i] = (T)acc;
                                        trq += r_loc[i] * acc;                           // lasso.py:129
                                        tqq += acc * acc;                                // lasso.py:132
                                    } else {
                                        ctl->qsc[i - rows_c] = acc;
                                    }
                                    done[h] = true;
                                }
                            }
                        }
                        // watchdog every 16th trip (the poll period is the L2 round trip)
                        if (((++spin & 15u) == 0u && !__all_sync(0xffffffffu, hw.again())) || (DBG & 1)) {
#pragma unroll
                            for (int h = 0; h < CH; ++h) done[h] = true;   // aborted: the consumers find the abort flag
                        }
                        int ready = i0 + 32 * CH;                // first row of this batch that is not summed yet
                        bool any = false;
#pragma unroll
                        for (int h = CH - 1; h >= 0; --h) {
                            const unsigned nd = __ballot_sync(0xffffffffu, !done[h]);
                            if (nd) { ready = i0 + 32 * h + __ffs(nd) - 1; any = true; }
                        }
                        __threadfence_block();
                        if (lane == 0)
                            *(volatile long long *)&ctl->qready = ((hs + 1) << 32) | (long long)min(ready, rows_c);
                        if (DIAG && p.ttrace && lane == 0) {
                            const unsigned long long now = tstamp();
                            for (; rel_t < 16 && rel_t * TR < rows_c && min((rel_t + 1) * TR, rows_c) <= ready; ++rel_t)
                                p.ttrace[((size_t)c * p.nsteps + hs) * NTTRACE + 80 + rel_t] = now;
                        }
                        if (!any) break;
                        // nothing new in this trip: nap instead of spinning -- this warp shares a scheduler
                        // with two consumer warps, and every tile waits for the slowest of the eight
                        if (ready == last_ready) __nanosleep(60);
                        last_ready = ready;
                    }
                }
                if (!live) break;
                trq = warp_sum(trq);
                tqq = warp_sum(tqq);
                __syncwarp();
                if (lane == 0) {
                    ctl->sp[0] = trq;
                    ctl->sp[1] = tqq;
                    ctl->sp[2] = ctl->qsc[0];
                    ctl->sp[3] = ctl->qsc[1];
                    __threadfence_block();
                    *(volatile long long *)&ctl->qready = ((hs + 1) << 32) | 0x7fffffffLL;
                    *(volatile long long *)&ctl->sc_go = hs + 1;         // the scalar warp takes them from here
                    if (DIAG && p.trace)
                        p.trace[((size_t)c * p.nsteps + hs) * NTRACE + 15] =
                            tstamp() - *(volatile unsigned long long *)&ctl->t_start;
                }
            }
        }
    } else if (wid == NW + 3) {
        // ============== scalar warp: all-reduce of the line-search scalars ==============
        // The four scalars of a step (r.q, q.q, the l1 difference, the error) are final when its
        // pass 2 ends and are needed one pass later, when the NEXT step resolves gamma.  This warp
        // runs their all-reduce in that window, off the consumers' critical path: publish my four
        // words, fetch everybody's (lane = scalar lane % 4, writers lane / 4 + 8 i, SB in flight),
        // add in writer order, combine the lanes with a fixed shuffle tree -> bitwise the same
        // totals in every CTA, in ctl->tot.
        {
            constexpr int SB = 5;
            Waiter hw{p.abort_flag, &ctl->abort, p.wait_limit_ns, 0u, 0ull, p.state + 4, 0};
            volatile int *stopf = &ctl->stop;
            const int ks = lane & 3;
            bool live = true;
            for (int64_t sidx = 0; sidx < p.nsteps && live; ++sidx) {
                while (*(volatile long long *)&ctl->sc_go <= sidx) {
                    if (*stopf || *(volatile int *)&ctl->abort) { live = false; break; }
                    __nanosleep(64);
                }
                if (!live) break;
                __threadfence_block();
                const uint32_t tag = p.tag_base + (uint32_t)sidx + 2u;     // the tag of the step that consumes them
                if (lane < 2) {                                            // two whole sectors
                    const double s0 = *(volatile double *)&ctl->sp[2 * lane], s1 = *(volatile double *)&ctl->sp[2 * lane + 1];
                    ll_st2(p.sLL + (size_t)c * 4 + 2 * lane,
                           ll_pack((uint32_t)__double2loint(s0), tag), ll_pack((uint32_t)__double2hiint(s0), tag),
                           ll_pack((uint32_t)__double2loint(s1), tag), ll_pack((uint32_t)__double2hiint(s1), tag));
                }
                hw.begin(((long long)sidx << 32) | (1LL << 30) | (long long)lane);
                double acc = 0.0;
#pragma unroll 1
                for (int base = lane >> 2; base < G && live; base += 8 * SB) {
                    ulonglong2 v[SB];
                    unsigned miss = 0;
#pragma unroll
                    for (int i = 0; i < SB; ++i) {
                        const int wr = base + 8 * i;
                        if (wr < G) { v[i] = ll_ld(p.sLL + (size_t)wr * 4 + ks); miss |= 1u << i; }
                    }
                    const unsigned have = miss;
#pragma unroll
                    for (int i = 0; i < SB; ++i)
                        if (((miss >> i) & 1u) && ll_ok(v[i], tag)) miss &= ~(1u << i);
#pragma unroll 1
                    while (miss && !(DBG & 1)) {
                        if (*stopf || !hw.again()) { live = false; break; }
#pragma unroll
                        for (int i = 0; i < SB; ++i)
                            if ((miss >> i) & 1u) v[i] = ll_ld(p.sLL + (size_t)(base + 8 * i) * 4 + ks);
#pragma unroll
                        for (int i = 0; i < SB; ++i)
                            if (((miss >> i) & 1u) && ll_ok(v[i], tag)) miss &= ~(1u << i);
                    }
#pragma unroll
                    for (int i = 0; i < SB; ++i)
                        if ((have >> i) & 1u) acc = ks == 3 ? fmax(acc, ll_dbl(v[i])) : acc + ll_dbl(v[i]);
                }
                live = __all_sync(0xffffffffu, live);
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, acc, o);
                    acc = ks == 3 ? fmax(acc, ob) : acc + ob;
                }
                if (lane < 4) ctl->tot[lane] = acc;
                __threadfence_block();
                __syncwarp();
                if (lane == 0) *(volatile long long *)&ctl->sc_done = sidx + 1;
            }
        }
    }
    } else {
        // ============================ consumer warps ===============================
        if (MG) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(CONSUMER_REGS_MG));
        else asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(CONSUMER_REGS));
        for (int i = tid; i < rows_c; i += NTC) {
            const double rv = p.r[row0 + i];
            r_loc[i] = rv;
            rT[i] = (T)rv;
            q_loc[i] = 0.0;
            qT[i] = (T)0;
        }
        for (int i = rows_c + tid; i < p.rows_pad; i += NTC) { rT[i] = (T)0; qT[i] = (T)0; }
        if (TRANS)
            for (int i = tid; i < p.nt_t * p.TJ; i += NTC) delta_s[i] = (T)0;   // columns past ld stay 0
        cbar();

        unsigned long long kc = 0;
        Cursor cur{0, 0u};
        bool have_prev = false;
        int m_prev = 0;
        int64_t step_prev = -1;
        double dprev = 0, xprev = 0;                          // column threads
        int64_t prev_idx = -1;
        long long block_cnt = p.state[2];
        double gamma_last = p.gamma_state[0];
        int stopped = 0, aborted = 0;
        int64_t steps_done = 0;
        const unsigned long long t_start = globaltimer_ns();
        const unsigned long long c_start = tstamp();
        if (DIAG && tid == 0) ctl->t_start = c_start;
        const int cs = p.cs, nrg = p.nrg;
        const double mu = p.mu;
        const uint32_t tag0 = p.tag_base;
        const ulonglong2 *inbox = p.gLL + (size_t)c * G * p.mw;
        Waiter waiter{p.abort_flag, &ctl->abort, p.wait_limit_ns, 0u, 0ull, p.state + 4, 0};
        // multi-GPU: wait until the collector warp has summed `rows` rows of the pending step's
        // A_m D over the ranks (0x7fffffff: all rows and the scalars)
        auto wait_q = [&](int64_t pending_step, int rows) {
            const long long want = ((pending_step + 1) << 32) | (long long)rows;
            while (*(volatile long long *)&ctl->qready < want) {
                if (*(volatile int *)&ctl->abort) break;
            }
            __threadfence_block();
        };
        unsigned long long *trace =
            (DIAG && p.trace != nullptr && tid == 0) ? p.trace + (size_t)c * p.nsteps * NTRACE : nullptr;
        unsigned long long *ttrace =
            (DIAG && p.ttrace != nullptr && tid == 0) ? p.ttrace + (size_t)c * p.nsteps * NTTRACE : nullptr;
        int mc = (int)(p.step0 % p.nblocks);

        // pass-1 mapping: thread = (column group cg0 [+k*NTC], row group rg of nrg)
        int cg0, rg;
        bool p1_active;
        if (CPT == 1) {
            p1_active = tid < nrg * ncg;
            cg0 = tid % ncg;
            rg = tid / ncg;
        } else {
            p1_active = true;
            cg0 = tid;
            rg = 0;
        }
        // pass-2 mapping: warp = rows wid, wid+NW, .. of a tile; lane = column groups lane+32k
        const int dk_n = (ncg + 31) >> 5;
        // stage-2 mapping: thread jl < cs owns column j0+jl of every block
        const int j0 = c * cs;
        const int jcol = j0 + tid;
        const bool colthr = tid < cs && jcol < ld;
        const bool has_col = colthr && jcol < p.w;
        VecT dreg[DK > 0 ? DK : 1];

        for (int64_t step = 0;; ++step) {
            // the iteration after the last step only resolves the pending step
            const bool drain = step == p.nsteps;
            if (drain && !have_prev) break;
            const int m = drain ? 0 : (p.order ? p.order[step] : mc);
            if (++mc == p.nblocks) mc = 0;
            const uint32_t tag = tag0 + (uint32_t)step + 1u;
            if (trace && !drain) trace[step * NTRACE + 0] = tstamp() - c_start;

            // prox operands of my column: issued now, consumed after the gather
            const int64_t idx = (int64_t)m * ld + jcol;
            double xj = 0.0, dj = 0.0, drj = 0.0;
            if (!drain) {
                if (has_col) {
                    dj = p.d[idx];
                    drj = p.drec[idx];
                    if (idx != prev_idx) xj = __ldcg(p.x + idx);
                }

                // ---------------- pass 1: partial (A_m^T r, A_m^T q) over the slab ------
                Acc ar[CPT], aq[CPT];
#pragma unroll
                for (int k = 0; k < CPT; ++k) { OP::zero(ar[k]); OP::zero(aq[k]); }

#pragma unroll 1
                for (int t = 0; t < nt; ++t, ++kc) {
                    mbar_wait(full + cur.slot, cur.phase);
                    if (ttrace && t < 16) ttrace[step * NTTRACE + t] = tstamp();
                    const T *tile = reinterpret_cast<const T *>(ring + (size_t)cur.slot * p.slot_bytes);
                    const int rows_t = min(TR, rows_c - t * TR);
                    const T *rTt = rT + t * TR, *qTt = qT + t * TR;
                    if (WORLD > 1 && have_prev) wait_q(step_prev, TRANS ? rows_c : t * TR + rows_t);
                    if (TRANS) {
                        // P1 threads (adjacent lanes) per block column t*TJ + jl: dot products of the column's BX
                        // entries with r and q, complete for this CTA's rows, published at once (one tagged
                        // word per column)
                        const int P1 = TGEN ? p.P1 : 1;
                        const int part = tid & (P1 - 1), jl = tid / P1;
                        const int j = t * p.TJ + jl;
                        Acc a0, a1;
                        OP::zero(a0);
                        OP::zero(a1);
                        if (j < p.w && !(DBG & 2)) {
                            if (!TGEN) {                          // one thread, one box per column (C2)
                                const T *col = tile + (size_t)tid * p.BX;
#pragma unroll 4
                                for (int iv = 0; iv < p.BXV; ++iv) {
                                    const VecT v = *reinterpret_cast<const VecT *>(col + iv * V);
                                    OP::mac(a0, v, *reinterpret_cast<const VecT *>(rT + iv * V));
                                    OP::mac(a1, v, *reinterpret_cast<const VecT *>(qT + iv * V));
                                }
                            } else {
                                for (int bx = 0; bx < p.NBX; ++bx) {
                                    const T *col = tile + ((size_t)bx * p.TJ + jl) * p.BXb;
                                    const T *rb = rT + bx * p.BXb, *qb = qT + bx * p.BXb;
#pragma unroll 4
                                    for (int iv = part; iv < p.BXVb; iv += P1) {
                                        const VecT v = *reinterpret_cast<const VecT *>(col + iv * V);
                                        OP::mac(a0, v, *reinterpret_cast<const VecT *>(rb + iv * V));
                                        OP::mac(a1, v, *reinterpret_cast<const VecT *>(qb + iv * V));
                                    }
                                }
                            }
                        }
                        T sr = OP::hsum(a0), sq = OP::hsum(a1);
                        if (TGEN) {
#pragma unroll
                            for (int o = 1; o < 8; o <<= 1) {
                                if (o < P1) {
                                    sr += __shfl_xor_sync(0xffffffffu, sr, o);
                                    sq += __shfl_xor_sync(0xffffffffu, sq, o);
                                }
                            }
                        }
                        if (part == 0 && j < G * cs) {
                            const int rd = j >> p.cs_shift;
                            const int jj = j & (cs - 1);
                            LL::put(p.gLL + ((size_t)rd * G + c) * p.mw + jj * WPC, sr, sq, tag);
                        }
                    } else if (p1_active && !(DBG & 2)) {
                        if (TR >= 4) {
                            // whole quads: a row past rows_t meets r = q = 0, but what the slot holds
                            // there is stale (possibly words of an exchange fetch, i.e. NaN bit
                            // patterns), so the last row of the tile is read in its place
                            const int nquad = (rows_t + 3) >> 2;
#pragma unroll 1
                            for (int q4 = rg; q4 < nquad; q4 += nrg) {
                                T rv[4], qv[4];
                                load4(rTt + 4 * q4, rv);
                                load4(qTt + 4 * q4, qv);
                                const T *trow = tile + (size_t)(4 * q4) * ld + cg0 * V;
                                int roff[4];
#pragma unroll
                                for (int i = 0; i < 4; ++i) roff[i] = min(i, rows_t - 1 - 4 * q4) * ld;
#pragma unroll
                                for (int k = 0; k < CPT; ++k) {
                                    if (CPT == 1 || cg0 + k * NTC < ncg) {
                                        VecT v[4];
#pragma unroll
                                        for (int i = 0; i < 4; ++i)
                                            v[i] = *reinterpret_cast<const VecT *>(trow + roff[i] + k * NTC * V);
#pragma unroll
                                        for (int i = 0; i < 4; ++i) {
                                            OP::axpy(ar[k], v[i], rv[i]);
                                            OP::axpy(aq[k], v[i], qv[i]);
                                        }
                                    }
                                }
                            }
                        } else {
#pragma unroll 1
                            for (int rr = rg; rr < rows_t; rr += nrg) {
                                const T rv = rTt[rr], qv = qTt[rr];
                                const T *trow = tile + (size_t)rr * ld + cg0 * V;
#pragma unroll
                                for (int k = 0; k < CPT; ++k) {
                                    if (CPT == 1 || cg0 + k * NTC < ncg) {
                                        const VecT v = *reinterpret_cast<const VecT *>(trow + k * NTC * V);
                                        OP::axpy(ar[k], v, rv);
                                        OP::axpy(aq[k], v, qv);
                                    }
                                }
                            }
                        }
                    }
                    __syncwarp();                   // hand the slot back to the producer
                    if (lane == 0) mbar_arrive(empty + cur.slot);
                    if (ttrace && t < 16) ttrace[step * NTTRACE + 16 + t] = tstamp();
                    cur.advance(S);
                }
                if (trace) trace[step * NTRACE + 1] = tstamp() - c_start;

                // when every thread holds complete column sums (one row group) the partial
                // gradient goes out straight from registers: the V columns of a column group
                // are 4 adjacent words of one reader's message, two 256-bit stores
                if (TRANS) {
                    // published tile by tile above
                } else if (p.direct_pub) {
                    if (p1_active) {
#pragma unroll
                        for (int k = 0; k < CPT; ++k) {
                            const int cg = cg0 + k * NTC;
                            if (CPT == 1 || cg < ncg) {
                                const int j = cg * V;
                                const int rd = j >> p.cs_shift;
                                const int jj = j & (cs - 1);
                                LL::put_group(p.gLL + ((size_t)rd * G + c) * p.mw + jj * WPC, OP::pack(ar[k]),
                                              OP::pack(aq[k]), tag);
                            }
                        }
                    }
                } else if (p1_active) {
                    // combine the row groups of this CTA through shared memory
#pragma unroll
                    for (int k = 0; k < CPT; ++k) {
                        const int cg = cg0 + k * NTC;
                        if (CPT == 1 || cg < ncg) {
                            *reinterpret_cast<VecT *>(redT + (size_t)(rg * 2 + 0) * ld + cg * V) = OP::pack(ar[k]);
                            *reinterpret_cast<VecT *>(redT + (size_t)(rg * 2 + 1) * ld + cg * V) = OP::pack(aq[k]);
                        }
                    }
                }
            }
            if (!p.direct_pub && !drain) cbar();       // the row-group partials in shared memory are complete
            // ---------------- publish: one message of MW words per reader -------------------
            // the partial gradient (g_r, g_q) of the cs columns that reader owns: MW = cs * WPC
            // words, a power of two (C2: 8 words = one 128-byte line per reader).  My four
            // line-search scalars of the pending step go to a small array of their own: every CTA
            // needs all of them, so they are written once instead of once per reader.
            {
                const int MW = p.mw;
                ulonglong2 *out = p.gLL + (size_t)c * MW;            // + reader * G * MW
                if (!p.direct_pub || drain) {
#pragma unroll 1
                    for (int j = tid; j < G * cs; j += NTC) {
                        T sr = (T)0, sq = (T)0;
                        if (j < ld && !drain) {
#pragma unroll 1
                            for (int g2 = 0; g2 < nrg; ++g2) {
                                sr += redT[(size_t)(g2 * 2 + 0) * ld + j];
                                sq += redT[(size_t)(g2 * 2 + 1) * ld + j];
                            }
                        }
                        const int rd = j >> p.cs_shift;
                        const int jj = j & (cs - 1);
                        LL::put(out + (size_t)rd * G * MW + jj * WPC, sr, sq, tag);
                    }
                } else {
                    // columns past ld (readers' padding columns) still have to carry the tag
#pragma unroll 1
                    for (int j = (TRANS ? nt * p.TJ : ncg * V) + tid; j < G * cs; j += NTC) {
                        const int rd = j >> p.cs_shift;
                        const int jj = j & (cs - 1);
                        LL::put(out + (size_t)rd * G * MW + jj * WPC, (T)0, (T)0, tag);
                    }
                }
            }
            if (trace && !drain) trace[step * NTRACE + 2] = tstamp() - c_start;

            // ---------------- gather -------------------------------------------------------
            // Straight from L2 into registers, no landing area and no TMA (the ring and the TMA
            // queue stay free for the tiles of pass 2, which the producer stages meanwhile):
            // thread = (message word k = tid % MW, writers tid / MW + i * NTC / MW), up to NB loads
            // in flight, issued as one batch; a word whose tags do not match yet had not been
            // written when the load read it and is polled by itself.  Each thread adds its words
            // in writer order, the threads of a word are combined by a fixed shuffle tree and a
            // fixed-order sum over the warps: bitwise deterministic.  (The four line-search scalars
            // are not part of this exchange any more: the scalar warp reduces them during pass 1.)
            double g_r = 0.0, g_q = 0.0;
            {
                const int MW = p.mw, wshift = p.mw_shift;
                const int kq = tid & (MW - 1), wstride = NTC >> wshift;
                const ulonglong2 *inb = inbox + kq;                   // + writer * MW
                double a0 = 0.0, a1 = 0.0;
                waiter.spins = 0;
#pragma unroll 1
                for (int base = tid >> wshift; base < G; base += wstride * NB) {
                    ulonglong2 v[NB];
                    unsigned miss = 0;
#pragma unroll
                    for (int i = 0; i < NB; ++i) {
                        const int wr = base + wstride * i;
                        if (wr < G) { v[i] = ll_ld(inb + (size_t)wr * MW); miss |= 1u << i; }
                    }
                    const unsigned have = miss;
#pragma unroll
                    for (int i = 0; i < NB; ++i)
                        if (((miss >> i) & 1u) && ll_ok(v[i], tag)) miss &= ~(1u << i);
                    if (miss && !(DBG & 1)) {
                        waiter.begin(((long long)step << 32) | ((long long)(base * MW + kq) & 0x7fffffff));
#pragma unroll 1
                        do {
#pragma unroll
                            for (int i = 0; i < NB; ++i)
                                if ((miss >> i) & 1u) v[i] = ll_ld(inb + (size_t)(base + wstride * i) * MW);
#pragma unroll
                            for (int i = 0; i < NB; ++i)
                                if (((miss >> i) & 1u) && ll_ok(v[i], tag)) miss &= ~(1u << i);
                        } while (miss && waiter.again());
                    }
#pragma unroll
                    for (int i = 0; i < NB; ++i) {
                        if ((have >> i) & 1u) {
                            if (WPC == 2) {
                                a0 += ll_dbl(v[i]);
                            } else {
                                a0 += (double)__uint_as_float((uint32_t)v[i].x);
                                a1 += (double)__uint_as_float((uint32_t)v[i].y);
                            }
                        }
                    }
                }
                if (trace && !drain) trace[step * NTRACE + 10] = tstamp() - c_start;
                if (trace && !drain) trace[step * NTRACE + 11] = waiter.spins;
                // the threads of one word: lanes k, k + MW, .. of a warp, then the warps
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    if (o >= MW) {
                        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
                        if (WPC == 1) a1 += __shfl_xor_sync(0xffffffffu, a1, o);
                    }
                }
                red[tid] = make_double2(a0, a1);
                cbar();
                if (trace && !drain) trace[step * NTRACE + 12] = tstamp() - c_start;
                // column threads: their column, warps in order
                if (tid < cs) {
                    // (at most NW partials per word: one per warp, or one per NTC / MW threads)
                    const int stepk = MW < 32 ? 32 : MW;
                    double2 v0[NW], v1[NW];
#pragma unroll
                    for (int j = 0; j < NW; ++j) {
                        const int e = min(tid * WPC + stepk * j, NTC - WPC);
                        v0[j] = red[e];
                        v1[j] = red[e + (WPC - 1)];
                    }
#pragma unroll
                    for (int j = 0; j < NW; ++j) {
                        if (tid * WPC + stepk * j < NTC) {
                            g_r += v0[j].x;
                            g_q += WPC == 2 ? v1[j].x : v0[j].y;
                        }
                    }
                }
            }
            if (tid == 0) *(volatile long long *)&ctl->gate = step + 1;   // the producer may re-stream the slab
            if (trace && !drain) trace[step * NTRACE + 3] = trace[step * NTRACE + 4] = tstamp() - c_start;

            // ---------------- resolve the pending step: error, stop rule, gamma ---------
            bool go = true;
            double gamma_prev = 0.0;
            if (have_prev) {
                // the scalars of the pending step, summed over all CTAs by the scalar warp during pass 1
                while (*(volatile long long *)&ctl->sc_done < step) {
                    if (*(volatile int *)&ctl->abort) break;
                }
                __threadfence_block();
                const double rq = *(volatile double *)&ctl->tot[0], qq = *(volatile double *)&ctl->tot[1],
                             l1 = *(volatile double *)&ctl->tot[2], err = *(volatile double *)&ctl->tot[3];
                if (c == 0 && tid == 0 && p.err_hist) p.err_hist[step_prev] = err;
                if (p.bounded) {                                   // lasso.py:141-150
                    if (err < p.err_bound) ++block_cnt;
                    if (m_prev == p.nblocks - 1) {
                        if (block_cnt == p.nblocks) go = false;
                        else block_cnt = 0;
                    }
                }
                if (go && qq != 0.0)                               // lasso.py:133-136
                    gamma_last = fmin(fmax(-(rq + mu * l1) / qq, 0.0), 1.0);
                gamma_prev = gamma_last;
            }
            if (trace && !drain) trace[step * NTRACE + 5] = tstamp() - c_start;

            // ---------------- my column: apply the pending update, prox, publish D ------
            double my_l1 = 0.0, my_err = 0.0, delta = 0.0;
            if (colthr) {
                if (have_prev && go && prev_idx >= 0) {
                    const double xn = xprev + gamma_prev * dprev;                // lasso.py:153
                    __stcg(p.x + prev_idx, xn);
                    if (idx == prev_idx) xj = xn;
                } else if (idx == prev_idx) {
                    xj = xprev;
                }
                prev_idx = -1;
                if (!drain) {
                    if (has_col && dj > 0.0) {
                        const double g = g_r + gamma_prev * g_q;
                        const double u = dj * xj - g;                             // lasso.py:114
                        const double au = fabs(u) - mu;                           // cpu_calculation.py:5-6
                        const double soft = au > 0.0 ? copysign(au, u) : 0.0;
                        const double Bx = drj * soft;                             // lasso.py:117
                        delta = Bx - xj;                                          // lasso.py:119
                        my_l1 = fabs(Bx) - fabs(xj);
                        const double gx = g - xj;                                 // cpu_calculation.py:15-20
                        const double proj = fmin(fmax(gx, -mu), mu);
                        my_err = fabs(g - proj);
                        dprev = delta;
                        xprev = xj;
                        prev_idx = idx;
                    }
                }
            }
            // D goes out in whole 32-byte sectors, one store per sector (the columns of a sector sit in
            // adjacent lanes: the first lane collects the others' words).  Pieces of a sector written
            // by different store instructions become visible MUCH later (measured: packing two columns
            // per word with 8-byte stores cost 1.5 us per step).
            if (!drain && wid * 32 < cs) {
                unsigned long long w0, w1;
                LL::dwords((T)delta, tag, w0, w1);
                if (p.dsec && p.dpw == 2) {                    // four columns per sector
                    const unsigned long long a1 = __shfl_down_sync(0xffffffffu, w0, 1);
                    const unsigned long long a2 = __shfl_down_sync(0xffffffffu, w0, 2);
                    const unsigned long long a3 = __shfl_down_sync(0xffffffffu, w0, 3);
                    if (colthr && (lane & 3) == 0) ll_st2(p.dLL + (jcol >> 1), w0, a1, a2, a3);
                } else if (p.dsec) {                           // two columns per sector
                    const unsigned long long b0 = __shfl_down_sync(0xffffffffu, w0, 1);
                    const unsigned long long b1 = __shfl_down_sync(0xffffffffu, w1, 1);
                    if (colthr && (lane & 1) == 0) ll_st2(p.dLL + jcol, w0, w1, b0, b1);
                } else if (colthr) {
                    ll_st(p.dLL + jcol, w0, w1);
                }
            }
            // A CTA that owns no column publishes an acknowledgement (a sector of its own) instead.
            // Nobody starts pass 2 before every word of this fetch is there, i.e. before EVERY CTA has
            // finished its gather -- which is what allows a writer to overwrite inbox words next step.
            if (!drain && tid == 0 && j0 >= ld) {
                const unsigned long long tw = ll_pack(0u, tag);
                ll_st2(p.dLL + p.ackbase + 2 * (c - p.nown), tw, tw, tw, tw);
            }
            if (trace && !drain) trace[step * NTRACE + 6] = tstamp() - c_start;

            // ---------------- the step D from all slice owners -------------------------
            // every thread loads, checks, polls and decodes its own words (tid + i * NTC), NB in
            // flight: no vote, no barrier until the decoded D is complete
            if (!drain) {
                const int dwords = ld / p.dpw;
                const int dtot = p.ackbase + 2 * (G - p.nown);    // D words + acknowledgements
#pragma unroll 1
                for (int base = tid; base < dtot; base += NTC * NB) {
                    ulonglong2 v[NB];
                    unsigned miss = 0;
#pragma unroll
                    for (int i = 0; i < NB; ++i) {
                        const int e = base + NTC * i;
                        if (e < dtot && (e < dwords || e >= p.ackbase)) { v[i] = ll_ld(p.dLL + e); miss |= 1u << i; }
                    }
                    const unsigned have = miss;
#pragma unroll
                    for (int i = 0; i < NB; ++i)
                        if (((miss >> i) & 1u) && ll_ok(v[i], tag)) miss &= ~(1u << i);
                    if (miss && !(DBG & 1)) {
                        waiter.begin(((long long)step << 32) | (1LL << 31) | (long long)base);
#pragma unroll 1
                        do {
#pragma unroll
                            for (int i = 0; i < NB; ++i)
                                if ((miss >> i) & 1u) v[i] = ll_ld(p.dLL + base + NTC * i);
#pragma unroll
                            for (int i = 0; i < NB; ++i)
                                if (((miss >> i) & 1u) && ll_ok(v[i], tag)) miss &= ~(1u << i);
                        } while (miss && waiter.again());
                    }
#pragma unroll
                    for (int i = 0; i < NB; ++i) {
                        const int e = base + NTC * i;
                        if (((have >> i) & 1u) && e < dwords) LL::dget(v[i], p.dpw, delta_s + e * p.dpw);
                    }
                }
                // the l1 / err terms of my columns (the threads of the first cs / 32 warps), summed per
                // warp here, where the warp would otherwise sit in the barrier; thread 0 adds the warps
                if (wid * 32 < cs) {
                    const double a = warp_sum(my_l1), e = warp_max(my_err);
                    if (lane == 0) { l1s[wid] = a; es[wid] = e; }
                }
            }
            cbar();
            if (tid == 0 && p.gate2_tiles) *(volatile long long *)&ctl->gate2 = step + 1;
            if (trace && !drain) trace[step * NTRACE + 7] = tstamp() - c_start;
            if (*(volatile int *)&ctl->abort) {
                aborted = 1;
                break;
            }
            if (!go) {
                stopped = 1;
                steps_done = step_prev + 1;
                break;
            }
            // r += gamma q of the pending step (lasso.py:155).  Pass 2 does not read r: on one GPU the
            // update rides in the loop after pass 2 that reads and writes the same entries anyway; with
            // peers the collector warp reads r while pass 2 runs, so it is applied here
            if (have_prev && (WORLD > 1 || drain)) {
#pragma unroll 1
                for (int i = tid; i < rows_c; i += NTC) {
                    const double rn = r_loc[i] + gamma_prev * q_loc[i];
                    r_loc[i] = rn;
                    rT[i] = (T)rn;
                }
            }
            if (drain) break;
            if (tid == 0) {
                ctl->sp[2] = cs > 32 ? l1s[0] + l1s[1] : l1s[0];
                ctl->sp[3] = cs > 32 ? fmax(es[0], es[1]) : es[0];
            }
            if (DK > 0) {
#pragma unroll
                for (int k = 0; k < DK; ++k) {
                    const int cg = lane + 32 * k;
                    dreg[k] = cg < ncg ? *reinterpret_cast<const VecT *>(delta_s + cg * V) : vzero(VecT());
                }
            }

            // multi-GPU: a finished row of the partial product goes to the peers at once, so the
            // NVLink latency overlaps the rest of the pass (see the exchange below)
            const size_t cell = (((size_t)(tag & 1u) * G + c) * WORLD) * p.qw;
            auto send_row = [&](int idx, double v) {
                if (WORLD > 1) {
                    if (p.mc) {
                        mm_st_dbl(p.mc + cell + (size_t)p.rank * p.qw + idx, v, tag);
                    } else {
#pragma unroll 1
                        for (int pr = 0; pr < WORLD; ++pr)
                            if (pr != p.rank) ll_st_dbl(p.peer[pr] + cell + (size_t)p.rank * p.qw + idx, v, tag);
                    }
                }
            };
            if (WORLD > 1 && tid == 0) {   // my l1 / err terms of this step travel with the rows
                if (!p.tile_sends) {       // (otherwise the sender warp sends them)
                    send_row(rows_c, ctl->sp[2]);
                    send_row(rows_c + 1, ctl->sp[3]);
                }
                __threadfence_block();
                *(volatile long long *)&ctl->p2start = step + 1;
            }

            // ---------------- pass 2: q = A_m D over the slab ---------------------------
            Acc accT;                      // TRANS: this thread's residual entries, all columns
            OP::zero(accT);
            const int ivT = TRANS ? tid % p.BXV : 0, partT = TRANS ? tid / p.BXV : 0;
            // (my group inside its box: box ivT / BXVb, all TJ columns of a box are adjacent in the slot)
            const size_t offT = TGEN ? (size_t)(ivT / p.BXVb) * p.TJ * p.BXb + (size_t)(ivT % p.BXVb) * V : (size_t)ivT * V;
            const int strideT = TGEN ? p.BXb : p.BX;
            {
                // Rows of the tile against D.  Narrow blocks (D in registers): all loads of a row pair
                // go out as one batch (NK per row: the smallest of 2 / 4 / 8 that covers the block; a
                // lane past the last column group reads the last one against a zero D) and only then
                // the multiply-adds -- a load / use / load chain leaves the two warps of a scheduler
                // waiting for shared memory most of the time.
                auto pair_dot = [&](auto nk_tag, const T *rowa, const T *rowb, T &qa, T &qb) {
                    constexpr int NK = decltype(nk_tag)::value;
                    VecT va[NK], vb[NK];
#pragma unroll
                    for (int k = 0; k < NK; ++k) {
                        const int cg = min(lane + 32 * k, ncg - 1);
                        va[k] = *reinterpret_cast<const VecT *>(rowa + cg * V);
                        vb[k] = *reinterpret_cast<const VecT *>(rowb + cg * V);
                    }
                    Acc a0, a1, b0, b1;
                    OP::zero(a0); OP::zero(a1); OP::zero(b0); OP::zero(b1);
#pragma unroll
                    for (int k = 0; k < NK; ++k) {
                        const VecT d = dreg[k < (DK > 0 ? DK : 1) ? k : 0];
                        if (k & 1) { OP::mac(a1, va[k], d); OP::mac(b1, vb[k], d); }
                        else       { OP::mac(a0, va[k], d); OP::mac(b0, vb[k], d); }
                    }
                    qa = OP::hsum(a0) + OP::hsum(a1);
                    qb = OP::hsum(b0) + OP::hsum(b1);
                };
                auto row_pair = [&](const T *rowa, const T *rowb, T &qa, T &qb) {
                    if (DK > 0) {
                        if (dk_n > 4) pair_dot(std::integral_constant<int, 8>(), rowa, rowb, qa, qb);
                        else if (dk_n > 2) pair_dot(std::integral_constant<int, 4>(), rowa, rowb, qa, qb);
                        else pair_dot(std::integral_constant<int, 2>(), rowa, rowb, qa, qb);
                    } else {
                        // wide blocks: D from shared memory, two rows share every D load
                        Acc a0, b0;
                        OP::zero(a0); OP::zero(b0);
#pragma unroll 2
                        for (int cg = lane; cg < ncg; cg += 32) {
                            const VecT d0 = *reinterpret_cast<const VecT *>(delta_s + cg * V);
                            OP::mac(a0, *reinterpret_cast<const VecT *>(rowa + cg * V), d0);
                            OP::mac(b0, *reinterpret_cast<const VecT *>(rowb + cg * V), d0);
                        }
                        qa = OP::hsum(a0);
                        qb = OP::hsum(b0);
                    }
                };
                // a finished pair: sum over the lanes (a in lanes 0..15, b in 16..31), store, send
                auto flush_pair = [&](int row_a, bool two, T qa, T qb) {
                    const T qs = warp_sum_pair(qa, qb, lane);
                    if (row_a >= 0 && (lane & 15) == 0 && (two || lane == 0)) {
                        const int row = row_a + (lane >> 4) * NW;
                        qpart[row] = (double)qs;
                        if (!p.tile_sends) send_row(row, (double)qs);
                    }
                };
                if (trace) trace[step * NTRACE + 14] = tstamp() - c_start;
                // multi-GPU: the sender warp sends a tile's rows to the peers when all NW warps have
                // counted it
                auto count_tile = [&](int tile_idx) {
                    if (WORLD > 1 && p.tile_sends) {
                        __syncwarp();
                        if (lane == 0) {
                            __threadfence_block();
                            atomicAdd(tilecnt + (tile_idx & 127), 1);
                        }
                    }
                };
                T pqa = (T)0, pqb = (T)0;
                int pend_row = -1;
                bool pend_two = false;
#pragma unroll 1
                for (int t2 = 0; t2 < nt; ++t2) {
                    const int t = t2;
                    mbar_wait(full + cur.slot, cur.phase);
                    const int slot = cur.slot;
                    cur.advance(S);
                    ++kc;
                    if (ttrace && t2 < 16) ttrace[step * NTTRACE + 32 + t2] = tstamp();
                    const T *tile = reinterpret_cast<const T *>(ring + (size_t)slot * p.slot_bytes);
                    const int rows_t = min(TR, rows_c - t * TR);
                    if (TRANS) {
                        // thread = (16-byte group ivT of my residual entries, column part partT)
                        const int cols_t = min(p.TJ, p.w - t * p.TJ);
                        if (partT < p.nparts && !(DBG & 4)) {
#pragma unroll 4
                            for (int j = partT; j < cols_t; j += p.nparts) {
                                const VecT v = *reinterpret_cast<const VecT *>(tile + offT + (size_t)j * strideT);
                                OP::axpy(accT, v, delta_s[t * p.TJ + j]);
                            }
                        }
                    } else if (!(DBG & 4)) {
                        // two rows per trip (the odd last row is paired with itself).  The shuffle tree
                        // of a pair is a chain of dependent instructions: it runs one trip late, in
                        // front of the loads of the next pair (multi-GPU: at once, the sender warp waits
                        // for the rows; deferring there was measured slower)
#pragma unroll 1
                        for (int rr = wid; rr < rows_t; rr += 2 * NW) {
                            const bool two = rr + NW < rows_t;
                            T qa, qb;
                            if (WORLD == 1) {
                                // (unconditional, only the store is predicated: one basic block, so that
                                // the loads below are scheduled over the shuffle chain)
                                flush_pair(pend_row, pend_two, pqa, pqb);
                                row_pair(tile + (size_t)rr * ld, tile + (size_t)(two ? rr + NW : rr) * ld, qa, qb);
                                pqa = qa; pqb = qb; pend_row = t * TR + rr; pend_two = two;
                            } else {
                                row_pair(tile + (size_t)rr * ld, tile + (size_t)(two ? rr + NW : rr) * ld, qa, qb);
                                flush_pair(t * TR + rr, two, qa, qb);
                            }
                        }
                        count_tile(t2);
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(empty + slot);
                    if (ttrace && t2 < 16) ttrace[step * NTTRACE + 48 + t2] = tstamp();
                }
                if (!TRANS) flush_pair(pend_row, pend_two, pqa, pqb);
            }
            if (TRANS) {
                // combine the column parts through shared memory
                T *red2 = reinterpret_cast<T *>(smem + p.off_red2);
                if (partT < p.nparts) *reinterpret_cast<VecT *>(red2 + (size_t)partT * p.BX + ivT * V) = OP::pack(accT);
                cbar();
#pragma unroll 1
                for (int i = tid; i < rows_c; i += NTC) {
                    T sum = (T)0;
#pragma unroll 1
                    for (int pt = 0; pt < p.nparts; ++pt) sum += red2[(size_t)pt * p.BX + i];
                    qpart[i] = (double)sum;
                    send_row(i, (double)sum);
                }
            } else {
                cbar();
            }
            if (trace) trace[step * NTRACE + 8] = tstamp() - c_start;
            if (WORLD > 1) {
                // multi-GPU: my partial rows are complete (and sent); the collector warp sums them
                // with the peers' rows and computes the line-search partials while the next step's
                // pass 1 is already running (see the collector warp above)
                if (tid == 0) {
                    __threadfence_block();
                    *(volatile long long *)&ctl->p2done = step + 1;
                }
            } else
            {
                double trq = 0.0, tqq = 0.0;
                const double gp = have_prev ? gamma_prev : 0.0;
#pragma unroll 1
                for (int i = tid; i < rows_c; i += NTC) {
                    const double rn = r_loc[i] + gp * q_loc[i];              // lasso.py:155 (pending step)
                    const double q = qpart[i];
                    r_loc[i] = rn;
                    rT[i] = (T)rn;
                    q_loc[i] = q;
                    qT[i] = (T)q;
                    trq += rn * q;                                           // lasso.py:129
                    tqq += q * q;                                            // lasso.py:132
                }
                trq = warp_sum(trq);
                tqq = warp_sum(tqq);
                if (lane == 0) { lsred[wid] = trq; lsred[NW + wid] = tqq; }
                cbar();
                if (wid == 0) {
                    const double a = warp_sum(lane < NW ? lsred[lane] : 0.0);
                    const double b = warp_sum(lane < NW ? lsred[NW + lane] : 0.0);
                    if (lane == 0) {
                        ctl->sp[0] = a;
                        ctl->sp[1] = b;
                        __threadfence_block();
                        *(volatile long long *)&ctl->sc_go = step + 1;   // the scalar warp takes them from here
                    }
                }
            }
            have_prev = true;
            m_prev = m;
            step_prev = step;
            steps_done = step + 1;
            if (c == 0 && tid == 0 && p.time_hist) p.time_hist[step] = globaltimer_ns() - t_start;
            if (trace) trace[step * NTRACE + 9] = tstamp() - c_start;
        }

        if (trace && p.nsteps >= 2) {      // cycles -> time: a (globaltimer, cycle) pair at both ends of the launch
            trace[13] = t_start;
            trace[(p.nsteps - 1) * NTRACE + 13] = globaltimer_ns();
            trace[(p.nsteps - 1) * NTRACE + 11] = tstamp() - c_start;
        }
        if (WORLD > 1) {
            // the collector warp finishes the step it is working on (its waits are bounded) before
            // it is shown the stop flag
            if (have_prev) {
                const long long want = ((step_prev + 1) << 32) | 0x7fffffffLL;
                while (*(volatile long long *)&ctl->qready < want) __nanosleep(32);
            }
            if (tid == 0) *(volatile int *)&ctl->hstop = 1;
        }
        cbar();
        for (int i = tid; i < rows_c; i += NTC) p.r[row0 + i] = r_loc[i];
        if (c == 0 && tid == 0) {
            p.state[0] = steps_done;
            p.state[1] = stopped;
            p.state[2] = block_cnt;
            p.state[3] = aborted;
            p.gamma_state[0] = gamma_last;
        }
        if (tid == 0) {
            ctl->kc = kc;
            *(volatile int *)&ctl->stop = 1;
        }
    }
    __syncthreads();
    // drain TMA copies the producer issued past the stop point
    if (tid == 0) {
        unsigned long long k = ctl->kc;
        Cursor cur{(int)(k % (unsigned)S), (uint32_t)((k / (unsigned)S) & 1ULL)};
        for (; k < ctl->k_issued; ++k) {
            mbar_wait(full + cur.slot, cur.phase);
            cur.advance(S);
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------
// plain (non-persistent) kernels: weighted column sums, row dots, reductions
// ------------------------------------------------------------------------------------
// part[y][chunk][col] = sum_{rows in chunk} A_y[row][col] * (SQ ? A_y[row][col] : vec[row]); blockIdx.y
// selects one of several equally shaped matrices (the column blocks: diag(A^T A) of all blocks is
// ONE launch).  Thread = 16-byte column group, eight rows in flight per thread.
template <typename T, bool SQ>
__global__ void __launch_bounds__(256) colwsum_partial(const T *__restrict__ A, int64_t M, int ncols,
                                                       int64_t ld, const double *__restrict__ vec,
                                                       double *__restrict__ part, int rows_per_chunk,
                                                       int64_t mat_stride) {
    using VecT = typename VT<T>::type;
    constexpr int V = VT<T>::V;
    constexpr int U = 8;
    const int chunk = blockIdx.x;
    A += (int64_t)blockIdx.y * mat_stride;
    part += (int64_t)blockIdx.y * gridDim.x * ncols;
    const int64_t r0 = (int64_t)chunk * rows_per_chunk;
    const int64_t r1 = min(M, r0 + rows_per_chunk);
    const int ncg = ncols / V;  // ncols is a multiple of V (padded)
    for (int cg = threadIdx.x; cg < ncg; cg += blockDim.x) {
        double acc[V];
#pragma unroll
        for (int e = 0; e < V; ++e) acc[e] = 0.0;
        const T *col = A + (int64_t)cg * V;
        int64_t r = r0;
        for (; r + U <= r1; r += U) {
            VecT v[U];
            double s[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                v[u] = __ldg(reinterpret_cast<const VecT *>(col + (r + u) * ld));
                s[u] = SQ ? 0.0 : __ldg(vec + r + u);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const T *ve = reinterpret_cast<const T *>(&v[u]);
#pragma unroll
                for (int e = 0; e < V; ++e) acc[e] += (double)ve[e] * (SQ ? (double)ve[e] : s[u]);
            }
        }
        for (; r < r1; ++r) {
            const VecT v = __ldg(reinterpret_cast<const VecT *>(col + r * ld));
            const T *ve = reinterpret_cast<const T *>(&v);
            const double sc = SQ ? 0.0 : __ldg(vec + r);
#pragma unroll
            for (int e = 0; e < V; ++e) acc[e] += (double)ve[e] * (SQ ? (double)ve[e] : sc);
        }
#pragma unroll
        for (int e = 0; e < V; ++e) part[(int64_t)chunk * ncols + cg * V + e] = acc[e];
    }
}

// out[y * out_stride + col] (+)= sum_chunk part[y][chunk][col] for col < ncols_out, fixed order
// (deterministic): 8 columns x 32 chunk groups per CTA -- many small CTAs, the partials are a few MB --
// each thread adds every 32nd chunk, then the 32 groups of a column are added in order
__global__ void __launch_bounds__(256) reduce_partials(const double *__restrict__ part, int nchunks, int ncols,
                                                       double *__restrict__ out, int accumulate, int64_t out_stride,
                                                       int ncols_out) {
    __shared__ double sm[32][9];
    const int cx = threadIdx.x & 7, gy = threadIdx.x >> 3;
    const int col = blockIdx.x * 8 + cx;
    part += (int64_t)blockIdx.y * nchunks * ncols;
    double s = 0.0;
    if (col < ncols_out) {
#pragma unroll 4
        for (int ch = gy; ch < nchunks; ch += 32) s += part[(int64_t)ch * ncols + col];
    }
    sm[gy][cx] = s;
    __syncthreads();
    if (gy == 0 && col < ncols_out) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 32; ++k) t += sm[k][cx];
        double *o = out + (int64_t)blockIdx.y * out_stride + col;
        *o = accumulate ? *o + t : t;
    }
}

// out[col] (+)= sum_row A[row][col] * vec[row] for ONE matrix in ONE launch (the step-wise A_m^T r of the
// row-major layout, A_m d of the pre-transposed one).  Grid = (RC row chunks) x (column slabs of 256 16-byte
// groups), launched cooperatively when RC > 1 so that all CTAs are co-resident.  A CTA is 4 row sub-groups x 256
// column groups, eight rows in flight per thread; its partial sums go out as self-validating 16-byte words
// (value, launch number) -- the exchange of the fused kernel, no fence, no flag, no second launch -- and the RC
// CTAs of a slab each add up a share of the slab's columns: warp per column, lane = chunk, fixed order,
// fixed shuffle tree (deterministic).
constexpr int CW_THREADS = 1024;
constexpr int CW_CG = 256;
constexpr int CW_SUB = CW_THREADS / CW_CG;
constexpr int CW_MAXP = 8;         // chunks per lane in the gather: RC <= 32 * CW_MAXP

// partial sums of a chunk -> exchange words -> my share of the slab's columns (colwsum_fused, matvec_stream)
template <int SL>
__device__ __forceinline__ void cw_exchange(double mine, int c_l, int nthreads, int RC, int i, int j,
                                            ulonglong2 *words, unsigned long long seq, double *out, int accumulate,
                                            int ncols_out) {
    if (RC == 1) {
        const int colg = j * SL + c_l;
        if (c_l < SL && colg < ncols_out) out[colg] = accumulate ? out[colg] + mine : mine;
        return;
    }
    if (c_l < SL) ll_st(words + (size_t)(j * RC + i) * SL + c_l, (unsigned long long)__double_as_longlong(mine), seq);
    const int c_lo = (int)((int64_t)SL * i / RC), c_hi = (int)((int64_t)SL * (i + 1) / RC);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned long long t_start = globaltimer_ns();
    for (int cc = c_lo + warp; cc < c_hi; cc += nthreads / 32) {
        const int colg = j * SL + cc;
        if (colg >= ncols_out) break;
        const ulonglong2 *src = words + (size_t)j * RC * SL + cc;
        ulonglong2 w[CW_MAXP];
#pragma unroll
        for (int k = 0; k < CW_MAXP; ++k)
            if (lane + 32 * k < RC) w[k] = ll_ld(src + (size_t)(lane + 32 * k) * SL);
        double sum = 0.0;
#pragma unroll
        for (int k = 0; k < CW_MAXP; ++k) {
            if (lane + 32 * k < RC) {
                unsigned spin = 0;
                while (w[k].y != seq) {
                    if ((++spin & 1023u) == 0u && globaltimer_ns() - t_start > 4000000000ULL) __trap();
                    w[k] = ll_ld(src + (size_t)(lane + 32 * k) * SL);
                }
                sum += __longlong_as_double((long long)w[k].x);
            }
        }
        sum = warp_sum(sum);
        if (lane == 0) out[colg] = accumulate ? out[colg] + sum : sum;
    }
}

template <typename T>
__global__ void __launch_bounds__(CW_THREADS, 1) colwsum_fused(const T *__restrict__ A, int64_t M, int ncols,
                                                               int64_t ld, const double *__restrict__ vec,
                                                               ulonglong2 *words, unsigned long long seq,
                                                               double *out, int accumulate, int ncols_out) {
    using VecT = typename VT<T>::type;
    constexpr int V = VT<T>::V;
    constexpr int U = 8;
    constexpr int SL = CW_CG * V;                 // columns of a slab
    __shared__ double red[CW_SUB][V][CW_CG];
    const int RC = gridDim.x, i = blockIdx.x, j = blockIdx.y;
    const int tid = threadIdx.x, cgl = tid & (CW_CG - 1), sub = tid / CW_CG;
    const int ncg = ncols / V;                    // ncols is a multiple of V (padded)
    const int cg = j * CW_CG + cgl;
    const int64_t r0 = M * i / RC, r1 = M * (i + 1) / RC;
    double acc[V];
#pragma unroll
    for (int e = 0; e < V; ++e) acc[e] = 0.0;
    if (cg < ncg) {
        const T *col = A + (int64_t)cg * V;
        int64_t r = r0 + sub;                     // the sub-groups take adjacent rows (one DRAM page)
        for (; r + (U - 1) * CW_SUB < r1; r += U * CW_SUB) {
            VecT v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = __ldg(reinterpret_cast<const VecT *>(col + (r + u * CW_SUB) * ld));
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const double sc = __ldg(vec + r + u * CW_SUB);
                const T *ve = reinterpret_cast<const T *>(&v[u]);
#pragma unroll
                for (int e = 0; e < V; ++e) acc[e] += (double)ve[e] * sc;
            }
        }
        for (; r < r1; r += CW_SUB) {
            const VecT v = __ldg(reinterpret_cast<const VecT *>(col + r * ld));
            const double sc = __ldg(vec + r);
            const T *ve = reinterpret_cast<const T *>(&v);
#pragma unroll
            for (int e = 0; e < V; ++e) acc[e] += (double)ve[e] * sc;
        }
    }
#pragma unroll
    for (int e = 0; e < V; ++e) red[sub][e][cgl] = acc[e];
    __syncthreads();
    // the CTA's partial of column c_l of the slab: sub-groups added in order
    double mine = 0.0;
    const int c_l = tid;
    if (c_l < SL) {
        const int g = c_l / V, e = c_l % V;
        mine = ((red[0][e][g] + red[1][e][g]) + red[2][e][g]) + red[3][e][g];
    }
    cw_exchange<SL>(mine, c_l, CW_THREADS, RC, i, j, words, seq, out, accumulate, ncols_out);
}

// ------------------------------------------------------------------------------------
// TMA-streamed row dots of ONE matrix (the step-wise path on blocks that fill the machine)
// ------------------------------------------------------------------------------------
// out[row] (+)= A[row][:] . vec, one CTA per SM: a producer warp streams the CTA's rows -- tiles of TR rows x one
// column slab, one bulk copy per tile when the slab is the whole row, else one per row -- through a ring of S
// shared-memory slots (mbarrier full/empty pairs); 8 consumer warps work from shared memory.  The bytes in
// flight (the whole ring, 150-220 KB per SM) no longer depend on registers, which the load-batch kernel below
// cannot offer: measured on C2 blocks 11.0 us per 40 MB block against 14.2 us.  (Column sums stay with
// colwsum_fused: their cross-CTA exchange, not the stream, is what is left of their time; a streamed variant
// measured 13.6 us against 12.3 us.)
//   short rows: the warp that owns a row (rows round-robin over the warps) walks its slabs and keeps its sum;
//               VREG: the row is one batch of the warp and its part of vec stays in registers, else vec sits
//               in shared memory, split in two arrays so that 16-byte reads are conflict-free;
//   long rows (one row per tile, `coop`): every warp takes an eighth of each tile, the warps' sums of a row are
//               added in order through shared memory.
constexpr int MS_NW = 8;
constexpr int MS_NTC = MS_NW * 32;
constexpr int MS_THREADS = MS_NTC + 32;
constexpr int MS_MAXS = 16;

struct MsParams {
    const void *A;
    int64_t M, ld;
    int ncols;                     // multiple of V
    const double *vec;
    double *out;
    int accumulate;
    int RC, ncs, SG;               // row chunks (= grid), column slabs, 16-byte groups per slab
    int TR, S, slot_bytes, contig, coop;
    int off_vec, off_part, off_ring;   // shared memory: barriers at 0, vec, the warps' sums of a shared row, ring
};

__device__ __forceinline__ void mbar_wait_bounded(uint64_t *bar, uint32_t parity) {
    unsigned spin = 0;
    unsigned long long t0 = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spin & 255u) == 0u) {            // (a lost copy must not hang the GPU)
            const unsigned long long now = globaltimer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 2000000000ULL) __trap();
        }
    }
}
__device__ __forceinline__ void ms_cbar() { asm volatile("bar.sync 2, %0;" ::"n"(MS_NTC) : "memory"); }

template <typename T, bool VREG>
__global__ void __launch_bounds__(MS_THREADS, 1) rowdot_stream(const MsParams p) {
    using VecT = typename VT<T>::type;
    constexpr int V = VT<T>::V;
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem);
    uint64_t *empty = full + MS_MAXS;
    unsigned char *ring = smem + p.off_ring;
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    const int i = blockIdx.x;
    const int ncg = p.ncols / V;
    const int64_t r0 = p.M * i / p.RC, r1 = p.M * (i + 1) / p.RC;
    const int nrg = (int)((r1 - r0 + p.TR - 1) / p.TR);          // row groups of this CTA
    const T *A = reinterpret_cast<const T *>(p.A);
    if (tid == 0) {
        for (int s = 0; s < p.S; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, MS_NW); }
        fence_mbar_init();
    }
    __syncthreads();
    if (wid == MS_NW) {
        // ---- producer warp
        int slot = 0;
        uint32_t ph = 1;
        for (int g = 0; g < nrg; ++g) {
            const int64_t rk0 = r0 + (int64_t)g * p.TR;
            const int nrows = (int)min((int64_t)p.TR, r1 - rk0);
            for (int j = 0; j < p.ncs; ++j) {
                const int sg = min(p.SG, ncg - j * p.SG);         // groups of this slab
                const uint32_t sb = (uint32_t)sg * 16u;
                mbar_wait_bounded(empty + slot, ph);
                unsigned char *dst = ring + (size_t)slot * p.slot_bytes;
                const T *src = A + rk0 * p.ld + (int64_t)j * p.SG * V;
                if (p.contig) {
                    if (lane == 0) {
                        mbar_expect_tx(full + slot, sb * (uint32_t)nrows);
                        tma_bulk_g2s(dst, src, sb * (uint32_t)nrows, full + slot);
                    }
                } else {
                    if (lane == 0) mbar_expect_tx(full + slot, sb * (uint32_t)nrows);
                    __syncwarp();
                    if (lane < nrows) tma_bulk_g2s(dst + (size_t)lane * sb, src + (int64_t)lane * p.ld, sb, full + slot);
                }
                if (++slot == p.S) { slot = 0; ph ^= 1u; }
            }
        }
        return;
    }
    // ---- consumers
    int slot = 0;
    uint32_t ph = 0;
    double vr[VREG ? 8 * V : 1];
    double2 *vlo = reinterpret_cast<double2 *>(smem + p.off_vec), *vhi = vlo + ncg;
    if (VREG) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int cg = lane + 32 * u;
#pragma unroll
            for (int e = 0; e < V; ++e) vr[u * V + e] = cg < ncg ? __ldg(p.vec + (int64_t)cg * V + e) : 0.0;
        }
    } else {
        for (int cg = tid; cg < ncg; cg += MS_NTC) {
            vlo[cg] = make_double2(__ldg(p.vec + (int64_t)cg * V), __ldg(p.vec + (int64_t)cg * V + 1));
            if (V == 4) vhi[cg] = make_double2(__ldg(p.vec + (int64_t)cg * V + 2), __ldg(p.vec + (int64_t)cg * V + 3));
        }
        ms_cbar();
    }
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    // one 16-byte group of the row against its part of vec in shared memory
    auto fma_group = [&](const unsigned char *gp, int cg) {
        const VecT v = *reinterpret_cast<const VecT *>(gp);
        const T *ve = reinterpret_cast<const T *>(&v);
        const double2 lo = vlo[cg];
        acc[0] += (double)ve[0] * lo.x;
        acc[1] += (double)ve[1] * lo.y;
        if (V == 4) {
            const double2 hi = vhi[cg];
            acc[2] += (double)ve[V == 4 ? 2 : 0] * hi.x;
            acc[3] += (double)ve[V == 4 ? 3 : 0] * hi.y;
        }
    };
    if (!VREG && p.coop) {
        double *part = reinterpret_cast<double *>(smem + p.off_part);     // [2][MS_NW], one barrier per row
        for (int g = 0; g < nrg; ++g) {
            for (int j = 0; j < p.ncs; ++j) {
                const int sg = min(p.SG, ncg - j * p.SG);
                mbar_wait_bounded(full + slot, ph);
                const unsigned char *row = ring + (size_t)slot * p.slot_bytes;
#pragma unroll 4
                for (int c = tid; c < sg; c += MS_NTC) fma_group(row + (size_t)c * 16, j * p.SG + c);
                __syncwarp();
                if (lane == 0) mbar_arrive(empty + slot);
                if (++slot == p.S) { slot = 0; ph ^= 1u; }
            }
            const double total = warp_sum((acc[0] + acc[1]) + (acc[2] + acc[3]));
            acc[0] = acc[1] = acc[2] = acc[3] = 0.0;
            if (lane == 0) part[(g & 1) * MS_NW + wid] = total;
            ms_cbar();
            if (tid == 0) {
                double t = 0.0;
#pragma unroll
                for (int k = 0; k < MS_NW; ++k) t += part[(g & 1) * MS_NW + k];
                double *o = p.out + r0 + g;
                *o = p.accumulate ? *o + t : t;
            }
        }
        return;
    }
    for (int g = 0; g < nrg; ++g) {
        const int64_t rk0 = r0 + (int64_t)g * p.TR;
        const int nrows = (int)min((int64_t)p.TR, r1 - rk0);
        // my row of this group (TR <= MS_NW: at most one)
        const int l = (wid - (int)(((int64_t)g * p.TR) % MS_NW) + MS_NW) % MS_NW;
        const bool mine = l < nrows;
        for (int j = 0; j < p.ncs; ++j) {
            const int sg = min(p.SG, ncg - j * p.SG);
            mbar_wait_bounded(full + slot, ph);
            if (mine) {
                const unsigned char *row = ring + (size_t)slot * p.slot_bytes + (size_t)l * sg * 16;
                if (VREG) {
                    VecT v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u)
                        if (lane + 32 * u < sg) v[u] = *reinterpret_cast<const VecT *>(row + (size_t)(lane + 32 * u) * 16);
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (lane + 32 * u < sg) {
                            const T *ve = reinterpret_cast<const T *>(&v[u]);
#pragma unroll
                            for (int e = 0; e < V; ++e) acc[u & 3] += (double)ve[e] * vr[VREG ? u * V + e : 0];
                        }
                    }
                } else {
#pragma unroll 4
                    for (int c = lane; c < sg; c += 32) fma_group(row + (size_t)c * 16, j * p.SG + c);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty + slot);
            if (++slot == p.S) { slot = 0; ph ^= 1u; }
        }
        if (mine) {
            const double total = warp_sum((acc[0] + acc[1]) + (acc[2] + acc[3]));
            if (lane == 0) {
                double *o = p.out + rk0 + l;
                *o = p.accumulate ? *o + total : total;
            }
            acc[0] = acc[1] = acc[2] = acc[3] = 0.0;
        }
    }
}

// out[row] (+)= sum_col A[row][col] * (SQ ? A[row][col] : vec[col]).  WPR warps of a CTA share a row (each a
// contiguous range of 16-byte column groups; their sums are added in order through shared memory), eight
// 16-byte loads in flight per lane; at any time the grid works on a contiguous window of rows.  VREG: a warp's
// range is one batch (a C2 row on one warp), its part of vec stays in registers for all its rows.  Rows are
// written to out[(row / group) * out_stride + row % group] (group = rows per column block when the rows
// of all blocks are processed in one launch).
template <typename T, bool SQ, bool VREG>
__global__ void __launch_bounds__(256, 2) rowdot_kernel(const T *__restrict__ A, int64_t M, int ncols,
                                                        int64_t ld, const double *__restrict__ vec,
                                                        double *__restrict__ out, int accumulate, int64_t group,
                                                        int64_t out_stride, int wpr) {
    using VecT = typename VT<T>::type;
    constexpr int V = VT<T>::V;
    constexpr int U = 8;
    __shared__ double sm[2][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncg = ncols / V;
    const int rpc = 8 / wpr;                       // rows of a CTA per trip
    const int seg = warp % wpr, rslot = warp / wpr;
    const int gper = (ncg + wpr - 1) / wpr;
    const int g0 = seg * gper, g1 = min(ncg, g0 + gper);
    double vr[VREG && !SQ ? U * V : 1];
    if (VREG && !SQ) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int cg = g0 + lane + 32 * u;
#pragma unroll
            for (int e = 0; e < V; ++e) vr[u * V + e] = cg < g1 ? __ldg(vec + (int64_t)cg * V + e) : 0.0;
        }
    }
    const int64_t stride = (int64_t)gridDim.x * rpc;
    const int64_t ntrips = (M + stride - 1) / stride;
    for (int64_t trip = 0; trip < ntrips; ++trip) {
        const int64_t rbase = trip * stride + (int64_t)blockIdx.x * rpc;
        const int64_t r = rbase + rslot;
        double total = 0.0;
        if (r < M) {
            const T *row = A + r * ld;
            double acc[4] = {0.0, 0.0, 0.0, 0.0};
            for (int c0 = g0 + lane; c0 < g1; c0 += 32 * U) {
                VecT v[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int cg = c0 + 32 * u;
                    if (cg < g1) v[u] = __ldg(reinterpret_cast<const VecT *>(row + (int64_t)cg * V));
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int cg = c0 + 32 * u;
                    if (cg < g1) {
                        const T *ve = reinterpret_cast<const T *>(&v[u]);
#pragma unroll
                        for (int e = 0; e < V; ++e) {
                            const double m = SQ ? (double)ve[e]
                                                : (VREG ? vr[(VREG && !SQ ? u * V + e : 0)] : __ldg(vec + (int64_t)cg * V + e));
                            acc[u & 3] += (double)ve[e] * m;
                        }
                    }
                }
                if (VREG) break;
            }
            total = warp_sum((acc[0] + acc[1]) + (acc[2] + acc[3]));
        }
        if (wpr == 1) {
            if (r < M && lane == 0) {
                double *o = out + (r / group) * out_stride + r % group;
                *o = accumulate ? *o + total : total;
            }
        } else {
            if (lane == 0) sm[trip & 1][warp] = total;
            __syncthreads();
            const int64_t rr = rbase + threadIdx.x;
            if ((int)threadIdx.x < rpc && rr < M) {
                double t = 0.0;
                for (int k = 0; k < wpr; ++k) t += sm[trip & 1][threadIdx.x * wpr + k];
                double *o = out + (rr / group) * out_stride + rr % group;
                *o = accumulate ? *o + t : t;
            }
        }
    }
}

__global__ void finish_diag(const double *__restrict__ dsum, double *__restrict__ d,
                            double *__restrict__ drec, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = dsum[i];
    d[i] = v;
    drec[i] = v > 0.0 ? 1.0 / v : 0.0;   // lasso.py:29-30
}

__global__ void neg_copy(const double *__restrict__ b, double *__restrict__ r, int64_t n, double sign) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) r[i] = sign * b[i];
}

// single-CTA deterministic objective: 0.5*|r|^2 + mu*|x|_1
__global__ void __launch_bounds__(1024) objective_kernel(const double *__restrict__ r, int64_t n,
                                                         const double *__restrict__ x, int64_t nx,
                                                         double mu, double *out) {
    __shared__ double s1[32], s2[32];
    double a = 0.0, b = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) a += r[i] * r[i];
    for (int64_t i = threadIdx.x; i < nx; i += blockDim.x) b += fabs(x[i]);
    a = warp_sum(a);
    b = warp_sum(b);
    if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a; s2[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double A2 = 0.0, B2 = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { A2 += s1[i]; B2 += s2[i]; }
        out[0] = 0.5 * A2 + mu * B2;
        out[1] = A2;
        out[2] = B2;
    }
}

// ------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------
// synthetic instances on the device (parameters.py:20-28: A iid N(0,1), unit-l2 rows)
// ------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  The entry (row i, GLOBAL column k) is a pure function of
// (seed, i, k): counter = (k / 4, i, 0, "LASO"), key = seed; the four outputs make the normals of
// columns 4*(k/4) .. +3 (Box-Muller on 24-bit uniforms).  Any column sharding therefore yields
// the same matrix.
__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t (&out)[4]) {
    for (int r = 0; r < 10; ++r) {
        const unsigned long long p0 = 0xD2511F53ull * c0, p1 = 0xCD9E8D57ull * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ __forceinline__ float gauss_entry(unsigned long long seed, uint32_t row, unsigned long long gcol) {
    uint32_t x[4];
    philox4x32_10((uint32_t)(gcol >> 2), row, (uint32_t)(gcol >> 34), 0x4c41534fu, (uint32_t)seed,
                  (uint32_t)(seed >> 32), x);
    const int e = (int)(gcol & 3);
    const uint32_t a = (e & 2) ? x[2] : x[0], b = (e & 2) ? x[3] : x[1];
    const float u1 = ((float)(a >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(b >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float rad = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincospif(2.0f * u2, &sn, &cs);
    return rad * ((e & 1) ? sn : cs);
}
// local column j of block m on rank `rank` of `world` is global column m*w*world + rank*w + j
template <typename T, bool TRANS>
__global__ void __launch_bounds__(256) gen_fill(T *A, int64_t N, int w, int nblocks, int64_t brows, int64_t ld,
                                                unsigned long long seed, int rank, int world) {
    const int64_t total = (int64_t)nblocks * N * w;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t i, j, m;
        if (TRANS) { i = idx % N; j = (idx / N) % w; m = idx / (N * (int64_t)w); }
        else       { j = idx % w; i = (idx / w) % N; m = idx / (N * (int64_t)w); }
        const unsigned long long gcol = (unsigned long long)m * w * world + (unsigned long long)rank * w + j;
        const float v = gauss_entry(seed, (uint32_t)i, gcol);
        A[TRANS ? (m * brows + j) * ld + i : (m * brows + i) * ld + j] = (T)v;
    }
}
// out[i] = sum over the local columns of A_ik^2 (one thread per row i; TRANS reads are coalesced,
// row-major uses a warp per row)
template <typename T, bool TRANS>
__global__ void __launch_bounds__(256) row_sumsq(const T *A, int64_t N, int w, int nblocks, int64_t brows, int64_t ld,
                                                 double *out) {
    if (TRANS) {
        const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= N) return;
        double acc = 0.0;
        for (int64_t mj = 0; mj < (int64_t)nblocks * w; ++mj) {
            const int64_t m = mj / w, j = mj % w;
            const double v = (double)A[(m * brows + j) * ld + i];
            acc += v * v;
        }
        out[i] = acc;
    } else {
        const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
        const int lane = threadIdx.x & 31;
        if (i >= N) return;
        double acc = 0.0;
        for (int m = 0; m < nblocks; ++m) {
            const T *row = A + ((int64_t)m * brows + i) * ld;
            for (int j = lane; j < w; j += 32) {
                const double v = (double)row[j];
                acc += v * v;
            }
        }
        acc = warp_sum(acc);
        if (lane == 0) out[i] = acc;
    }
}
template <typename T, bool TRANS>
__global__ void __launch_bounds__(256) scale_rows(T *A, int64_t N, int w, int nblocks, int64_t brows, int64_t ld,
                                                  const double *scale) {
    const int64_t total = (int64_t)nblocks * N * w;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t i, j, m;
        if (TRANS) { i = idx % N; j = (idx / N) % w; m = idx / (N * (int64_t)w); }
        else       { j = idx % w; i = (idx / w) % N; m = idx / (N * (int64_t)w); }
        T *e = A + (TRANS ? (m * brows + j) * ld + i : (m * brows + i) * ld + j);
        *e = (T)((double)*e * scale[i]);
    }
}

struct b200l_ctx {
    int dtype, layout, device;
    int64_t N, K;
    int32_t nblocks, w;
    int64_t ld;        // padded leading dimension of a device block row
    int64_t brows;     // rows of a device block (N row-major, w transposed)
    int64_t xld;       // stride of x/d per block
    size_t esize;
    cudaStream_t stream;
    const void *A;
    int sm_count, smem_optin, l2_bytes;
    // solver state
    double *x, *d, *drec, *r, *b, *dsum;
    // scratch
    double *vin, *vout, *part;
    int part_chunks;
    ulonglong2 *cw_words;         // exchange words of colwsum_fused: one slab of partials per CTA
    unsigned long long cw_seq;    // launches of colwsum_fused so far (the tag of their words)
    int cw_occ, ms_ready;
    // cross-CTA exchange buffers of the fused kernel (LL words, see above)
    ulonglong2 *gLL, *dLL, *sLL;
    size_t gLL_bytes;
    int *abort_flag;
    uint32_t tag_base;            // tags already used by earlier launches
    double *gamma_state, *err_hist, *objbuf;
    unsigned long long *time_hist, *trace, *ttrace;
    int64_t trace_cap, ttrace_cap;
    long long *state;
    int32_t *order;
    int64_t hist_cap, order_cap;
    int64_t step_counter;
    int have_problem, have_diag;
    cudaEvent_t ev0, ev1;
    // tuning
    int32_t slot_target, dbg;
    CUtensorMap tmap;             // transposed layout only
    int tmap_valid;
    // multi-GPU
    int world, rank;
    ulonglong2 *peer[B200L_MAX_WORLD];   // peer[rank] = own inbox (cudaMalloc), others IPC-mapped
    size_t inbox_bytes;
    int peer_ipc;                        // the inboxes are CUDA IPC mappings owned by this library
    ulonglong2 *mc;                      // multicast (NVLS) mapping of all ranks' inboxes, or NULL
    // cached geometry
    RunParams geo;
    int grid, smem_bytes, cpt, nt_max;
    unsigned long long wait_limit_ns;
    int geo_valid;
};

static int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }
static int comm_release(b200l_ctx *c);
static int plan_geometry(b200l_ctx *c);

extern "C" const char *b200l_last_error(void) { return g_err; }
extern "C" int b200l_abi_version(void) { return B200L_ABI_VERSION; }

extern "C" int b200l_device_count(int *count) {
    if (!count) return fail("count is NULL");
    int n = 0;
    CK(cudaGetDeviceCount(&n));
    if (n <= 0) return fail("no CUDA device present (this library has no CPU fallback)");
    *count = n;
    return 0;
}

extern "C" int b200l_device_info(int device, char *name, int name_len, int *sm_count,
                                 int *smem_optin, int *l2_bytes) {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (name && name_len > 0) {
        strncpy(name, prop.name, (size_t)name_len - 1);
        name[name_len - 1] = 0;
    }
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (smem_optin) *smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (l2_bytes) *l2_bytes = prop.l2CacheSize;
    return 0;
}

extern "C" int b200l_ctx_create(b200l_ctx **out, int dtype, int layout, int64_t N, int64_t K,
                                int32_t nblocks, int device) {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (dtype != B200L_F32 && dtype != B200L_F64) return fail("dtype must be B200L_F32 or B200L_F64");
    if (layout != B200L_ROWMAJOR && layout != B200L_TRANSPOSED) return fail("bad layout %d", layout);
    if (N <= 0 || K <= 0 || nblocks <= 0) return fail("N, K, nblocks must be positive");
    if (K % nblocks != 0)
        return fail("K=%lld is not divisible by nblocks=%d (reference requirement, cpu_calculation.py:27)",
                    (long long)K, nblocks);
    int ndev = 0;
    if (b200l_device_count(&ndev)) return 1;
    if (device < 0 || device >= ndev) return fail("device %d out of range (have %d)", device, ndev);
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail("device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);

    b200l_ctx *c = new b200l_ctx();
    memset(c, 0, sizeof(*c));
    c->dtype = dtype;
    c->layout = layout;
    c->device = device;
    c->N = N;
    c->K = K;
    c->nblocks = nblocks;
    c->w = (int32_t)(K / nblocks);
    c->esize = dtype == B200L_F32 ? 4 : 8;
    const int V = (int)(16 / c->esize);
    if (layout == B200L_ROWMAJOR) {
        c->ld = round_up(c->w, V);
        c->brows = N;
        c->xld = c->ld;
    } else {
        c->ld = round_up(N, V);
        c->brows = c->w;
        c->xld = round_up(c->w, V);
    }
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = (int)prop.sharedMemPerBlockOptin;
    c->l2_bytes = prop.l2CacheSize;
    c->slot_target = 0;
    c->wait_limit_ns = 5000000000ULL;
    c->world = 1;
    c->rank = 0;

    const int64_t nx = (int64_t)nblocks * c->xld;
    const int64_t vmax = std::max<int64_t>(std::max<int64_t>(N, K), nx) + 64;
    c->part_chunks = 4 * c->sm_count;
    const int64_t part_cols = std::max<int64_t>(c->ld, c->xld);
#define ALLOC(ptr, bytes) CK(cudaMalloc((void **)&(ptr), (size_t)(bytes)))
    ALLOC(c->x, nx * 8);
    ALLOC(c->d, nx * 8);
    ALLOC(c->drec, nx * 8);
    ALLOC(c->dsum, nx * 8);
    const int64_t npad = round_up(N, 4) + 4;   // the pre-transposed layout reduces ld >= N entries into r
    ALLOC(c->r, npad * 8);
    ALLOC(c->b, npad * 8);
    ALLOC(c->vin, vmax * 8);
    ALLOC(c->vout, vmax * 8);
    ALLOC(c->part, (int64_t)c->part_chunks * part_cols * 8);
    ALLOC(c->cw_words, (int64_t)c->sm_count * CW_CG * 4 * 16);
    ALLOC(c->dLL, (c->xld + 2 * GMAX + 2) * 16);
    ALLOC(c->sLL, GMAX * 4 * 16);
    ALLOC(c->abort_flag, 64);
    ALLOC(c->gamma_state, 8);
    ALLOC(c->objbuf, 64);
    ALLOC(c->state, 64);
#undef ALLOC
    CK(cudaMemset(c->x, 0, nx * 8));
    CK(cudaMemset(c->d, 0, nx * 8));
    CK(cudaMemset(c->drec, 0, nx * 8));
    CK(cudaMemset(c->r, 0, npad * 8));
    CK(cudaMemset(c->b, 0, npad * 8));
    CK(cudaMemset(c->gamma_state, 0, 8));
    CK(cudaMemset(c->cw_words, 0, (size_t)c->sm_count * CW_CG * 4 * 16));
    CK(cudaMemset(c->state, 0, 64));
    CK(cudaMemset(c->dLL, 0, (size_t)(c->xld + 2 * GMAX + 2) * 16));
    CK(cudaMemset(c->sLL, 0, (size_t)GMAX * 4 * 16));
    CK(cudaMemset(c->abort_flag, 0, 64));
    CK(cudaEventCreate(&c->ev0));
    CK(cudaEventCreate(&c->ev1));
    *out = c;
    return 0;
}

extern "C" int b200l_ctx_destroy(b200l_ctx *c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    comm_release(c);
    void *ptrs[] = {c->x, c->d, c->drec, c->dsum, c->r, c->b, c->vin, c->vout, c->part, c->cw_words, c->gLL,
                    c->dLL, c->sLL, c->abort_flag, c->gamma_state, c->objbuf, c->state, c->err_hist,
                    c->time_hist, c->trace, c->ttrace, c->order};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    delete c;
    return 0;
}

extern "C" int b200l_ctx_ld(const b200l_ctx *c, int64_t *ld) {
    if (!c || !ld) return fail("NULL argument");
    *ld = c->ld;
    return 0;
}

extern "C" int b200l_ctx_set_stream(b200l_ctx *c, void *stream) {
    if (!c) return fail("ctx is NULL");
    c->stream = (cudaStream_t)stream;
    return 0;
}

extern "C" int b200l_ctx_bind_A(b200l_ctx *c, const void *A_dev) {
    if (!c || !A_dev) return fail("NULL argument");
    if (((uintptr_t)A_dev) % 128 != 0) return fail("A_dev must be 128-byte aligned");
    cudaPointerAttributes attr;
    CK(cudaPointerGetAttributes(&attr, A_dev));
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)
        return fail("A_dev is not a device pointer");
    c->A = A_dev;
    c->have_problem = 0;
    c->have_diag = 0;
    c->tmap_valid = 0;
    return 0;
}

// ------------------------------------------------------------------------------------
// device-level mat-vecs on block m (vectors are device doubles)
// ------------------------------------------------------------------------------------
// nmat equally shaped matrices (stride mat_stride elements), results out[y * out_stride + col], col < ncols_out
template <typename T>
static int colwsum_dev(b200l_ctx *c, const T *Ablk, int64_t M, int ncols, int64_t ld, const double *vec,
                       double *out, bool sq, int accumulate, int nmat = 1, int64_t mat_stride = 0,
                       int64_t out_stride = 0, int ncols_out = -1) {
    // chunks of rows: enough CTAs to fill the machine (a CTA is 256 threads, eight loads in flight each), few
    // partials: two per SM for one block, four per SM over all blocks of the one-pass diag(A^T A)
    const int budget = std::max(1, (nmat > 1 ? 4 : 2) * c->sm_count / nmat);
    int chunks = (int)std::min<int64_t>(budget, (M + 7) / 8);
    chunks = std::max(chunks, 1);
    int rpc = (int)((M + chunks - 1) / chunks);
    chunks = (int)((M + rpc - 1) / rpc);
    if (ncols_out < 0) ncols_out = ncols;
    const dim3 grid(chunks, nmat);
    if (sq)
        colwsum_partial<T, true><<<grid, 256, 0, c->stream>>>(Ablk, M, ncols, ld, vec, c->part, rpc, mat_stride);
    else
        colwsum_partial<T, false><<<grid, 256, 0, c->stream>>>(Ablk, M, ncols, ld, vec, c->part, rpc, mat_stride);
    reduce_partials<<<dim3((ncols_out + 7) / 8, nmat), 256, 0, c->stream>>>(c->part, chunks, ncols, out, accumulate,
                                                                           out_stride, ncols_out);
    CK(cudaGetLastError());
    return 0;
}

// one matrix, one launch (colwsum_fused): the exchange words of the chunks live in c->cw_words
template <typename T>
static int colwsum_one(b200l_ctx *c, const T *Ablk, int64_t M, int ncols, int64_t ld, const double *vec,
                       double *out, int accumulate, int ncols_out) {
    constexpr int V = VT<T>::V;
    const int ncg = ncols / V;
    const int ncs = (ncg + CW_CG - 1) / CW_CG;
    if (!c->cw_occ) {
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void *)colwsum_fused<T>, CW_THREADS, 0));
        if (occ < 1) return fail("internal: colwsum_fused does not fit on an SM");
        c->cw_occ = occ;
    }
    // row chunks: as many CTAs as SMs, at least 32 rows (one batch of every sub-group) per chunk
    int64_t rc = std::min<int64_t>(c->sm_count / std::max(ncs, 1), (M + 31) / 32);
    rc = std::max<int64_t>(1, std::min<int64_t>(rc, 32 * CW_MAXP));
    int RC = (int)rc;
    const unsigned long long seq = ++c->cw_seq;
    void *args[] = {(void *)&Ablk, (void *)&M, (void *)&ncols, (void *)&ld, (void *)&vec, (void *)&c->cw_words,
                    (void *)&seq, (void *)&out, (void *)&accumulate, (void *)&ncols_out};
    if (RC > 1)
        CK(cudaLaunchCooperativeKernel((const void *)colwsum_fused<T>, dim3(RC, ncs), dim3(CW_THREADS), args, 0,
                                       c->stream));
    else
        CK(cudaLaunchKernel((const void *)colwsum_fused<T>, dim3(1, ncs), dim3(CW_THREADS), args, 0, c->stream));
    return 0;
}

template <typename T>
static int rowdot_dev(b200l_ctx *c, const T *Ablk, int64_t M, int ncols, int64_t ld, const double *vec,
                      double *out, bool sq, int accumulate, int64_t group = 0, int64_t out_stride = 0) {
    constexpr int V = VT<T>::V;
    const int ncg = ncols / V;
    // two CTAs of eight warps per SM; short matrices: several warps per row until most warps have one
    const int blocks_max = 2 * c->sm_count;
    int wpr = 1;
    while (wpr < 8 && M * wpr * 4 < (int64_t)blocks_max * 8 * 3 && ncg / (2 * wpr) >= 32) wpr *= 2;
    const int64_t ctas_needed = (M * wpr + 7) / 8;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(blocks_max, ctas_needed));
    const bool vreg = (ncg + wpr - 1) / wpr <= 32 * 8;
    if (group <= 0) { group = M; out_stride = 0; }
#define RD_LAUNCH(SQ_, VR_)                                                                                         \
    rowdot_kernel<T, SQ_, VR_><<<blocks, 256, 0, c->stream>>>(Ablk, M, ncols, ld, vec, out, accumulate, group, \
                                                               out_stride, wpr)
    if (sq) { if (vreg) RD_LAUNCH(true, true); else RD_LAUNCH(true, false); }
    else    { if (vreg) RD_LAUNCH(false, true); else RD_LAUNCH(false, false); }
#undef RD_LAUNCH
    CK(cudaGetLastError());
    return 0;
}

// the TMA-streamed row dots (rowdot_stream) for matrices that fill the machine; *done stays false when the
// shape is left to the load-batch kernel (small matrices, few rows, vec too long for shared memory)
constexpr int64_t MS_MIN_BYTES = 4 << 20;
constexpr int MS_TILE_TARGET = 24 << 10;
template <typename T>
static int rowdot_stream_try(b200l_ctx *c, const T *Ablk, int64_t M, int ncols, int64_t ld, const double *vec,
                             double *out, int accumulate, bool *done) {
    constexpr int V = VT<T>::V;
    *done = false;
    if (c->dbg & DBG_LOAD_BATCH) return 0;                       // (load-batch kernels only: tests, comparisons)
    if ((int64_t)M * ncols * (int64_t)sizeof(T) < MS_MIN_BYTES || M < 2 * c->sm_count) return 0;
    const int ncg = ncols / V;
    MsParams p;
    memset(&p, 0, sizeof(p));
    p.A = Ablk; p.M = M; p.ld = ld; p.ncols = ncols; p.vec = vec; p.out = out; p.accumulate = accumulate;
    p.SG = ncg <= 256 ? ncg : std::min(ncg, 1024);
    p.ncs = (ncg + p.SG - 1) / p.SG;
    const bool vreg = ncg <= 256;
    const int vec_bytes = vreg ? 0 : (int)round_up((int64_t)ncols * 8, 128);
    if (vec_bytes > 96 * 1024) return 0;
    p.TR = std::max(1, std::min(MS_NW, MS_TILE_TARGET / (p.SG * 16)));
    p.RC = (int)std::min<int64_t>(c->sm_count, M / p.TR);
    if (p.RC < 1) return 0;
    p.coop = (!vreg && p.TR == 1) ? 1 : 0;
    p.contig = p.ncs == 1 && ld == ncols;
    p.slot_bytes = (int)round_up((int64_t)p.TR * p.SG * 16, 128);
    p.off_vec = 256;
    p.off_part = p.off_vec + vec_bytes;
    p.off_ring = (int)round_up(p.off_part + 2 * MS_NW * 8, 1024);
    p.S = std::min(MS_MAXS, (c->smem_optin - p.off_ring) / p.slot_bytes);
    if (p.S < 3) return 0;
    const int smem = p.off_ring + p.S * p.slot_bytes;
    const void *fn = vreg ? (const void *)rowdot_stream<T, true> : (const void *)rowdot_stream<T, false>;
    const int fidx = vreg ? 1 : 2;
    if (!(c->ms_ready & (1 << fidx))) {
        CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, c->smem_optin));
        c->ms_ready |= 1 << fidx;
    }
    void *args[] = {(void *)&p};
    CK(cudaLaunchKernel(fn, dim3(p.RC), dim3(MS_THREADS), args, (size_t)smem, c->stream));
    *done = true;
    return 0;
}

// g[xld] = A_m^T r[N]
template <typename T>
static int gemv_t_dev(b200l_ctx *c, int m, const double *r, double *g) {
    const T *Ablk = reinterpret_cast<const T *>(c->A) + (int64_t)m * c->brows * c->ld;
    if (c->layout == B200L_ROWMAJOR)        // only the w real columns are written (g may hold exactly w entries)
        return colwsum_one<T>(c, Ablk, c->N, (int)c->ld, c->ld, r, g, 0, c->w);
    bool done = false;
    if (rowdot_stream_try<T>(c, Ablk, c->w, (int)c->ld, c->ld, r, g, 0, &done)) return 1;
    return done ? 0 : rowdot_dev<T>(c, Ablk, c->w, (int)c->ld, c->ld, r, g, false, 0);
}
// q[N] (+)= A_m d[xld]
template <typename T>
static int gemv_n_dev(b200l_ctx *c, int m, const double *dvec, double *q, int accumulate) {
    const T *Ablk = reinterpret_cast<const T *>(c->A) + (int64_t)m * c->brows * c->ld;
    if (c->layout == B200L_ROWMAJOR) {
        bool done = false;
        if (rowdot_stream_try<T>(c, Ablk, c->N, (int)c->ld, c->ld, dvec, q, accumulate, &done)) return 1;
        return done ? 0 : rowdot_dev<T>(c, Ablk, c->N, (int)c->ld, c->ld, dvec, q, false, accumulate);
    }
    // (the pre-transposed block has ld >= N padded entries per column: only the N real ones are written)
    return colwsum_one<T>(c, Ablk, c->w, (int)c->ld, c->ld, dvec, q, accumulate, (int)c->N);
}

static int need_A(b200l_ctx *c) {
    if (!c) return fail("ctx is NULL");
    if (!c->A) return fail("no device matrix bound (call b200l_ctx_bind_A first)");
    CK(cudaSetDevice(c->device));
    return 0;
}

// d = diag(A^T A) of every block in ONE pass over A (two or three launches in all); kept until another
// matrix is bound or its entries change (gpu_calculation.py:246-261 recomputes it per call)
template <typename T>
static int compute_diag_t(b200l_ctx *c) {
    const T *A = reinterpret_cast<const T *>(c->A);
    if (c->layout == B200L_ROWMAJOR)
        return colwsum_dev<T>(c, A, c->N, (int)c->ld, c->ld, nullptr, c->dsum, true, 0, c->nblocks,
                              c->brows * c->ld, c->xld);
    // transposed: the blocks are consecutive rows of one (nblocks * w) x ld matrix; the padding of
    // a row (entries N .. ld-1) is zero
    return rowdot_dev<T>(c, A, (int64_t)c->nblocks * c->w, (int)c->ld, c->ld, nullptr, c->dsum, true, 0, c->w, c->xld);
}

static int compute_diag(b200l_ctx *c) {
    if (c->have_diag) return 0;
    const int64_t nx = (int64_t)c->nblocks * c->xld;
    CK(cudaMemsetAsync(c->dsum, 0, (size_t)nx * 8, c->stream));
    const int rc = c->dtype == B200L_F32 ? compute_diag_t<float>(c) : compute_diag_t<double>(c);
    if (rc) return rc;
    finish_diag<<<(int)((nx + 255) / 256), 256, 0, c->stream>>>(c->dsum, c->d, c->drec, nx);
    CK(cudaGetLastError());
    c->have_diag = 1;
    return 0;
}

extern "C" int b200l_diag_ata(b200l_ctx *c, double *out_host) {
    if (need_A(c)) return 1;
    if (!out_host) return fail("out_host is NULL");
    if (compute_diag(c)) return 1;
    CK(cudaMemcpy2DAsync(out_host, (size_t)c->w * 8, c->d, (size_t)c->xld * 8, (size_t)c->w * 8,
                         (size_t)c->nblocks, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int b200l_gemv_t(b200l_ctx *c, int32_t m, const double *r_host, double *g_host) {
    if (need_A(c)) return 1;
    if (m < 0 || m >= c->nblocks) return fail("block index %d out of range", m);
    if (!r_host || !g_host) return fail("NULL vector");
    const int64_t nin = c->layout == B200L_ROWMAJOR ? c->N : c->ld;
    CK(cudaMemsetAsync(c->vin, 0, (size_t)nin * 8, c->stream));
    CK(cudaMemcpyAsync(c->vin, r_host, (size_t)c->N * 8, cudaMemcpyHostToDevice, c->stream));
    int rc = c->dtype == B200L_F32 ? gemv_t_dev<float>(c, m, c->vin, c->vout)
                                   : gemv_t_dev<double>(c, m, c->vin, c->vout);
    if (rc) return rc;
    CK(cudaMemcpyAsync(g_host, c->vout, (size_t)c->w * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int b200l_gemv_n(b200l_ctx *c, int32_t m, const double *d_host, double *q_host) {
    if (need_A(c)) return 1;
    if (m < 0 || m >= c->nblocks) return fail("block index %d out of range", m);
    if (!d_host || !q_host) return fail("NULL vector");
    CK(cudaMemsetAsync(c->vin, 0, (size_t)c->xld * 8, c->stream));
    CK(cudaMemcpyAsync(c->vin, d_host, (size_t)c->w * 8, cudaMemcpyHostToDevice, c->stream));
    int rc = c->dtype == B200L_F32 ? gemv_n_dev<float>(c, m, c->vin, c->vout, 0)
                                   : gemv_n_dev<double>(c, m, c->vin, c->vout, 0);
    if (rc) return rc;
    CK(cudaMemcpyAsync(q_host, c->vout, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// device-vector variants: no staging copy, no synchronisation (the work is queued on the
// context's stream).  r_dev needs N doubles (the pre-transposed layout reads ld >= N: the
// vector has to be padded with zeros up to b200l_ctx_ld), g_dev gets w doubles.
static int check_dev_ptr(const void *p, const char *what) {
    cudaPointerAttributes attr;
    CK(cudaPointerGetAttributes(&attr, p));
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)
        return fail("%s is not a device pointer", what);
    return 0;
}

extern "C" int b200l_gemv_t_dev(b200l_ctx *c, int32_t m, const double *r_dev, double *g_dev) {
    if (need_A(c)) return 1;
    if (m < 0 || m >= c->nblocks) return fail("block index %d out of range", m);
    if (!r_dev || !g_dev) return fail("NULL vector");
    if (check_dev_ptr(r_dev, "r_dev") || check_dev_ptr(g_dev, "g_dev")) return 1;
    const double *rin = r_dev;
    if (c->layout == B200L_TRANSPOSED && c->ld != c->N) {     // zero-padded copy for the 16-byte row reads
        CK(cudaMemsetAsync(c->vin, 0, (size_t)c->ld * 8, c->stream));
        CK(cudaMemcpyAsync(c->vin, r_dev, (size_t)c->N * 8, cudaMemcpyDeviceToDevice, c->stream));
        rin = c->vin;
    }
    return c->dtype == B200L_F32 ? gemv_t_dev<float>(c, m, rin, g_dev) : gemv_t_dev<double>(c, m, rin, g_dev);
}

extern "C" int b200l_gemv_n_dev(b200l_ctx *c, int32_t m, const double *d_dev, double *q_dev) {
    if (need_A(c)) return 1;
    if (m < 0 || m >= c->nblocks) return fail("block index %d out of range", m);
    if (!d_dev || !q_dev) return fail("NULL vector");
    if (check_dev_ptr(d_dev, "d_dev") || check_dev_ptr(q_dev, "q_dev")) return 1;
    const double *din = d_dev;
    if (c->xld != c->w) {                                     // zero-padded copy for the 16-byte row reads
        CK(cudaMemsetAsync(c->vin, 0, (size_t)c->xld * 8, c->stream));
        CK(cudaMemcpyAsync(c->vin, d_dev, (size_t)c->w * 8, cudaMemcpyDeviceToDevice, c->stream));
        din = c->vin;
    }
    return c->dtype == B200L_F32 ? gemv_n_dev<float>(c, m, din, q_dev, 0) : gemv_n_dev<double>(c, m, din, q_dev, 0);
}

// ------------------------------------------------------------------------------------
// synthetic instance generation (SURVEY.md 8f-2; reference recipe parameters.py:20-28)
// ------------------------------------------------------------------------------------
template <typename T>
static int gen_dispatch(b200l_ctx *c, int what, unsigned long long seed, int rank, int world, const double *scale,
                        double *out) {
    T *A = reinterpret_cast<T *>(const_cast<void *>(c->A));
    const bool trans = c->layout == B200L_TRANSPOSED;
    const int64_t total = (int64_t)c->nblocks * c->N * c->w;
    const int grid = (int)std::min<int64_t>((total + 255) / 256, (int64_t)c->sm_count * 32);
    if (what == 0) {
        if (trans) gen_fill<T, true><<<grid, 256, 0, c->stream>>>(A, c->N, c->w, c->nblocks, c->brows, c->ld, seed, rank, world);
        else gen_fill<T, false><<<grid, 256, 0, c->stream>>>(A, c->N, c->w, c->nblocks, c->brows, c->ld, seed, rank, world);
    } else if (what == 1) {
        if (trans) row_sumsq<T, true><<<(int)((c->N + 255) / 256), 256, 0, c->stream>>>(A, c->N, c->w, c->nblocks, c->brows, c->ld, out);
        else row_sumsq<T, false><<<(int)((c->N * 32 + 255) / 256), 256, 0, c->stream>>>(A, c->N, c->w, c->nblocks, c->brows, c->ld, out);
    } else {
        if (trans) scale_rows<T, true><<<grid, 256, 0, c->stream>>>(A, c->N, c->w, c->nblocks, c->brows, c->ld, scale);
        else scale_rows<T, false><<<grid, 256, 0, c->stream>>>(A, c->N, c->w, c->nblocks, c->brows, c->ld, scale);
    }
    CK(cudaGetLastError());
    return 0;
}

extern "C" int b200l_gen_gaussian(b200l_ctx *c, uint64_t seed, int32_t rank, int32_t world) {
    if (need_A(c)) return 1;
    if (world < 1 || rank < 0 || rank >= world) return fail("bad rank %d / world %d", rank, world);
    const int rc = c->dtype == B200L_F32 ? gen_dispatch<float>(c, 0, seed, rank, world, nullptr, nullptr)
                                         : gen_dispatch<double>(c, 0, seed, rank, world, nullptr, nullptr);
    if (rc) return rc;
    c->have_problem = 0;
    c->have_diag = 0;
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int b200l_row_sumsq(b200l_ctx *c, double *out_host) {
    if (need_A(c)) return 1;
    if (!out_host) return fail("out_host is NULL");
    const int rc = c->dtype == B200L_F32 ? gen_dispatch<float>(c, 1, 0, 0, 1, nullptr, c->vout)
                                         : gen_dispatch<double>(c, 1, 0, 0, 1, nullptr, c->vout);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out_host, c->vout, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int b200l_scale_rows(b200l_ctx *c, const double *scale_host) {
    if (need_A(c)) return 1;
    if (!scale_host) return fail("scale_host is NULL");
    CK(cudaMemcpyAsync(c->vin, scale_host, (size_t)c->N * 8, cudaMemcpyHostToDevice, c->stream));
    const int rc = c->dtype == B200L_F32 ? gen_dispatch<float>(c, 2, 0, 0, 1, c->vin, nullptr)
                                         : gen_dispatch<double>(c, 2, 0, 0, 1, c->vin, nullptr);
    if (rc) return rc;
    c->have_problem = 0;
    c->have_diag = 0;
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------------------------
// solver state
// ------------------------------------------------------------------------------------
static int reset_state(b200l_ctx *c) {
    const int64_t nx = (int64_t)c->nblocks * c->xld;
    CK(cudaMemsetAsync(c->x, 0, (size_t)nx * 8, c->stream));
    neg_copy<<<(int)((c->N + 255) / 256), 256, 0, c->stream>>>(c->b, c->r, c->N, -1.0);
    CK(cudaGetLastError());
    CK(cudaMemsetAsync(c->state, 0, 64, c->stream));
    CK(cudaMemsetAsync(c->gamma_state, 0, 8, c->stream));
    c->step_counter = 0;
    return 0;
}

extern "C" int b200l_set_problem(b200l_ctx *c, const double *b_host) {
    if (need_A(c)) return 1;
    if (!b_host) return fail("b_host is NULL");
    CK(cudaMemcpyAsync(c->b, b_host, (size_t)c->N * 8, cudaMemcpyHostToDevice, c->stream));
    if (compute_diag(c)) return 1;          // no-op when b200l_diag_ata already ran on this matrix
    c->have_problem = 1;
    return reset_state(c);
}

extern "C" int b200l_reset(b200l_ctx *c) {
    if (need_A(c)) return 1;
    if (!c->have_problem) return fail("b200l_set_problem has not been called");
    return reset_state(c);
}

// warm start of the next solve from the current x and r (regularisation path): only the
// per-sweep stop counter and the position in the cyclic block order restart
extern "C" int b200l_restart_counters(b200l_ctx *c) {
    if (need_A(c)) return 1;
    if (!c->have_problem) return fail("b200l_set_problem has not been called");
    CK(cudaMemsetAsync(c->state, 0, 64, c->stream));
    c->step_counter = 0;
    return 0;
}

extern "C" int b200l_set_x(b200l_ctx *c, const double *x_host) {
    if (need_A(c)) return 1;
    if (!c->have_problem) return fail("b200l_set_problem has not been called");
    if (!x_host) return fail("x_host is NULL");
    const int64_t nx = (int64_t)c->nblocks * c->xld;
    CK(cudaMemsetAsync(c->x, 0, (size_t)nx * 8, c->stream));
    CK(cudaMemcpy2DAsync(c->x, (size_t)c->xld * 8, x_host, (size_t)c->w * 8, (size_t)c->w * 8,
                         (size_t)c->nblocks, cudaMemcpyHostToDevice, c->stream));
    neg_copy<<<(int)((c->N + 255) / 256), 256, 0, c->stream>>>(c->b, c->r, c->N, -1.0);
    CK(cudaGetLastError());
    for (int m = 0; m < c->nblocks; ++m) {
        const double *xm = c->x + (int64_t)m * c->xld;
        int rc = c->dtype == B200L_F32 ? gemv_n_dev<float>(c, m, xm, c->r, 1)
                                       : gemv_n_dev<double>(c, m, xm, c->r, 1);
        if (rc) return rc;
    }
    CK(cudaMemsetAsync(c->state, 0, 64, c->stream));
    c->step_counter = 0;
    return 0;
}

extern "C" int b200l_get_x(b200l_ctx *c, double *x_host) {
    if (!c || !x_host) return fail("NULL argument");
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpy2DAsync(x_host, (size_t)c->w * 8, c->x, (size_t)c->xld * 8, (size_t)c->w * 8,
                         (size_t)c->nblocks, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int b200l_get_r(b200l_ctx *c, double *r_host) {
    if (!c || !r_host) return fail("NULL argument");
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(r_host, c->r, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int b200l_objective(b200l_ctx *c, double mu, double *value) {
    if (!c || !value) return fail("NULL argument");
    CK(cudaSetDevice(c->device));
    objective_kernel<<<1, 1024, 0, c->stream>>>(c->r, c->N, c->x, (int64_t)c->nblocks * c->xld, mu,
                                                c->objbuf);
    CK(cudaGetLastError());
    double h[3];
    CK(cudaMemcpyAsync(h, c->objbuf, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    *value = h[0];
    return 0;
}

// the two terms separately: with column shards over several GPUs every rank holds the full
// residual (rss is the global 0.5*|Ax-b|^2 when halved) but only its slice of x, so the l1
// term has to be summed over the ranks by the caller (path.lasso_path and bench.py do)
extern "C" int b200l_objective_terms(b200l_ctx *c, double *rss, double *l1) {
    if (!c || !rss || !l1) return fail("NULL argument");
    CK(cudaSetDevice(c->device));
    objective_kernel<<<1, 1024, 0, c->stream>>>(c->r, c->N, c->x, (int64_t)c->nblocks * c->xld, 0.0, c->objbuf);
    CK(cudaGetLastError());
    double h[3];
    CK(cudaMemcpyAsync(h, c->objbuf, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    *rss = h[1];
    *l1 = h[2];
    return 0;
}

// caller-supplied diagonal (the d_ATA argument of the solver classes, lasso.py:26-30) instead of
// the one computed from the bound matrix: d (nblocks, w) doubles, 1/d taken like lasso.py:29-30
extern "C" int b200l_set_diag(b200l_ctx *c, const double *d_host) {
    if (need_A(c)) return 1;
    if (!d_host) {                      // back to the diagonal of the bound matrix (recomputed when next needed)
        c->have_diag = 0;
        return 0;
    }
    const int64_t nx = (int64_t)c->nblocks * c->xld;
    CK(cudaMemsetAsync(c->dsum, 0, (size_t)nx * 8, c->stream));
    CK(cudaMemcpy2DAsync(c->dsum, (size_t)c->xld * 8, d_host, (size_t)c->w * 8, (size_t)c->w * 8,
                         (size_t)c->nblocks, cudaMemcpyHostToDevice, c->stream));
    finish_diag<<<(int)((nx + 255) / 256), 256, 0, c->stream>>>(c->dsum, c->d, c->drec, nx);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(c->stream));
    c->have_diag = 1;
    return 0;
}

// ------------------------------------------------------------------------------------
// fused launch
// ------------------------------------------------------------------------------------
extern "C" int b200l_set_tuning(b200l_ctx *c, int32_t slot_bytes_target, int32_t max_inflight_tiles) {
    if (!c) return fail("ctx is NULL");
    // the ring's empty barriers already cap the copies in flight at the ring size; no other cap is offered
    if (max_inflight_tiles != 0)
        return fail("max_inflight_tiles=%d: only 0 (as many bulk copies in flight as ring slots) is supported",
                    max_inflight_tiles);
    c->slot_target = slot_bytes_target > 0 ? slot_bytes_target : 0;   // 0: chosen per shape
    c->geo_valid = 0;
    return 0;
}

typedef void (*fused_fn)(const RunParams, const CUtensorMap);

template <typename T, int MODE>
static fused_fn pick_kernel(int cpt, bool trans) {
    if (trans) return cpt == 1 ? lasso_fused<T, 1, true, MODE> : lasso_fused<T, 2, true, MODE>;
    switch (cpt) {
        case 1: return lasso_fused<T, 1, false, MODE>;
        case 2: return lasso_fused<T, 2, false, MODE>;
        case 4: return lasso_fused<T, 4, false, MODE>;
        case 8: return lasso_fused<T, 8, false, MODE>;
        default: return nullptr;
    }
}

// mode: 0 plain single GPU, 1 multi-GPU, 2 tracing or diagnostic switches in use (see MODE)
static fused_fn ctx_kernel(const b200l_ctx *c, int mode) {
    const bool trans = c->layout == B200L_TRANSPOSED;
    const bool f32 = c->dtype == B200L_F32;
    if (mode == 2) return f32 ? pick_kernel<float, 2>(c->cpt, trans) : pick_kernel<double, 2>(c->cpt, trans);
    if (mode == 1) return f32 ? pick_kernel<float, 1>(c->cpt, trans) : pick_kernel<double, 1>(c->cpt, trans);
    return f32 ? pick_kernel<float, 0>(c->cpt, trans) : pick_kernel<double, 0>(c->cpt, trans);
}

// tensor map of the pre-transposed matrix: 2-D (ldT residual entries, nblocks*w columns)
typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

static int make_tensor_map(b200l_ctx *c) {
    static encode_tiled_fn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) return fail("cuTensorMapEncodeTiled is not available");
        encode = (encode_tiled_fn)fn;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)c->ld, (cuuint64_t)c->nblocks * (cuuint64_t)c->brows};
    const cuuint64_t strides[1] = {(cuuint64_t)c->ld * c->esize};
    const cuuint32_t box[2] = {(cuuint32_t)c->geo.BXb, (cuuint32_t)c->geo.TJ};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&c->tmap, c->dtype == B200L_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64,
                              2, const_cast<void *>(c->A), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    c->tmap_valid = 1;
    return 0;
}

static int plan_geometry(b200l_ctx *c) {
    if (c->geo_valid) return 0;
    const bool trans = c->layout == B200L_TRANSPOSED;
    RunParams &g = c->geo;
    memset(&g, 0, sizeof(g));
    const int es = (int)c->esize, V = 16 / es;
    // columns of a block incl. padding (stride of x / d per block, width of the exchange)
    const int ld = trans ? (int)c->xld : (int)c->ld;
    const int64_t rowbytes = (int64_t)ld * es;
    if (!trans && rowbytes > 32768)
        return fail("block width w=%d needs %lld-byte rows; the fused kernel supports rows up to 32 KiB "
                    "(use more column blocks)", c->w, (long long)rowbytes);
    const int G = std::min(c->sm_count, GMAX);
    const int rows_max = trans ? V * (int)(((c->N + V - 1) / V + G - 1) / G) : (int)((c->N + G - 1) / G);
    const int ncg = ld / V;
    int cpt = 1;
    while (!trans && cpt * NTC < ncg) cpt *= 2;
    if (cpt > 8) return fail("internal: cpt=%d", cpt);
    const int nrg = (!trans && cpt == 1) ? std::max(1, NTC / ncg) : 1;
    // rows per tile: as many as fit the slot target, whole quads when possible, at most 64
    // default tile size (measured): blocks that stay in L2 between the passes (C2: 40 MB) are
    // bound by the exchanges and like 48 KB tiles and one more ring slot; blocks that stream from
    // HBM in both passes (C3, C4: 250-320 MB) like 64 KB tiles
    const bool l2_resident = 2 * (int64_t)c->brows * c->ld * es <= (int64_t)c->l2_bytes * 3 / 4;
    const int64_t slot_target = c->slot_target > 0 ? c->slot_target : (l2_resident && !trans ? 49152 : 65536);
    int TR = (int)std::min<int64_t>(64, std::max<int64_t>(1, slot_target / rowbytes));
    TR = std::min(TR, (int)round_up(std::max(rows_max, 1), 4));
    if (TR >= 4) TR &= ~3;
    // transposed layout: a tile is TJ columns x BX residual entries, fetched as NBX boxes of BXb = BXVb * V entries
    // (at most 256 elements per box dimension).  P1 = NTC / TJ threads share a column in pass 1; BXVb = P1 * odd
    // keeps the 16-byte reads of a quarter-warp (8 / P1 columns x P1 parts) on distinct banks.  The values are
    // chosen below, once the fixed part of the shared memory is known.
    int BXV = 1, BX = V, TJ = NTC, nt_t = 1, nparts = 1, NBX = 1, BXVb = 1, P1 = 1;
    // columns of every block owned by one CTA: a power of two (shift/mask addressing)
    int cs = 1, cs_shift = 0;
    while (cs * G < ld) { cs *= 2; ++cs_shift; }
    if (cs > MAX_CS)
        return fail("block width w=%d is too wide for the fused kernel: each of the %d CTAs owns at most %d columns "
                    "of a block, so blocks of up to %d columns (padded) are supported (use more column blocks)",
                    c->w, G, MAX_CS, G * MAX_CS);
    // the partial gradient goes out straight from registers when every thread holds complete column sums
    // (one row group) and a column group (4 words, two 256-bit stores) fits one message of cs * es / 4 words;
    // otherwise the row groups are combined through shared memory first
    const int direct = (trans || (nrg == 1 && cs * (es / 4) >= 4)) ? 1 : 0;
    int slot_bytes = trans ? 0 : (int)round_up((int64_t)TR * rowbytes, 128);
    int rows_pad = trans ? 0 : (int)round_up(std::max(rows_max, 1), std::max(TR, 8));

    int off = 0;
    auto take = [&](int bytes) { int o = off; off += (int)round_up(bytes, 128); return o; };
    auto fixed_part = [&](RunParams *out) {
        const int o_bar = take(2 * 64 * 8);                       // barriers (up to 64 slots)
        const int o_ctl = take((int)sizeof(Ctl));
        const int o_rloc = take(rows_pad * 8);
        const int o_qloc = take(rows_pad * 8);
        const int o_rT = take(rows_pad * es);
        const int o_qT = take(rows_pad * es);
        // the step D (written after the gather, read in pass 2) overlays the row-group
        // partials (written after pass 1, read before the gather): two barriers apart
        const int o_redT = take(trans ? nt_t * TJ * es : (direct ? ld * es : nrg * 2 * ld * es));
        const int o_red2 = take(trans ? nparts * BX * es : 16);
        const int o_delta = o_redT;
        const int o_red = take(NTC * 16);                          // gather partials per thread
        const int o_small = take((2 * MAX_CS + 2 * NW) * 8);      // l1s, es, lsred
        const int o_qpart = take(rows_pad * 8);
        const int o_tilecnt = take(128 * 4);
        if (out) {
            out->off_bar = o_bar; out->off_ctl = o_ctl; out->off_rloc = o_rloc; out->off_qloc = o_qloc;
            out->off_rT = o_rT; out->off_qT = o_qT; out->off_delta = o_delta; out->off_redT = o_redT;
            out->off_red = o_red; out->off_small = o_small; out->off_qpart = o_qpart;
            out->off_red2 = o_red2; out->off_tilecnt = o_tilecnt;
        }
    };
    if (trans) {
        // columns per tile: one per thread in pass 1 when a CTA's share of a column is short; longer shares halve
        // TJ (P1 = 2, 4, 8 threads per column) until the ring holds at least two tiles.  Among the feasible
        // shapes the one that fetches the fewest padding entries wins, then the one with three or more slots,
        // then the widest tile.  (fp32 C2: 256 x 68, three slots; fp64 C2: 128 x 68; fp32 C4 shard: 64 x 352 in
        // two boxes of 176.)
        const int need = (rows_max + V - 1) / V;             // 16-byte groups of residual entries per CTA
        const int maxb = 256 / V;                            // groups per box
        double best = 1e30;
        int bP1 = 0, bNBX = 0, bBXVb = 0;
        for (int p1 = 1; p1 <= 8; p1 *= 2) {
            const int nb0 = (need + maxb - 1) / maxb;
            for (int nb = nb0; nb <= nb0 + 2; ++nb) {
                int k = ((need + nb - 1) / nb + p1 - 1) / p1;
                if (!(k & 1)) ++k;
                const int bxvb = p1 * k;
                if (bxvb > maxb || nb * bxvb > NTC) continue;
                BXV = nb * bxvb; BX = BXV * V; TJ = NTC / p1;
                nt_t = (c->w + TJ - 1) / TJ;
                nparts = std::max(1, std::min(NTC / BXV, 32));
                rows_pad = (int)round_up(BX, 8);
                slot_bytes = (int)round_up((int64_t)TJ * BX * es, 128);
                if (c->slot_target > 0 && slot_bytes > c->slot_target && p1 < 8) continue;   // (b200l_set_tuning)
                off = 0;
                fixed_part(nullptr);
                const int slots = (c->smem_optin - off) / slot_bytes;
                if (slots < 2) continue;
                const double cost = (double)BXV / need * (slots >= 3 ? 1.0 : 1.03) * (1.0 + 1e-3 * (nb - nb0)) *
                                    (1.0 + 1e-4 * p1);
                if (cost < best) { best = cost; bP1 = p1; bNBX = nb; bBXVb = bxvb; }
            }
        }
        if (!bP1)
            return fail("transposed layout: N/#SM = %d residual entries per CTA do not fit the fused kernel "
                        "(at most %d); use the row-major layout", rows_max, NTC * V);
        P1 = bP1; NBX = bNBX; BXVb = bBXVb;
        cpt = (P1 == 1 && NBX == 1) ? 1 : 2;              // (selects the kernel instantiation, see TGEN)
        BXV = NBX * BXVb; BX = BXV * V; TJ = NTC / P1;
        nt_t = (c->w + TJ - 1) / TJ;
        nparts = std::max(1, std::min(NTC / BXV, 32));
        rows_pad = (int)round_up(BX, 8);
        slot_bytes = (int)round_up((int64_t)TJ * BX * es, 128);
    }
    // the ring goes first (offset 0); sized after the fixed part is known
    off = 0;
    fixed_part(nullptr);
    const int fixed = off;
    const int avail = c->smem_optin - fixed;
    int S = avail / slot_bytes;
    if (S > 60) S = 60;
    if (S < 2)
        return fail("shared memory too small for the fused kernel: fixed=%d slot=%d optin=%d (N/SM=%d rows, "
                    "w=%d)", fixed, slot_bytes, c->smem_optin, rows_max, c->w);
    const int nt_max = trans ? nt_t : (rows_max + TR - 1) / TR;
    if (S > 2 * nt_max + 2) S = 2 * nt_max + 2;   // more slots than two passes of tiles is useless
    off = 0;
    take(S * slot_bytes);
    fixed_part(&g);
    c->smem_bytes = off;
    c->grid = G;
    c->cpt = cpt;
    c->nt_max = nt_max;
    // multi-GPU send side: the sender warp sends the rows of a pass-2 tile when the consumer warps are
    // done with it (row-major, up to 128 tiles: its counters); otherwise the lane that finishes a row
    // stores it to every peer itself.  With a single peer the consumer lanes win: +1 % on 2 GPUs.  On 8
    // GPUs the sender warp wins even when a multicast mapping makes it one store per row -- measured per
    // block step: sender warp + multimem 18.9 us, sender warp + 7 unicast stores 19.2, consumer lanes
    // + multimem 20.2, consumer lanes + unicast 23.9
    g.tile_sends = (c->world > 2 && !trans && nt_max <= 128) ? 1 : 0;
    // exchange geometry
    const int wpc = es / 4;
    // message = the cs columns of one reader, cs * wpc words: a power of two that divides NTC
    // (thread = word in the gather)
    const int mw = cs * wpc;
    int mw_shift = 0;
    while ((1 << mw_shift) < mw) ++mw_shift;
    if ((1 << mw_shift) != mw || mw > NTC) return fail("internal: message width %d", mw);
    const int nown = (ld + cs - 1) / cs;                 // CTAs that own at least one column
    g.TR = TR; g.S = S; g.slot_bytes = slot_bytes; g.cs = cs; g.cs_shift = cs_shift;
    g.ring_bytes = S * slot_bytes;
    g.nrg = nrg; g.ncg = ncg; g.rows_pad = rows_pad; g.rows_max_ = rows_max;
    g.mw = mw; g.mw_shift = mw_shift; g.nown = nown; g.direct_pub = direct;
    // the step D: fp32 packs two columns per word when a CTA owns at least four (a whole 32-byte sector
    // per store); a sector then holds 2 * dpw columns of ONE owner CTA
    g.dpw = (es == 4 && cs >= 4) ? 2 : 1;
    g.dsec = cs >= 2 * g.dpw ? 1 : 0;
    g.ackbase = (int)round_up(ld / g.dpw, 2);
    g.BX = BX; g.BXV = BXV; g.TJ = TJ; g.nparts = nparts; g.nt_t = nt_t;
    g.NBX = NBX; g.BXb = BXVb * V; g.BXVb = BXVb; g.P1 = P1;
    c->tmap_valid = 0;
    // HBM one block ahead through L2 only pays when this block (re-read by pass 2) and the next
    // one fit in L2 together; for larger blocks the prefetched lines would be evicted before use
    const int64_t block_bytes = (int64_t)c->brows * c->ld * es;
    g.l2_ahead = 2 * block_bytes > (int64_t)c->l2_bytes * 3 / 4 ? 0 : 1;
    // The producer starts re-streaming the slab for pass 2 once this CTA's gather is complete (the gate), so
    // that the tiles are staged in the ring while the rest of the exchange runs (measured on C2: 810 sweeps/s;
    // from the publish of the partial gradient on 788; at once 660-700, the gather's loads queue behind the
    // tiles on the L2 link).  The last ring slot is only filled once the step-D gather is complete (the second
    // gate, gate2_tiles early tiles): with all four slots in flight
    // the gather's polls queue behind one more tile on the L2 link (measured on C2, one GPU, same box: 832.5 vs
    // 822.5 sweeps/s; holding back two slots 812, three 760).  Blocks that stay in L2, one GPU, row-major, at
    // least four slots.
    g.gate2_tiles = (l2_resident && !trans && c->world == 1 && S >= 4) ? S - 1 : 0;

    // inboxes of the partial block gradients: [G readers][G writers][cs][WPC] LL words
    const size_t need = (size_t)G * G * mw * 16;
    if (c->gLL_bytes < need) {
        if (c->gLL) CK(cudaFree(c->gLL));
        c->gLL = nullptr;
        CK(cudaMalloc((void **)&c->gLL, need));
        c->gLL_bytes = need;
        CK(cudaMemsetAsync(c->gLL, 0, need, c->stream));
    }

    for (int full = 0; full < 3; ++full) {
        fused_fn fn = ctx_kernel(c, full);
        if (!fn) return fail("internal: no kernel for cpt=%d", cpt);
        CK(cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, c->smem_bytes));
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void *)fn, NTHREADS,
                                                         c->smem_bytes));
        if (occ < 1) return fail("fused kernel does not fit on an SM (smem=%d)", c->smem_bytes);
    }
    int coop = 0;
    CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, c->device));
    if (!coop) return fail("device does not support cooperative launch");
    c->geo_valid = 1;
    return 0;
}

extern "C" int b200l_run_config(b200l_ctx *c, int32_t *grid, int32_t *threads, int32_t *smem_bytes,
                                int32_t *tile_rows, int32_t *ring_slots, int32_t *tiles_per_slab) {
    if (need_A(c)) return 1;
    if (plan_geometry(c)) return 1;
    if (grid) *grid = c->grid;
    if (threads) *threads = NTHREADS;
    if (smem_bytes) *smem_bytes = c->smem_bytes;
    if (tile_rows) *tile_rows = c->geo.TR;
    if (ring_slots) *ring_slots = c->geo.S;
    if (tiles_per_slab) *tiles_per_slab = c->nt_max;
    return 0;
}

// launches the fused kernel for `nsteps` steps; trace (device) may be NULL
static int launch_fused(b200l_ctx *c, const int32_t *order_host, int64_t nsteps, double mu,
                        double err_bound, bool want_err, bool want_time, unsigned long long *trace_dev,
                        unsigned long long *ttrace_dev, bool timed) {
    if (nsteps > 0x7fff0000LL) return fail("nsteps=%lld is too large for one launch", (long long)nsteps);
    if (order_host) {
        for (int64_t i = 0; i < nsteps; ++i)
            if (order_host[i] < 0 || order_host[i] >= c->nblocks)
                return fail("order[%lld]=%d out of range", (long long)i, order_host[i]);
        if (c->order_cap < nsteps) {
            if (c->order) CK(cudaFree(c->order));
            c->order = nullptr;
            c->order_cap = 0;
            CK(cudaMalloc((void **)&c->order, (size_t)nsteps * 4));
            c->order_cap = nsteps;
        }
        CK(cudaMemcpyAsync(c->order, order_host, (size_t)nsteps * 4, cudaMemcpyHostToDevice, c->stream));
    }
    if ((want_err || want_time) && c->hist_cap < nsteps) {
        if (c->err_hist) CK(cudaFree(c->err_hist));
        if (c->time_hist) CK(cudaFree(c->time_hist));
        c->err_hist = nullptr;
        c->time_hist = nullptr;
        c->hist_cap = 0;
        CK(cudaMalloc((void **)&c->err_hist, (size_t)nsteps * 8));
        CK(cudaMalloc((void **)&c->time_hist, (size_t)nsteps * 8));
        c->hist_cap = nsteps;
    }
    if (want_err) CK(cudaMemsetAsync(c->err_hist, 0, (size_t)nsteps * 8, c->stream));
    if (want_time) CK(cudaMemsetAsync(c->time_hist, 0, (size_t)nsteps * 8, c->stream));
    // tags tag_base+1 .. tag_base+nsteps+1 are consumed by this launch; never reuse one
    if ((uint64_t)c->tag_base + (uint64_t)nsteps + 2 >= 0xffffffffULL) {
        CK(cudaMemsetAsync(c->gLL, 0, c->gLL_bytes, c->stream));
        CK(cudaMemsetAsync(c->dLL, 0, (size_t)(c->xld + 2 * GMAX + 2) * 16, c->stream));
        CK(cudaMemsetAsync(c->sLL, 0, (size_t)GMAX * 4 * 16, c->stream));
        c->tag_base = 0;
    }

    RunParams p = c->geo;
    p.A = c->A;
    p.N = c->N;
    p.blk_stride = c->brows * c->ld;
    p.w = c->w;
    p.ld = c->layout == B200L_TRANSPOSED ? (int32_t)c->xld : (int32_t)c->ld;
    p.nblocks = c->nblocks;
    p.x = c->x; p.d = c->d; p.drec = c->drec; p.r = c->r;
    p.gLL = c->gLL; p.dLL = c->dLL; p.sLL = c->sLL; p.abort_flag = c->abort_flag;
    p.order = order_host ? c->order : nullptr;
    p.nsteps = nsteps;
    p.step0 = c->step_counter;
    p.mu = mu;
    p.err_bound = err_bound;
    p.bounded = err_bound >= 0.0 ? 1 : 0;
    p.err_hist = want_err ? c->err_hist : nullptr;
    p.time_hist = want_time ? c->time_hist : nullptr;
    p.state = c->state;
    p.gamma_state = c->gamma_state;
    p.trace = trace_dev;
    p.ttrace = ttrace_dev;
    p.tag_base = c->tag_base;
    p.wait_limit_ns = c->wait_limit_ns;
    p.world = c->world;
    p.rank = c->rank;
    p.qw = c->world > 1 ? (int32_t)round_up(c->geo.rows_max_ + 2, 2) : 0;
    for (int r = 0; r < B200L_MAX_WORLD; ++r) p.peer[r] = c->peer[r];
    p.mc = c->world > 1 ? c->mc : nullptr;

    if (c->world > 1)
        for (int r = 0; r < c->world; ++r)
            if (!c->peer[r])
                return fail("multi-GPU run: the inbox of rank %d is not mapped (b200l_comm_connect has not "
                            "completed on this context)", r);
    if (c->layout == B200L_TRANSPOSED && !c->tmap_valid && make_tensor_map(c)) return 1;
    p.dbg = c->dbg & DBG_KNOCKOUTS;
    const bool diag = trace_dev != nullptr || ttrace_dev != nullptr || p.dbg != 0;
    fused_fn fn = ctx_kernel(c, diag ? 2 : (c->world > 1 ? 1 : 0));
    void *args[] = {(void *)&p, (void *)&c->tmap};
    if (timed) CK(cudaEventRecord(c->ev0, c->stream));
    CK(cudaLaunchCooperativeKernel((const void *)fn, dim3(c->grid), dim3(NTHREADS), args,
                                   (size_t)c->smem_bytes, c->stream));
    if (timed) CK(cudaEventRecord(c->ev1, c->stream));
    c->step_counter += nsteps;
    c->tag_base += (uint32_t)nsteps + 2u;
    return 0;
}

// reads back the launch status; fails when the kernel abandoned a cross-CTA wait
static int finish_fused(b200l_ctx *c, int64_t *steps_done, int32_t *stopped, double *kernel_ms) {
    long long st[8];
    CK(cudaMemcpyAsync(st, c->state, sizeof(st), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (st[3]) {
        CK(cudaMemsetAsync(c->abort_flag, 0, 64, c->stream));
        CK(cudaMemsetAsync(c->state, 0, 64, c->stream));
        return fail("fused kernel aborted: a cross-CTA wait exceeded %.1f s (CTA %lld thread %lld step %lld %s word "
                    "%lld; solver state is invalid; call b200l_reset)", (double)c->wait_limit_ns * 1e-9, st[4],
                    st[5], st[6] >> 32, (st[6] & 0x80000000LL) ? "step-D" : "inbox", st[6] & 0x7fffffffLL);
    }
    if (steps_done) *steps_done = st[0];
    if (stopped) *stopped = (int32_t)st[1];
    if (kernel_ms) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        *kernel_ms = (double)ms;
    }
    return 0;
}

extern "C" int b200l_run(b200l_ctx *c, const int32_t *order_host, int64_t nsteps, double mu,
                         double err_bound, double *err_hist_host, double *time_hist_host,
                         int64_t *steps_done, int32_t *stopped, double *kernel_ms) {
    if (need_A(c)) return 1;
    if (!c->have_problem) return fail("b200l_set_problem has not been called");
    if (nsteps < 0) return fail("nsteps < 0");
    if (plan_geometry(c)) return 1;
    if (nsteps == 0) {
        if (steps_done) *steps_done = 0;
        if (stopped) *stopped = 0;
        if (kernel_ms) *kernel_ms = 0.0;
        return 0;
    }
    if (launch_fused(c, order_host, nsteps, mu, err_bound, err_hist_host != nullptr,
                     time_hist_host != nullptr, nullptr, nullptr, kernel_ms != nullptr))
        return 1;
    const bool want_sync = steps_done || stopped || kernel_ms || err_hist_host || time_hist_host;
    if (!want_sync) return 0;

    std::vector<unsigned long long> tbuf;
    if (err_hist_host)
        CK(cudaMemcpyAsync(err_hist_host, c->err_hist, (size_t)nsteps * 8, cudaMemcpyDeviceToHost, c->stream));
    if (time_hist_host) {
        tbuf.resize((size_t)nsteps);
        CK(cudaMemcpyAsync(tbuf.data(), c->time_hist, (size_t)nsteps * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    if (finish_fused(c, steps_done, stopped, kernel_ms)) return 1;
    if (time_hist_host)
        for (int64_t i = 0; i < nsteps; ++i) time_hist_host[i] = (double)tbuf[(size_t)i] * 1e-9;
    return 0;
}

extern "C" int b200l_run_traced(b200l_ctx *c, int64_t nsteps, double mu, uint64_t *trace_host,
                                uint64_t *tile_trace_host, int32_t *grid_out, double *kernel_ms) {
    if (need_A(c)) return 1;
    if (!c->have_problem) return fail("b200l_set_problem has not been called");
    if (nsteps <= 0 || !trace_host) return fail("nsteps must be positive and trace_host non-NULL");
    if (plan_geometry(c)) return 1;
    const int64_t words = (int64_t)c->grid * nsteps * NTRACE;
    if (c->trace_cap < words) {
        if (c->trace) CK(cudaFree(c->trace));
        c->trace = nullptr;
        c->trace_cap = 0;
        CK(cudaMalloc((void **)&c->trace, (size_t)words * 8));
        c->trace_cap = words;
    }
    CK(cudaMemsetAsync(c->trace, 0, (size_t)words * 8, c->stream));
    const int64_t twords = (int64_t)c->grid * nsteps * NTTRACE;
    if (tile_trace_host) {
        if (c->ttrace_cap < twords) {
            if (c->ttrace) CK(cudaFree(c->ttrace));
            c->ttrace = nullptr;
            c->ttrace_cap = 0;
            CK(cudaMalloc((void **)&c->ttrace, (size_t)twords * 8));
            c->ttrace_cap = twords;
        }
        CK(cudaMemsetAsync(c->ttrace, 0, (size_t)twords * 8, c->stream));
    }
    if (launch_fused(c, nullptr, nsteps, mu, -1.0, false, false, c->trace,
                     tile_trace_host ? c->ttrace : nullptr, true))
        return 1;
    CK(cudaMemcpyAsync(trace_host, c->trace, (size_t)words * 8, cudaMemcpyDeviceToHost, c->stream));
    if (tile_trace_host)
        CK(cudaMemcpyAsync(tile_trace_host, c->ttrace, (size_t)twords * 8, cudaMemcpyDeviceToHost, c->stream));
    if (finish_fused(c, nullptr, nullptr, kernel_ms)) return 1;
    if (grid_out) *grid_out = c->grid;
    return 0;
}

extern "C" int b200l_set_wait_limit(b200l_ctx *c, double seconds) {
    if (!c) return fail("ctx is NULL");
    if (!(seconds > 0.0)) return fail("wait limit must be positive");
    c->wait_limit_ns = (unsigned long long)(seconds * 1e9);
    return 0;
}

// diagnostics (see DBG_KNOCKOUTS, DBG_LOAD_BATCH)
extern "C" int b200l_debug_flags(b200l_ctx *c, int32_t flags) {
    if (!c) return fail("ctx is NULL");
    if (flags & ~(DBG_KNOCKOUTS | DBG_LOAD_BATCH))
        return fail("debug flags 0x%x: only bits 0-2 (1, 2, 4: knock-outs) and bit 18 (262144: load-batch "
                    "mat-vecs) are accepted", (unsigned)flags);
    c->dbg = flags;
    return 0;
}

// ------------------------------------------------------------------------------------
// multi-GPU: one process per GPU, column slice `rank` of every block per rank
// ------------------------------------------------------------------------------------
// Teardown in two steps, with a barrier over the ranks between them (distributed.disconnect):
// first every rank closes the peers' inboxes it had mapped, then it frees its own -- freeing an
// exported allocation that an importer still has open is undefined behaviour.
static int comm_close_peers(b200l_ctx *c) {
    for (int r = 0; r < B200L_MAX_WORLD; ++r) {
        if (!c->peer[r] || r == c->rank) continue;
        if (c->peer_ipc) cudaIpcCloseMemHandle(c->peer[r]);
        c->peer[r] = nullptr;
    }
    return 0;
}

static int comm_release(b200l_ctx *c) {
    comm_close_peers(c);
    if (c->world > 1 && c->peer[c->rank] && c->peer_ipc) cudaFree(c->peer[c->rank]);
    for (int r = 0; r < B200L_MAX_WORLD; ++r) c->peer[r] = nullptr;
    c->world = 1;
    c->rank = 0;
    c->inbox_bytes = 0;
    c->peer_ipc = 0;
    c->mc = nullptr;
    c->geo_valid = 0;
    return 0;
}

extern "C" int b200l_comm_export(b200l_ctx *c, int32_t rank, int32_t world, void *handle_out,
                                 int32_t handle_bytes) {
    if (!c || !handle_out) return fail("NULL argument");
    if (world < 2 || world > B200L_MAX_WORLD) return fail("world must be 2..%d", B200L_MAX_WORLD);
    if (rank < 0 || rank >= world) return fail("rank %d out of range", rank);
    if (handle_bytes < (int32_t)sizeof(cudaIpcMemHandle_t))
        return fail("handle buffer must hold %d bytes", (int)sizeof(cudaIpcMemHandle_t));
    CK(cudaSetDevice(c->device));
    comm_release(c);
    c->world = world;               // the shared-memory plan depends on it
    c->rank = rank;
    c->geo_valid = 0;
    if (plan_geometry(c)) { c->world = 1; c->rank = 0; c->geo_valid = 0; return 1; }
    const size_t qw = (size_t)round_up(c->geo.rows_max_ + 2, 2);
    const size_t bytes = 2 * (size_t)c->grid * world * qw * 16;
    ulonglong2 *buf = nullptr;
    CK(cudaMalloc((void **)&buf, bytes));
    CK(cudaMemset(buf, 0, bytes));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, buf));
    memcpy(handle_out, &h, sizeof(h));
    c->world = world;
    c->rank = rank;
    c->peer[rank] = buf;
    c->inbox_bytes = bytes;
    c->peer_ipc = 1;
    return 0;
}

extern "C" int b200l_comm_connect(b200l_ctx *c, const void *all_handles, int32_t handle_stride) {
    if (!c || !all_handles) return fail("NULL argument");
    if (c->world < 2 || !c->peer[c->rank]) return fail("b200l_comm_export has not been called");
    if (handle_stride < (int32_t)sizeof(cudaIpcMemHandle_t)) return fail("handle stride too small");
    CK(cudaSetDevice(c->device));
    for (int r = 0; r < c->world; ++r) {
        if (r == c->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)all_handles + (size_t)r * handle_stride, sizeof(h));
        void *ptr = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            comm_close_peers(c);      // what was mapped so far; the run refuses to start without all peers
            return fail("cudaIpcOpenMemHandle for rank %d failed: %s", r, cudaGetErrorString(e));
        }
        c->peer[r] = (ulonglong2 *)ptr;
    }
    return 0;
}

// first half of the teardown: unmap the peers' inboxes (collective: every rank, then a barrier,
// then b200l_comm_destroy)
extern "C" int b200l_comm_close_peers(b200l_ctx *c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    return comm_close_peers(c);
}

// number of words (16 bytes each) of one rank's inbox for the current shape and world size
extern "C" int b200l_comm_inbox_bytes(b200l_ctx *c, int32_t world, int64_t *bytes) {
    if (need_A(c) || !bytes) return c ? fail("bytes is NULL") : 1;
    if (world < 2 || world > B200L_MAX_WORLD) return fail("world must be 2..%d", B200L_MAX_WORLD);
    const int w0 = c->world, r0 = c->rank;
    c->world = world; c->geo_valid = 0;
    const int rc = plan_geometry(c);
    const size_t qw = (size_t)round_up(c->geo.rows_max_ + 2, 2);
    *bytes = rc ? 0 : (int64_t)(2 * (size_t)c->grid * world * qw * 16);
    c->world = w0; c->rank = r0; c->geo_valid = 0;
    return rc;
}

// inboxes allocated and mapped by the caller (e.g. torch symmetric memory): peer_ptrs[r] is the
// address, in THIS process, of rank r's inbox (b200l_comm_inbox_bytes bytes each, zero-filled);
// mc_ptr, when not NULL, is a multicast (NVLS) mapping of the same buffers: one multimem store
// then reaches every rank's inbox.  The caller keeps ownership of the memory.
extern "C" int b200l_comm_attach(b200l_ctx *c, int32_t rank, int32_t world, void *const *peer_ptrs, void *mc_ptr) {
    if (!c || !peer_ptrs) return fail("NULL argument");
    if (world < 2 || world > B200L_MAX_WORLD) return fail("world must be 2..%d", B200L_MAX_WORLD);
    if (rank < 0 || rank >= world) return fail("rank %d out of range", rank);
    CK(cudaSetDevice(c->device));
    comm_release(c);
    for (int r = 0; r < world; ++r)
        if (!peer_ptrs[r]) return fail("peer_ptrs[%d] is NULL", r);
    c->world = world;
    c->rank = rank;
    c->mc = (ulonglong2 *)mc_ptr;
    c->geo_valid = 0;
    if (plan_geometry(c)) { c->world = 1; c->rank = 0; c->mc = nullptr; c->geo_valid = 0; return 1; }
    for (int r = 0; r < world; ++r) c->peer[r] = (ulonglong2 *)peer_ptrs[r];
    c->peer_ipc = 0;
    const size_t qw = (size_t)round_up(c->geo.rows_max_ + 2, 2);
    c->inbox_bytes = 2 * (size_t)c->grid * world * qw * 16;
    return 0;
}

extern "C" int b200l_comm_destroy(b200l_ctx *c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    return comm_release(c);
}
