// zkm_common.cuh -- process-wide context, error plumbing and launch helpers shared by the
// NTT and MSM translation units.  Host-side C++ only wraps CUDA: there is no CPU compute path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>
#include <condition_variable>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/zkm_b200.h"
#include "zkm_curve.cuh"

namespace zkm {

void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

struct ZkmError {
    int32_t code;
};

#define ZKM_CUDA(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            ::zkm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            throw ::zkm::ZkmError{_e == cudaErrorMemoryAllocation ? ZKM_ERR_OOM : ZKM_ERR_CUDA};          \
        }                                                                                     \
    } while (0)

#define ZKM_FAIL(code, ...)              \
    do {                                 \
        ::zkm::set_error(__VA_ARGS__);   \
        throw ::zkm::ZkmError{code};     \
    } while (0)

// count + launch-check in one place
#define ZKM_LAUNCH(kernel, grid, block, smem, stream, ...)                   \
    do {                                                                     \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);          \
        ::zkm::g_launches.fetch_add(1, std::memory_order_relaxed);           \
        ZKM_CUDA(cudaGetLastError());                                        \
    } while (0)

// A growable device buffer (never shrinks; freed at shutdown).  Growth is STREAM-ORDERED (cudaFreeAsync + cudaMallocAsync
// on the stream of the call in progress, from the device's default memory pool, whose release threshold zkm_init* raises
// so that freed blocks stay with the process): no device-wide synchronisation.  The plain cudaFree + cudaMalloc it
// replaces stalls every stream of the GPU -- with asynchronous MSMs on 48 lanes a lane that met a larger shape for the
// first time (a G2 MSM on a lane that had only run G1) froze all proofs in flight for milliseconds (measured r2m:
// 4 proofs in flight 13-20 ms per proof against 3.3 ms with 2).
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaStream_t* cur = nullptr;    // -> Context::cur_stream of the owning lane (nullptr: legacy default stream)
    void* get(size_t bytes) {
        if (bytes > cap) {
            cudaStream_t s = cur ? *cur : nullptr;
            if (p) ZKM_CUDA(cudaFreeAsync(p, s));   // ordered after everything the lane has enqueued so far
            p = nullptr;
            cap = 0;
            size_t want = bytes + (bytes >> 3) + 256;
            cudaError_t e = cudaMallocAsync(&p, want, s);
            if (e == cudaErrorMemoryAllocation) {
                // the pool keeps freed blocks (fragmentation, blocks still owed to other streams): hand everything that is
                // really free back to the device and try once more before reporting ZKM_ERR_OOM
                cudaGetLastError();
                p = nullptr;
                trim_pool();
                e = cudaMallocAsync(&p, want, s);
            }
            if (e != cudaSuccess) {
                p = nullptr;
                ZKM_CUDA(e);
            }
            cap = want;
        }
        return p;
    }
    template <class T>
    T* as(size_t count) { return reinterpret_cast<T*>(get(count * sizeof(T))); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    // synchronise the current device and release the unused memory of its default pool
    static void trim_pool() {
        int dev = 0;
        cudaMemPool_t pool;
        cudaDeviceSynchronize();
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
        cudaGetLastError();
    }
};

// cudaMalloc for the long-lived allocations (registered bases, tables): if the device is full because the default pool is
// holding freed workspace blocks, trim the pool and try once more
inline cudaError_t malloc_retry(void** p, size_t bytes) {
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        DevBuf::trim_pool();
        e = cudaMalloc(p, bytes);
    }
    return e;
}

struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    void* get(size_t bytes) {
        if (bytes > cap) {
            if (p) ZKM_CUDA(cudaFreeHost(p));
            p = nullptr;
            cap = 0;
            ZKM_CUDA(cudaMallocHost(&p, bytes + 256));
            cap = bytes + 256;
        }
        return p;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// One contiguous run of registered bases living on one device.
struct BasesPart {
    int dev = 0;              // index into the initialised device list (0 = primary)
    int ordinal = 0;          // CUDA ordinal of that device (needed to free the memory after shutdown)
    size_t first = 0, n = 0;  // bases [first, first + n) of the registration
    void* d_xy = nullptr;     // n affine records, 2 * W * 8 bytes each
    uint8_t* d_inf = nullptr; // n flags or nullptr
    // optional window multiples (ZKM_REG_PRECOMPUTE): table[w * n + i] = 2^(pre_c w) P_i
    void* d_table = nullptr;
    int pre_c = 0, pre_W = 0;
};
// A registration: one part (the usual case), or one part per device when registered with ZKM_REG_SHARD.
// Held by shared_ptr: zkm_bases_release drops the registry's reference, the memory goes when the last
// call that looked the handle up has finished.
struct BasesReg {
    int curve = 0, group = 0;
    size_t n = 0;
    std::vector<BasesPart> parts;
    size_t bytes = 0;         // device bytes held (registration cache accounting)
    ~BasesReg();
};

struct Options {
    int msm_window_bits = 0;
    int msm_chunk = 0;
    int ntt_max_radix_log = 12;
    int profile = 0;  // record CUDA events at the MSM stage boundaries
    int msm_precompute = 0;  // legacy switch: registrations made while set behave as if ZKM_REG_PRECOMPUTE was passed
    int msm_affine_levels = -1;  // batched-affine pairwise levels before the XYZZ tasks (-1 = automatic)
    int msm_pair_m = 64, msm_pair_m2 = 32;  // outputs per thread / totals per inversion thread in the pair levels
    // L2 prefetch distance of the level-0 gathers: measured SLOWER in round 1 (+10 ms each at 2^24: the passes are bound by
    // random-access DRAM throughput, not latency); the prefetch code is gone, the options are accepted and ignored.
    int msm_prefetch_fwd = 0, msm_prefetch_bwd = 0;
    int msm_xarr = 1;            // level-0 forward pass gathers x from an array of 64-byte slots (48-byte coordinates)
    int msm_fold = 0;            // (round 1: fan-in of the host-sized fold levels) accepted and ignored: see k_fold_*
    // zkm_msm_g1 / zkm_msm_g2 (the literal multi_scalar_mul(bases, scalars) signature): keep the uploaded bases as an
    // internal registration keyed by (host pointer, n, content fingerprint).  0 = off, 1 = fingerprint of 512 sampled
    // records (default: proving keys / SRS are immutable while a prover runs), 2 = fingerprint of every byte.
    int msm_cache = 1;
    int64_t msm_cache_max_mb = 32768;   // cached registrations are evicted least-recently-used above this
    int msm_cache_precompute = 1;       // cached vectors of <= 2^18 bases get window multiples when they come back
    int spread_host_calls = 0;   // host-pointer NTT / witness-map calls rotate over the initialised devices
    // (round 1: how a call waited for its one device read-back) accepted and ignored: an MSM has no read-back any more
    int host_wait = 0;
};

// State of one initialised device.
struct Shared {
    int device = -1;                       // CUDA ordinal
    int index = 0;                         // position in the initialised device list
    int sm_count = 148;
    // The stream behind `stream == NULL` of the *_device entry points: ONE library-owned non-blocking stream per device,
    // so that successive NULL-stream calls stay ordered among themselves whichever lanes they borrow.
    cudaStream_t null_stream = nullptr;
    std::mutex tw_mu;                      // guards `twiddles`
    std::map<uint64_t, void*> twiddles;    // key -> device table (twiddles, coset powers, domain constants)
};

// A lane = one stream + one set of workspaces on one device.  Every compute call borrows a free lane for its
// duration, so independent calls from different host threads (e.g. the five MSMs of a Groth16 proof, the G2 MSM next
// to the G1 ones) run concurrently on the GPU instead of queueing behind one another's serial tails.
struct Context {
    Shared* sh;
    int& device;
    int& sm_count;
    Options opt;                           // snapshot taken when the lane was acquired: stable for the whole call
    std::map<uint64_t, void*>& twiddles;
    explicit Context(Shared* s) : sh(s), device(s->device), sm_count(s->sm_count), twiddles(s->twiddles) {
        DevBuf* all[] = {&ntt_a, &ntt_b, &io_scalars, &io_bases, &io_inf, &io_out, &gather};
        for (DevBuf* b : all) b->cur = &cur_stream;
        for (DevBuf& b : ws) b.cur = &cur_stream;
    }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    cudaStream_t cur_stream = nullptr;     // stream of the call in progress (StreamScope); the lane's own stream otherwise
    int lane_id = 0;
    bool busy = false;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;
    DevBuf ntt_a, ntt_b;
    DevBuf ws[40];
    DevBuf io_scalars, io_bases, io_inf, io_out;
    DevBuf gather;                         // partial result records of a sharded MSM, summed on this (home) device
    PinnedBuf pin_in, pin_out;
    // stage timing of the last MSM on this lane (opt.profile): events at the boundaries of
    // sort | affine pair levels | task lists | bucket accumulation | fold levels | window reduction
    cudaEvent_t pev[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool pev_valid = false;
    // work counters of the last profiled MSM (device words read back after the run): see zkm_profile_last_msm_counts
    uint64_t pcount[16] = {0};
    // The lane's workspaces may still be in use by kernels enqueued on the stream of its previous borrower:
    // every call orders itself after `done_ev` and re-records it when it has enqueued its work.
    cudaEvent_t done_ev = nullptr;
    cudaEvent_t feed_ev[9] = {nullptr};   // chunked scalar upload of the host entry points (see ScalarFeed); [8]: start marker
    cudaStream_t last_stream = nullptr;   // stream of the lane's previous call (lane selection: see pick_free_lane)
    uint64_t affinity = 0;                // job key of the lane's previous call (same key -> same workspace sizes)
    void begin(cudaStream_t s) {
        if (done_ev) ZKM_CUDA(cudaStreamWaitEvent(s, done_ev, 0));
        last_stream = s;
        cur_stream = s;
    }
    void end(cudaStream_t s) {
        if (!done_ev) ZKM_CUDA(cudaEventCreateWithFlags(&done_ev, cudaEventDisableTiming));
        ZKM_CUDA(cudaEventRecord(done_ev, s));
    }
};
// begin()/end() bracket of a call that enqueues on `s`: end() also runs when the call throws after kernels were
// queued (otherwise the next borrower of the lane could overwrite workspaces that are still in use); if even
// recording the event fails the stream is drained instead.
struct StreamScope {
    Context* c;
    cudaStream_t s;
    StreamScope(Context* c_, cudaStream_t s_) : c(c_), s(s_) { c->begin(s); }
    ~StreamScope() {
        try {
            c->end(s);
        } catch (...) {
            cudaStreamSynchronize(s);
            cudaGetLastError();
        }
    }
    StreamScope(const StreamScope&) = delete;
    StreamScope& operator=(const StreamScope&) = delete;
};

constexpr int ZKM_NUM_LANES = 48;
// blocks until a lane of device index `dev` is free; throws ZKM_ERR_NOT_INIT before zkm_init.  `hint`: the stream the
// call is going to enqueue on, if it is the caller's (a lane last used on that stream is preferred)
Context* acquire_lane(int dev = 0, cudaStream_t hint = nullptr, uint64_t key = 0);   // key: lane affinity (see pick_free_lane)
void release_lane(Context* c);
int device_count_initialised();
struct LaneGuard {
    Context* c;
    explicit LaneGuard(int dev = 0, cudaStream_t hint = nullptr, uint64_t key = 0) : c(acquire_lane(dev, hint, key)) {}
    ~LaneGuard() { release_lane(c); }
    LaneGuard(const LaneGuard&) = delete;
    LaneGuard& operator=(const LaneGuard&) = delete;
};

// Several lanes at once, all or nothing: a call that needs a lane per job never holds some while waiting for others,
// so concurrent multi-lane calls cannot deadlock each other.  devs[i] = device index of lane i.
std::vector<Context*> acquire_lanes(const std::vector<int>& devs, cudaStream_t hint0 = nullptr,
                                    const std::vector<uint64_t>* keys = nullptr);   // hint0: for devs[0]; keys[i]: affinity of lane i
struct MultiLaneGuard {
    std::vector<Context*> c;
    explicit MultiLaneGuard(const std::vector<int>& devs, cudaStream_t hint0 = nullptr, const std::vector<uint64_t>* keys = nullptr)
        : c(acquire_lanes(devs, hint0, keys)) {}
    ~MultiLaneGuard() { for (Context* x : c) release_lane(x); }
    MultiLaneGuard(const MultiLaneGuard&) = delete;
    MultiLaneGuard& operator=(const MultiLaneGuard&) = delete;
};

Context* ctx();            // lane 0 (non-compute queries); throws ZKM_ERR_NOT_INIT when zkm_init has not succeeded
inline bool curve_known(int curve) {
    return curve == ZKM_CURVE_BLS12_381 || curve == ZKM_CURVE_BN254 || curve == ZKM_CURVE_BW6_761;
}
// u64 words per coordinate: Fq for G1, Fq2 for G2 -- except BW6-761, whose G2 is a curve over Fq as well
inline int coord_words(int curve, int group) {
    if (curve == ZKM_CURVE_BW6_761) return 12;
    return (curve == ZKM_CURVE_BLS12_381 ? 6 : 4) * (group == 2 ? 2 : 1);
}
// u64 words of a scalar-field element / canonical scalar: BigInteger256, or BigInteger384 for BW6-761
inline int fr_words(int curve) { return curve == ZKM_CURVE_BW6_761 ? 6 : 4; }
inline int fr_two_adicity(int curve) { return curve == ZKM_CURVE_BLS12_381 ? 32 : (curve == ZKM_CURVE_BN254 ? 28 : 46); }
inline int fr_bits(int curve) { return curve == ZKM_CURVE_BLS12_381 ? 255 : (curve == ZKM_CURVE_BN254 ? 254 : 377); }

// entry points implemented by the two compute translation units
void ntt_run(Context* c, int curve, const uint64_t* d_in, uint64_t* d_out, uint32_t log_n, int inverse, int coset,
             cudaStream_t stream);
void ntt_domain_constants(Context* c, int curve, uint32_t log_n, uint64_t* out5x4_host);
void ntt_release_tables(Shared* sh);
void fr_into_repr_run(Context* c, int curve, const uint64_t* d_in, uint64_t* d_out, uint64_t n, cudaStream_t stream);
void witness_map_run(Context* c, int curve, uint64_t* d_a, uint64_t* d_b, uint64_t* d_c, uint32_t log_n, uint64_t* d_h,
                     cudaStream_t stream);
// Scalars that are still arriving in device memory: the caller copies them in `n` chunks on another stream, chunk i
// (scalars [begin[i], begin[i + 1])) is complete when ev[i] has fired.  msm_run then runs its histogram pass chunk by chunk
// behind the copies (everything after it needs all scalars).
struct ScalarFeed {
    int n = 0;
    size_t begin[9] = {0};
    cudaEvent_t ev[8] = {nullptr};
};
void msm_run(Context* c, int curve, int group, const void* d_bases, const uint8_t* d_inf, const uint64_t* d_scalars,
             size_t n, uint64_t* d_out, cudaStream_t stream, const BasesPart* pre = nullptr, size_t pre_offset = 0,
             const ScalarFeed* feed = nullptr);
void msm_precompute(Context* c, int curve, int group, BasesPart* part, cudaStream_t stream);
void kzg_quotient_run(Context* c, int curve, const uint64_t* d_coeffs, size_t n, const uint64_t* d_point, uint64_t* d_quot,
                      uint64_t* d_eval, cudaStream_t stream);
void points_sum_run(Context* c, int curve, int group, const uint64_t* d_points, size_t m, uint64_t* d_out,
                    cudaStream_t stream);
void testgen_progression(Context* c, int curve, int group, uint64_t a0, uint64_t d, size_t n, uint64_t* d_out,
                         cudaStream_t stream);
int msm_auto_window_bits(int curve, int group, size_t n);
// out[i] = s_i * base (zkm_fixed_base.cuh); base_xy: host record; d_flag: null or a zeroed device word (bit 0: s_i >= r)
void fixed_base_run(Context* c, int curve, int group, const uint64_t* base_xy, bool base_inf, const uint64_t* d_scalars, size_t n,
                    uint64_t* d_out_xy, uint8_t* d_out_inf, uint32_t* d_flag, cudaStream_t stream);
void note_profiled_lane(Context* c);   // zkm_profile_last_msm* report the lane that ran the last profiled MSM

// 128-bit vectorised global access for field elements (N is a multiple of 4 limbs)
template <class P>
__device__ __forceinline__ Fp<P> ld_fp(const void* p) {
    Fp<P> r;
    const uint4* q = reinterpret_cast<const uint4*>(p);
#pragma unroll
    for (int i = 0; i < P::N / 4; i++) {
        uint4 v = __ldg(q + i);
        r.l[4 * i] = v.x; r.l[4 * i + 1] = v.y; r.l[4 * i + 2] = v.z; r.l[4 * i + 3] = v.w;
    }
    return r;
}
// Random gathers of whole base records: ask L2 for 64-byte fills instead of the default 128-byte lines
// (a 96-byte record at a random 32-byte-aligned address otherwise drags in 192 bytes on average).
template <class P>
__device__ __forceinline__ Fp<P> ld_fp_gather(const void* p) {
    Fp<P> r;
    const uint4* q = reinterpret_cast<const uint4*>(p);
#pragma unroll
    for (int i = 0; i < P::N / 4; i++) {
        uint4 v;
        asm volatile("ld.global.nc.L2::64B.v4.u32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                     : "l"(q + i));
        r.l[4 * i] = v.x; r.l[4 * i + 1] = v.y; r.l[4 * i + 2] = v.z; r.l[4 * i + 3] = v.w;
    }
    return r;
}
template <class P>
__device__ __forceinline__ Fp<P> ld_fp_plain(const void* p) {  // coherent load (data written earlier in the same kernel)
    Fp<P> r;
    const uint4* q = reinterpret_cast<const uint4*>(p);
#pragma unroll
    for (int i = 0; i < P::N / 4; i++) {
        uint4 v = q[i];
        r.l[4 * i] = v.x; r.l[4 * i + 1] = v.y; r.l[4 * i + 2] = v.z; r.l[4 * i + 3] = v.w;
    }
    return r;
}
template <class P>
__device__ __forceinline__ void st_fp(void* p, const Fp<P>& a) {
    uint4* q = reinterpret_cast<uint4*>(p);
#pragma unroll
    for (int i = 0; i < P::N / 4; i++) q[i] = make_uint4(a.l[4 * i], a.l[4 * i + 1], a.l[4 * i + 2], a.l[4 * i + 3]);
}

// generic coordinate (Fp or Fp2) access
template <class F> struct CoordIO;
template <class P> struct CoordIO<Fp<P>> {
    static constexpr int BYTES = P::N * 4;
    static __device__ __forceinline__ Fp<P> ld(const void* p) { return ld_fp<P>(p); }
    static __device__ __forceinline__ Fp<P> ld_plain(const void* p) { return ld_fp_plain<P>(p); }
    static __device__ __forceinline__ Fp<P> ld_gather(const void* p) { return ld_fp_gather<P>(p); }
    static __device__ __forceinline__ void st(void* p, const Fp<P>& a) { st_fp<P>(p, a); }
};
template <class P> struct CoordIO<Fp2<P>> {
    static constexpr int BYTES = P::N * 8;
    static __device__ __forceinline__ Fp2<P> ld(const void* p) {
        Fp2<P> r;
        r.c0 = ld_fp<P>(p);
        r.c1 = ld_fp<P>(reinterpret_cast<const char*>(p) + P::N * 4);
        return r;
    }
    static __device__ __forceinline__ Fp2<P> ld_gather(const void* p) {
        Fp2<P> r;
        r.c0 = ld_fp_gather<P>(p);
        r.c1 = ld_fp_gather<P>(reinterpret_cast<const char*>(p) + P::N * 4);
        return r;
    }
    static __device__ __forceinline__ Fp2<P> ld_plain(const void* p) {
        Fp2<P> r;
        r.c0 = ld_fp_plain<P>(p);
        r.c1 = ld_fp_plain<P>(reinterpret_cast<const char*>(p) + P::N * 4);
        return r;
    }
    static __device__ __forceinline__ void st(void* p, const Fp2<P>& a) {
        st_fp<P>(p, a.c0);
        st_fp<P>(reinterpret_cast<char*>(p) + P::N * 4, a.c1);
    }
};

}  // namespace zkm
