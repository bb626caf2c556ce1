// zkm_api.cu -- the C ABI of include/zkm_b200.h: devices, lanes, registrations, error reporting, host<->device
// staging and the multi-GPU orchestration of one process.  Every compute call ends in the CUDA kernels of
// zkm_ntt*.cu / zkm_msm*.cu; there is no CPU path.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <thread>

#include "zkm_common.cuh"
#include "zkm_groth16_ops.cuh"

namespace zkm {

static thread_local char t_err[512] = "";
std::atomic<uint64_t> g_launches{0};

// A Groth16 proving key (zkm_groth16_pk_create): references to the five query registrations, the key's eight points
// as records and the window tables of delta_g1 / delta_g2, on every initialised device (a proof runs where its
// output lives).
struct G16Key {
    int curve = 0;
    size_t m = 0;                                 // num_inputs + num_aux = len(a_query) - 1
    std::shared_ptr<BasesReg> reg[5];             // h, l, a[1..], b_g1[1..], b_g2[1..]
    bool delta1_inf = false, delta2_inf = false;
    struct Dev {
        int ordinal = -1;
        uint64_t* d_key = nullptr;                // 5 G1 records, then 3 G2 records
        char* d_tab1 = nullptr;
        char* d_tab2 = nullptr;
    };
    std::vector<Dev> dev;                         // by device index
    ~G16Key() {
        int cur = -1;
        cudaGetDevice(&cur);
        for (Dev& d : dev) {
            if (d.ordinal < 0 || cudaSetDevice(d.ordinal) != cudaSuccess) { cudaGetLastError(); continue; }
            // no proof may still be reading the key: the same drain as ~BasesReg (cudaFree would synchronise anyway)
            cudaDeviceSynchronize();
            if (d.d_key) cudaFree(d.d_key);
            if (d.d_tab1) cudaFree(d.d_tab1);
            if (d.d_tab2) cudaFree(d.d_tab2);
            cudaGetLastError();
        }
        if (cur >= 0) cudaSetDevice(cur);
        cudaGetLastError();
    }
};

// Process-wide state: the initialised devices (index 0 = primary), their lanes, options, registrations.
struct Global {
    std::vector<Shared*> devs;
    std::vector<std::vector<Context*>> lanes;     // lanes[dev index]
    std::vector<int> ordinals;                    // the list zkm_init* was given (repeats = virtual shards for tests)
    Options opt;
    std::mutex reg_mu;                            // guards `bases` / `next_handle`
    std::map<uint64_t, std::shared_ptr<BasesReg>> bases;
    std::map<uint64_t, std::shared_ptr<G16Key>> pks;   // Groth16 proving keys (same handle counter)
    uint64_t next_handle = 1;
    // registration cache of the literal multi_scalar_mul(bases, scalars) call (zkm_msm_g1 / zkm_msm_g2)
    struct CacheKey {
        int curve, group;
        const void* ptr;
        const void* inf;
        size_t n;
        bool operator<(const CacheKey& o) const {
            if (curve != o.curve) return curve < o.curve;
            if (group != o.group) return group < o.group;
            if (ptr != o.ptr) return ptr < o.ptr;
            if (inf != o.inf) return inf < o.inf;
            return n < o.n;
        }
    };
    struct CacheEntry {
        std::shared_ptr<BasesReg> reg;
        uint64_t fingerprint;
        uint64_t last_use;
        uint64_t hits = 0;
    };
    std::mutex cache_mu;
    std::map<CacheKey, CacheEntry> cache;
    uint64_t cache_clock = 0, cache_hits = 0, cache_misses = 0;
    size_t cache_bytes = 0;
    std::atomic<Context*> last_prof{nullptr};     // lane of the last profiled MSM
    std::atomic<uint32_t> rr{0};                  // round robin of host-pointer transform calls
};
static Global* g = nullptr;
static std::mutex g_init_mu;
static std::mutex g_lane_mu;                      // guards lane busy flags AND g->opt
static std::condition_variable g_lane_cv;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
}

BasesReg::~BasesReg() {
    // no lane may still be reading the bases: drain the owning device before its memory goes
    for (BasesPart& p : parts) {
        if (!p.d_xy && !p.d_inf && !p.d_table) continue;
        if (cudaSetDevice(p.ordinal) != cudaSuccess) { cudaGetLastError(); continue; }
        cudaDeviceSynchronize();
        if (p.d_xy) cudaFree(p.d_xy);
        if (p.d_inf) cudaFree(p.d_inf);
        if (p.d_table) cudaFree(p.d_table);
        cudaGetLastError();
    }
}

Context* ctx() {
    std::lock_guard<std::mutex> lk(g_lane_mu);
    if (!g || g->lanes.empty()) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    return g->lanes[0][0];
}

int device_count_initialised() {
    std::lock_guard<std::mutex> lk(g_lane_mu);
    return g ? (int)g->devs.size() : 0;
}

// Which free lane of device index `dev` a call gets (g_lane_mu held).  A lane is "free" as soon as the host call that
// borrowed it has RETURNED -- its GPU work may still be running (MSMs are fully asynchronous), and the next borrower's
// stream is ordered after it (done_ev: the workspaces are shared).  Always handing out the first free lane would chain
// independent calls behind one another on the GPU (measured: two proofs in flight no faster than one); rotating over
// all lanes would allocate workspaces on every one of them (a 2^24-point MSM holds ~20 GB per lane).  So, in order:
//   1. the lowest lane whose previous work ran on the caller's own stream (stream order already serialises the two
//      calls: no new dependency, no new memory -- the sequential caller stays on one lane);
//   2. the lowest lane whose previous work has finished;
//   3. otherwise the free lanes in turn (the call then waits for that lane's previous work on the GPU).
static Context* pick_free_lane(int dev, cudaStream_t hint, uint64_t key = 0) {
    static unsigned cursor[64] = {0};
    auto& v = g->lanes[dev];
    const size_t L = v.size();
    if (hint)
        for (Context* c : v)
            if (!c->busy && c->last_stream == hint) return c;
    // among the lanes whose previous work has finished: one that last served the same job (`key`: the same registered
    // bases and size class -> its workspaces already have the right sizes, no reallocation), else the lowest
    auto idle = [](Context* c) { return !c->done_ev || cudaEventQuery(c->done_ev) == cudaSuccess; };
    Context* pick = nullptr;
    if (key)
        for (Context* c : v)
            if (!c->busy && c->affinity == key && idle(c)) {
                pick = c;
                break;
            }
    if (!pick && key)       // a lane nobody has a claim on, before taking over one that serves another job
        for (Context* c : v)
            if (!c->busy && c->affinity == 0 && idle(c)) {
                pick = c;
                break;
            }
    if (!pick)
        for (Context* c : v)
            if (!c->busy && idle(c)) {
                pick = c;
                break;
            }
    cudaGetLastError();   // cudaErrorNotReady from the queries is not an error
    if (pick) {
        pick->affinity = key;
        return pick;
    }
    unsigned& cur = cursor[dev & 63];
    for (size_t k = 0; k < L; k++) {
        Context* c = v[(cur + k) % L];
        if (!c->busy) {
            cur = (unsigned)((cur + k + 1) % L);
            c->affinity = key;
            return c;
        }
    }
    return nullptr;
}

Context* acquire_lane(int dev, cudaStream_t hint, uint64_t key) {
    std::unique_lock<std::mutex> lk(g_lane_mu);
    if (!g || g->lanes.empty()) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    if (dev < 0 || dev >= (int)g->lanes.size()) ZKM_FAIL(ZKM_ERR_ARG, "device index %d out of range (%zu initialised)", dev, g->lanes.size());
    for (;;) {
        if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "library was shut down");
        if (Context* c = pick_free_lane(dev, hint, key)) {
            c->busy = true;
            c->opt = g->opt;      // snapshot: stable for the whole call whatever zkm_set_option does meanwhile
            c->cur_stream = c->stream;
            return c;
        }
        g_lane_cv.wait(lk);
    }
}

std::vector<Context*> acquire_lanes(const std::vector<int>& devs, cudaStream_t hint0, const std::vector<uint64_t>* keys) {
    std::unique_lock<std::mutex> lk(g_lane_mu);
    if (!g || g->lanes.empty()) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    std::vector<int> need(g->lanes.size(), 0);
    for (int d : devs) {
        if (d < 0 || d >= (int)g->lanes.size()) ZKM_FAIL(ZKM_ERR_ARG, "device index %d out of range (%zu initialised)", d, g->lanes.size());
        if (++need[d] > ZKM_NUM_LANES) ZKM_FAIL(ZKM_ERR_ARG, "a single call needs more than %d lanes on device index %d", ZKM_NUM_LANES, d);
    }
    for (;;) {
        if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "library was shut down");
        bool ok = true;
        for (size_t d = 0; d < need.size() && ok; d++) {
            int free_lanes = 0;
            for (Context* c : g->lanes[d]) free_lanes += c->busy ? 0 : 1;
            ok = free_lanes >= need[d];
        }
        if (ok) {
            std::vector<Context*> out;
            for (size_t i = 0; i < devs.size(); i++) {
                Context* c = pick_free_lane(devs[i], i == 0 ? hint0 : nullptr, keys && i < keys->size() ? (*keys)[i] : 0);   // cannot fail: the free lanes were counted above
                c->busy = true;
                c->opt = g->opt;
                c->cur_stream = c->stream;
                out.push_back(c);
            }
            return out;
        }
        g_lane_cv.wait(lk);
    }
}

void release_lane(Context* c) {
    {
        std::lock_guard<std::mutex> lk(g_lane_mu);
        c->busy = false;
    }
    g_lane_cv.notify_all();
}

static Options current_options() {
    std::lock_guard<std::mutex> lk(g_lane_mu);
    if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    return g->opt;
}

template <class Fn>
static int32_t guarded(Fn&& fn) {
    try {
        fn();
        return ZKM_OK;
    } catch (const ZkmError& e) {
        cudaGetLastError();  // clear sticky-free errors so the next call starts clean
        return e.code;
    } catch (const std::exception& e) {
        set_error("internal: %s", e.what());
        return ZKM_ERR_CUDA;
    } catch (...) {
        set_error("internal: unknown exception");
        return ZKM_ERR_CUDA;
    }
}

static void check_curve_group(int curve, int group) {
    if (!curve_known(curve)) ZKM_FAIL(ZKM_ERR_ARG, "unknown curve id %d", curve);
    if (group != 1 && group != 2) ZKM_FAIL(ZKM_ERR_ARG, "group must be 1 or 2, got %d", group);
}

// host -> device through the copy engine; pageable memory is fine (driver stages it)
static void h2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (bytes) ZKM_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s));
}

static size_t rec_bytes(int curve, int group) { return (2 * (size_t)coord_words(curve, group) + 1) * 8; }
// flag word of a result record read back by a host entry point: 0 finite, 1 infinity, 2 = the MSM saw a scalar with
// bits at or above the modulus width (detected on the device, reported here: the run itself never waits for the host)
static uint8_t rec_flag(uint64_t flag) {
    if (flag == 2) ZKM_FAIL(ZKM_ERR_SCALAR_RANGE, "a scalar has bits at or above the modulus width (not a canonical Fr)");
    return flag ? 1 : 0;
}

// ------------------------------------------------------------------------------------------ registrations
static std::shared_ptr<BasesReg> build_registration(int curve, int group, const uint64_t* xy, const uint8_t* inf, size_t n,
                                                    uint32_t flags) {
    check_curve_group(curve, group);
    if (n && !xy) ZKM_FAIL(ZKM_ERR_ARG, "null bases");
    const int ndev = device_count_initialised();
    if (ndev == 0) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    const Options opt = current_options();
    const bool precompute = (flags & ZKM_REG_PRECOMPUTE) || opt.msm_precompute;
    const int placed = (int)((flags >> 8) & 0xff);           // ZKM_REG_DEVICE(i) = (i + 1) << 8
    if (placed > ndev) ZKM_FAIL(ZKM_ERR_ARG, "ZKM_REG_DEVICE(%d): only %d devices initialised", placed - 1, ndev);
    const size_t rec = 2 * (size_t)coord_words(curve, group) * 8;
    auto reg = std::make_shared<BasesReg>();                  // its destructor frees whatever was built if we throw
    reg->curve = curve;
    reg->group = group;
    reg->n = n;
    const int nparts = ((flags & ZKM_REG_SHARD) && ndev > 1 && n >= (size_t)ndev) ? ndev : 1;
    reg->parts.reserve(nparts);
    for (int i = 0; i < nparts; i++) {
        BasesPart p;
        p.dev = nparts > 1 ? i : (placed ? placed - 1 : 0);
        p.first = n * (size_t)i / nparts;
        p.n = n * (size_t)(i + 1) / nparts - p.first;
        reg->parts.push_back(p);
    }
    for (BasesPart& p : reg->parts) {
        LaneGuard lane(p.dev);
        Context* c = lane.c;
        p.ordinal = c->device;
        ZKM_CUDA(cudaSetDevice(c->device));
        const size_t bytes = p.n * rec;
        ZKM_CUDA(malloc_retry((void**)&p.d_xy, bytes ? bytes : 16));
        reg->bytes += bytes;
        // cudaMemcpyDefault: `xy` may be a host pointer or a device pointer on any device (UVA picks the route)
        if (bytes) ZKM_CUDA(cudaMemcpyAsync(p.d_xy, (const char*)xy + p.first * rec, bytes, cudaMemcpyDefault, c->stream));
        if (inf) {
            ZKM_CUDA(cudaMalloc((void**)&p.d_inf, p.n ? p.n : 16));
            reg->bytes += p.n;
            if (p.n) ZKM_CUDA(cudaMemcpyAsync(p.d_inf, inf + p.first, p.n, cudaMemcpyDefault, c->stream));
        }
        if (precompute) {
            msm_precompute(c, curve, group, &p, c->stream);
            reg->bytes += p.n * (size_t)p.pre_W * rec;
        }
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
    }
    return reg;
}

static uint64_t publish(std::shared_ptr<BasesReg> reg) {
    std::lock_guard<std::mutex> rl(g->reg_mu);
    uint64_t h = g->next_handle++;
    g->bases[h] = std::move(reg);
    return h;
}

static std::shared_ptr<BasesReg> lookup(uint64_t handle, size_t offset, size_t n) {
    if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    std::lock_guard<std::mutex> rl(g->reg_mu);
    auto it = g->bases.find(handle);
    if (it == g->bases.end()) ZKM_FAIL(ZKM_ERR_HANDLE, "unknown bases handle %llu", (unsigned long long)handle);
    if (offset > it->second->n || n > it->second->n - offset)
        ZKM_FAIL(ZKM_ERR_HANDLE, "range [%zu, %zu) outside the %zu registered bases", offset, offset + n, it->second->n);
    return it->second;
}

// ------------------------------------------------------------------------------------------ MSM over a registration
// A job = the slice of one MSM that falls on one part (one device).
struct Job {
    const BasesPart* part;
    size_t local_off, count, scal_off;    // within the part / within the caller's scalar array
};
static std::vector<Job> split_jobs(const BasesReg& r, size_t offset, size_t n) {
    std::vector<Job> jobs;
    for (const BasesPart& p : r.parts) {
        const size_t lo = offset > p.first ? offset : p.first;
        const size_t hi = (offset + n < p.first + p.n) ? offset + n : p.first + p.n;
        if (lo < hi) jobs.push_back(Job{&p, lo - p.first, hi - lo, lo - offset});
    }
    return jobs;
}

// lane affinity of an MSM job: the registered part it runs over and the size class of the run (workspaces are sized by both)
static uint64_t lane_key(const BasesPart* p, size_t n) {
    int lg = 0;
    while (((size_t)1 << lg) < n) lg++;
    return ((uint64_t)(uintptr_t)p) ^ ((uint64_t)(lg + 1) << 56);
}

static void run_part(Context* c, const BasesReg& r, const Job& j, const uint64_t* d_scal, uint64_t* d_rec, cudaStream_t s,
                     const ScalarFeed* feed = nullptr) {
    const size_t rec = 2 * (size_t)coord_words(r.curve, r.group) * 8;
    const BasesPart& p = *j.part;
    msm_run(c, r.curve, r.group, (const char*)p.d_xy + j.local_off * rec, p.d_inf ? p.d_inf + j.local_off : nullptr, d_scal,
            j.count, d_rec, s, &p, j.local_off, feed);
}

// Upload `count` scalars of `sbytes` bytes in up to 8 chunks on the lane's COPY stream, one event per chunk: the histogram
// pass of the MSM then runs behind the copies instead of after them (a 2^24-point MSM uploads 512 MB, ~9.5 ms over PCIe).
// The copy stream is ordered after everything the lane's stream holds so far (previous users of the buffer, its allocation).
static void upload_scalars_chunked(Context* c, uint64_t* d_scal, const void* h_scal, size_t count, size_t sbytes, ScalarFeed* feed) {
    for (int i = 0; i < 9; i++)
        if (!c->feed_ev[i]) ZKM_CUDA(cudaEventCreateWithFlags(&c->feed_ev[i], cudaEventDisableTiming));
    ZKM_CUDA(cudaEventRecord(c->feed_ev[8], c->stream));
    ZKM_CUDA(cudaStreamWaitEvent(c->copy_stream, c->feed_ev[8], 0));
    const int chunks = 8;
    const size_t per = ((count + chunks - 1) / chunks + 1023) & ~(size_t)1023;
    feed->n = 0;
    for (size_t b = 0; b < count; b += per) {
        const size_t e = b + per < count ? b + per : count;
        const int i = feed->n;
        ZKM_CUDA(cudaMemcpyAsync((char*)d_scal + b * sbytes, (const char*)h_scal + b * sbytes, (e - b) * sbytes, cudaMemcpyHostToDevice,
                                 c->copy_stream));
        ZKM_CUDA(cudaEventRecord(c->feed_ev[i], c->copy_stream));
        feed->begin[i] = b;
        feed->begin[i + 1] = e;
        feed->ev[i] = c->feed_ev[i];
        feed->n++;
    }
}

// Host scalars in, host affine point out.  One job: the part's device does everything.  Several jobs (bases registered
// with ZKM_REG_SHARD): one host thread + lane per device, each uploads its slice of the scalars and runs the full
// pipeline; the partial result records travel to the primary device over NVLink P2P (cudaMemcpyPeerAsync), are summed
// there (k_points_sum) and the one affine point is read back -- the only cross-device traffic is <= 8 x ~100 bytes.
static void msm_reg_host(const std::shared_ptr<BasesReg>& reg, size_t offset, const uint64_t* scalars, size_t n, uint64_t* out_xy,
                         uint8_t* out_inf, bool montgomery_coeffs = false) {
    const BasesReg& r = *reg;
    if (!out_xy || !out_inf) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
    if (n && !scalars) ZKM_FAIL(ZKM_ERR_ARG, "null scalars");
    const int W = coord_words(r.curve, r.group);
    const size_t sbytes = (size_t)fr_words(r.curve) * 8;   // BigInteger256 / BigInteger384
    const size_t rb = rec_bytes(r.curve, r.group);
    std::vector<Job> jobs = split_jobs(r, offset, n);
    auto one = [&](Context* c, const Job& j, uint64_t* d_rec) {
        ZKM_CUDA(cudaSetDevice(c->device));
        uint64_t* d_scal = (uint64_t*)c->io_scalars.get((j.count ? j.count : 1) * sbytes);
        if (!montgomery_coeffs && j.count >= ((size_t)1 << 22)) {
            ScalarFeed feed;
            upload_scalars_chunked(c, d_scal, (const char*)scalars + j.scal_off * sbytes, j.count, sbytes, &feed);
            run_part(c, r, j, d_scal, d_rec, c->stream, &feed);
            return;
        }
        h2d(d_scal, (const char*)scalars + j.scal_off * sbytes, j.count * sbytes, c->stream);
        if (montgomery_coeffs) fr_into_repr_run(c, r.curve, d_scal, d_scal, (uint64_t)j.count, c->stream);   // coeffs.into_repr()
        run_part(c, r, j, d_scal, d_rec, c->stream);
    };
    auto read_back = [&](Context* c, const uint64_t* d_rec) {
        uint64_t* h = (uint64_t*)c->pin_in.get(rb);
        ZKM_CUDA(cudaMemcpyAsync(h, d_rec, rb, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
        memcpy(out_xy, h, 2 * (size_t)W * 8);
        *out_inf = rec_flag(h[2 * W]);
    };
    if (jobs.size() <= 1) {
        LaneGuard lane(jobs.empty() ? 0 : jobs[0].part->dev, nullptr, jobs.empty() ? 0 : lane_key(jobs[0].part, jobs[0].count));
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        StreamScope scope(c, c->stream);
        uint64_t* d_out = (uint64_t*)c->io_out.get(rb);
        if (jobs.empty()) {
            msm_run(c, r.curve, r.group, nullptr, nullptr, nullptr, 0, d_out, c->stream);   // identity
        } else {
            one(c, jobs[0], d_out);
        }
        read_back(c, d_out);
        return;
    }
    // lane 0: the home lane (gather + final sum on the primary device); lanes 1..: one per shard -- taken together
    std::vector<int> devs{0};
    for (const Job& j : jobs) devs.push_back(j.part->dev);
    MultiLaneGuard lanes(devs);
    Context* hc = lanes.c[0];
    ZKM_CUDA(cudaSetDevice(hc->device));
    StreamScope hscope(hc, hc->stream);
    // k_msm_final / k_points_sum WRITE records with 128-bit stores (16-byte aligned destinations only); records are 8 n + 8
    // bytes long, so only the first slot of a packed array is aligned: the sum goes to offset 0, the gathered records
    // (which are only ever written by copies and read limb by limb) follow from offset `gofs`
    const size_t gofs = (rb + 15) & ~(size_t)15;
    char* d_gather = (char*)hc->gather.get(gofs + jobs.size() * rb);
    // the gather buffer is allocated in stream order on the home stream: the shard streams that copy into it wait for it
    cudaEvent_t ev_g;
    ZKM_CUDA(cudaEventCreateWithFlags(&ev_g, cudaEventDisableTiming));
    struct EvGuard { cudaEvent_t e; ~EvGuard() { cudaEventDestroy(e); } } ev_g_guard{ev_g};
    ZKM_CUDA(cudaEventRecord(ev_g, hc->stream));
    const int home_ord = hc->device;
    std::vector<int32_t> rc(jobs.size(), ZKM_OK);
    std::vector<std::string> msg(jobs.size());
    std::vector<std::thread> th;
    for (size_t i = 0; i < jobs.size(); i++) {
        th.emplace_back([&, i] {
            rc[i] = guarded([&] {
                Context* c = lanes.c[1 + i];
                ZKM_CUDA(cudaSetDevice(c->device));
                StreamScope scope(c, c->stream);
                uint64_t* d_rec = (uint64_t*)c->io_out.get(rb);
                one(c, jobs[i], d_rec);
                ZKM_CUDA(cudaStreamWaitEvent(c->stream, ev_g, 0));
                ZKM_CUDA(cudaMemcpyPeerAsync(d_gather + gofs + i * rb, home_ord, d_rec, c->device, rb, c->stream));
                ZKM_CUDA(cudaStreamSynchronize(c->stream));
            });
            if (rc[i] != ZKM_OK) msg[i] = t_err;
        });
    }
    for (auto& t : th) t.join();
    for (size_t i = 0; i < jobs.size(); i++)
        if (rc[i] != ZKM_OK) {
            set_error("shard %zu (device index %d): %s", i, jobs[i].part->dev, msg[i].c_str());
            throw ZkmError{rc[i]};
        }
    ZKM_CUDA(cudaSetDevice(hc->device));
    uint64_t* d_sum = (uint64_t*)d_gather;
    points_sum_run(hc, r.curve, r.group, (const uint64_t*)(d_gather + gofs), jobs.size(), d_sum, hc->stream);
    read_back(hc, d_sum);
}

// index of the initialised device that owns a device pointer (the caller's "home" device)
static int home_device_of(const void* dptr) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, dptr) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
        cudaGetLastError();
        ZKM_FAIL(ZKM_ERR_ARG, "not a device pointer");
    }
    std::lock_guard<std::mutex> lk(g_lane_mu);
    for (size_t i = 0; i < g->devs.size(); i++)
        if (g->devs[i]->device == at.device) return (int)i;
    ZKM_FAIL(ZKM_ERR_ARG, "device pointer lives on CUDA device %d, which zkm_init* did not initialise", at.device);
}

// the stream a *_device call enqueues on: the caller's, or the device's library stream when the caller passed NULL
static cudaStream_t call_stream(int dev, void* stream) {
    if (stream) return (cudaStream_t)stream;
    std::lock_guard<std::mutex> lk(g_lane_mu);
    return g->devs[dev]->null_stream;
}

// Device-resident MSMs over registrations, all ordered after the current point of `caller` and joined back into it.
// Items whose registration is one part on the caller's device and that are alone in the call run directly on the
// caller's stream.  Otherwise every job gets its own host thread, lane and stream (concurrent on the GPU: the five MSMs
// of create_proof, the G2 one on another GPU when its bases were registered there); scalars and result records cross
// devices with peer copies, sharded items are summed on the caller's device.
struct DevItem {
    std::shared_ptr<BasesReg> reg;
    size_t offset, n;
    const uint64_t* d_scalars;
    uint64_t* d_out;
    // non-null: when the item runs as one job on a lane of its own, its completion event is handed back here instead
    // of being joined into the caller's stream (the caller waits for it and destroys it); null on return otherwise
    cudaEvent_t* done = nullptr;
};
struct ItemsPlan {
    struct Flat { size_t item, k; Job job; };
    std::vector<Flat> flat;
    std::vector<size_t> njobs, goff;
    size_t gbytes = 0;       // sharded items gather their partial records at goff[item] + k * rec_bytes (copies only)
    bool fast = false;
    std::vector<int> devs;           // lane 0: the home lane; lanes 1..: one per job
    std::vector<uint64_t> keys;      // lane affinity: the part of the registration a job runs over (same workspace sizes)
};
static ItemsPlan plan_items(const std::vector<DevItem>& items, int home) {
    ItemsPlan p;
    p.njobs.assign(items.size(), 0);
    p.goff.assign(items.size(), 0);
    for (size_t i = 0; i < items.size(); i++) {
        std::vector<Job> jobs = split_jobs(*items[i].reg, items[i].offset, items[i].n);
        p.njobs[i] = jobs.size();
        for (size_t k = 0; k < jobs.size(); k++) p.flat.push_back(ItemsPlan::Flat{i, k, jobs[k]});
        if (jobs.size() > 1) {
            p.goff[i] = p.gbytes;
            p.gbytes += (jobs.size() * rec_bytes(items[i].reg->curve, items[i].reg->group) + 15) & ~(size_t)15;
        }
    }
    p.fast = items.size() == 1 && p.flat.size() == 1 && p.flat[0].job.part->dev == home;
    p.devs = {home};
    p.keys = {0};
    if (!p.fast)
        for (const ItemsPlan::Flat& f : p.flat) {
            p.devs.push_back(f.job.part->dev);
            p.keys.push_back(lane_key(f.job.part, f.job.count));
        }
    return p;
}
static void run_items(std::vector<DevItem>& items, const ItemsPlan& plan, Context* const* lanes, cudaStream_t caller);
static void msm_items_device(std::vector<DevItem>& items, int home, cudaStream_t caller_or_null) {
    const ItemsPlan plan = plan_items(items, home);
    // all lanes taken together (no hold-and-wait between concurrent calls)
    MultiLaneGuard lanes(plan.devs, caller_or_null, &plan.keys);
    run_items(items, plan, lanes.c.data(), caller_or_null);
}
// the MSMs of `items` on the lanes of plan.devs (lanes[0]: the home lane)
static void run_items(std::vector<DevItem>& items, const ItemsPlan& plan, Context* const* lanes, cudaStream_t caller) {
    const std::vector<ItemsPlan::Flat>& flat = plan.flat;
    const std::vector<size_t>& njobs = plan.njobs;
    const std::vector<size_t>& goff = plan.goff;
    for (DevItem& it : items)
        if (it.done) *it.done = nullptr;
    Context* hc = lanes[0];
    ZKM_CUDA(cudaSetDevice(hc->device));
    StreamScope hscope(hc, caller);
    // fast path: one job on the caller's device -> no threads, no events, the caller's stream itself
    if (plan.fast) {
        const BasesReg& r = *items[0].reg;
        const size_t sbytes = (size_t)fr_words(r.curve) * 8;
        run_part(hc, r, flat[0].job, (const uint64_t*)((const char*)items[0].d_scalars + flat[0].job.scal_off * sbytes),
                 items[0].d_out, caller);
        return;
    }
    for (size_t i = 0; i < items.size(); i++)
        if (njobs[i] == 0) {
            const BasesReg& r = *items[i].reg;
            msm_run(hc, r.curve, r.group, nullptr, nullptr, nullptr, 0, items[i].d_out, caller);   // identity
        }
    if (flat.empty()) return;
    char* d_gather = (char*)hc->gather.get(plan.gbytes + 16);
    cudaEvent_t ev_in;
    ZKM_CUDA(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
    ZKM_CUDA(cudaEventRecord(ev_in, caller));
    const int home_ord = hc->device;
    std::vector<int32_t> rc(flat.size(), ZKM_OK);
    std::vector<std::string> msg(flat.size());
    std::vector<cudaEvent_t> ev_out(flat.size(), nullptr);
    std::vector<std::thread> th;
    for (size_t f = 0; f < flat.size(); f++) {
        th.emplace_back([&, f] {
            rc[f] = guarded([&] {
                const ItemsPlan::Flat& fj = flat[f];
                const DevItem& it = items[fj.item];
                const BasesReg& r = *it.reg;
                const size_t sbytes = (size_t)fr_words(r.curve) * 8, rb = rec_bytes(r.curve, r.group);
                Context* c = lanes[1 + f];
                ZKM_CUDA(cudaSetDevice(c->device));
                cudaStream_t s = c->stream;
                StreamScope scope(c, s);
                ZKM_CUDA(cudaStreamWaitEvent(s, ev_in, 0));
                const uint64_t* d_scal = (const uint64_t*)((const char*)it.d_scalars + fj.job.scal_off * sbytes);
                const bool remote = c->device != home_ord;
                if (remote) {   // scalars live on the caller's device: bring this job's slice over NVLink
                    uint64_t* local = (uint64_t*)c->io_scalars.get((fj.job.count ? fj.job.count : 1) * sbytes);
                    ZKM_CUDA(cudaMemcpyPeerAsync(local, c->device, d_scal, home_ord, fj.job.count * sbytes, s));
                    d_scal = local;
                }
                // single-job items on the caller's device write their record straight to the caller's buffer (16-byte
                // aligned by contract); everything else goes through the lane's own aligned record and a copy
                const bool sharded = njobs[fj.item] > 1;
                uint64_t* dst = sharded ? (uint64_t*)(d_gather + goff[fj.item] + fj.k * rb) : it.d_out;
                if (remote || sharded) {
                    uint64_t* d_rec = (uint64_t*)c->io_out.get(rb);
                    run_part(c, r, fj.job, d_scal, d_rec, s);
                    ZKM_CUDA(cudaMemcpyPeerAsync(dst, home_ord, d_rec, c->device, rb, s));
                } else {
                    run_part(c, r, fj.job, d_scal, dst, s);
                }
                ZKM_CUDA(cudaEventCreateWithFlags(&ev_out[f], cudaEventDisableTiming));
                ZKM_CUDA(cudaEventRecord(ev_out[f], s));
            });
            if (rc[f] != ZKM_OK) msg[f] = t_err;
        });
    }
    for (auto& t : th) t.join();
    ZKM_CUDA(cudaSetDevice(hc->device));
    int32_t first = ZKM_OK;
    for (size_t f = 0; f < flat.size(); f++) {
        DevItem& it = items[flat[f].item];
        if (ev_out[f] && it.done && njobs[flat[f].item] == 1 && rc[f] == ZKM_OK) {
            *it.done = ev_out[f];      // joined by the caller
        } else if (ev_out[f]) {
            cudaStreamWaitEvent(caller, ev_out[f], 0);
            cudaEventDestroy(ev_out[f]);
        }
        if (rc[f] != ZKM_OK && first == ZKM_OK) {
            first = rc[f];
            set_error("item %zu: %s", flat[f].item, msg[f].c_str());
        }
    }
    cudaEventDestroy(ev_in);
    if (first != ZKM_OK) {
        for (DevItem& it : items)
            if (it.done && *it.done) {
                cudaStreamWaitEvent(caller, *it.done, 0);
                cudaEventDestroy(*it.done);
                *it.done = nullptr;
            }
        throw ZkmError{first};
    }
    for (size_t i = 0; i < items.size(); i++)
        if (njobs[i] > 1) {
            const BasesReg& r = *items[i].reg;
            points_sum_run(hc, r.curve, r.group, (const uint64_t*)(d_gather + goff[i]), njobs[i], items[i].d_out, caller);
        }
}

// ------------------------------------------------------------------------------------------ registration cache
static uint64_t fnv1a64(uint64_t h, const void* p, size_t bytes) {
    const uint64_t* w = (const uint64_t*)p;
    for (size_t i = 0; i < bytes / 8; i++) {
        h ^= w[i];
        h *= 0x100000001b3ull;
    }
    const unsigned char* t = (const unsigned char*)p + (bytes & ~(size_t)7);
    for (size_t i = 0; i < (bytes & 7); i++) {
        h ^= t[i];
        h *= 0x100000001b3ull;
    }
    return h;
}
// mode 1: 512 records spread evenly over the array (first and last included) + the flags of the same positions;
// mode 2: every byte.
static uint64_t fingerprint(const uint64_t* xy, const uint8_t* inf, size_t n, size_t rec, int mode) {
    uint64_t h = 0xcbf29ce484222325ull ^ (uint64_t)n;
    if (mode >= 2 || n <= 512) {
        h = fnv1a64(h, xy, n * rec);
        if (inf) h = fnv1a64(h, inf, n);
        return h;
    }
    for (size_t k = 0; k < 512; k++) {
        const size_t i = (size_t)((unsigned __int128)k * (n - 1) / 511);
        h = fnv1a64(h, (const char*)xy + i * rec, rec);
        if (inf) h = fnv1a64(h, inf + i, 1);
    }
    return h;
}

static std::shared_ptr<BasesReg> cached_registration(int curve, int group, const uint64_t* xy, const uint8_t* inf, size_t n,
                                                     const Options& opt) {
    const size_t rec = 2 * (size_t)coord_words(curve, group) * 8;
    const uint64_t fp = fingerprint(xy, inf, n, rec, opt.msm_cache);
    Global::CacheKey key{curve, group, xy, inf, n};
    std::shared_ptr<BasesReg> upgrade;       // a small vector that came back: give it window multiples (see below)
    {
        std::lock_guard<std::mutex> lk(g->cache_mu);
        auto it = g->cache.find(key);
        if (it != g->cache.end()) {
            if (it->second.fingerprint == fp) {
                it->second.last_use = ++g->cache_clock;
                g->cache_hits++;
                it->second.hits++;
                const BasesReg& r = *it->second.reg;
                const bool plain = r.parts.size() == 1 && !r.parts[0].d_table;
                if (!(opt.msm_cache_precompute && plain && it->second.hits == 1 && n <= ((size_t)1 << 18))) return it->second.reg;
                upgrade = it->second.reg;
            } else {
                g->cache_bytes -= it->second.reg->bytes;   // same address, different content: replace
                g->cache.erase(it);
            }
        }
        if (!upgrade) g->cache_misses++;
    }
    if (upgrade) {
        // Second call with the same bases (a proving key is used for every proof, benches/groth16.rs:107-115): rebuild the
        // registration from its device copy WITH the window multiples 2^(c w) P_i.  For the small MSMs of zkMember's
        // circuits (2^15-2^16 points) the Horner chain of c W doublings is half of the time (k_msm_final 1.6 of 3.3 ms at
        // 2^16); the table removes it.  Not done on the first call: a vector that never comes back would only pay for it.
        const BasesPart& p0 = upgrade->parts[0];
        std::shared_ptr<BasesReg> better =
            build_registration(curve, group, (const uint64_t*)p0.d_xy, p0.d_inf, n, ZKM_REG_PRECOMPUTE);
        std::lock_guard<std::mutex> lk(g->cache_mu);
        auto it = g->cache.find(key);
        if (it != g->cache.end() && it->second.reg == upgrade) {
            g->cache_bytes += better->bytes - upgrade->bytes;
            it->second.reg = better;
        }
        return better;
    }
    std::shared_ptr<BasesReg> reg = build_registration(curve, group, xy, inf, n, 0);
    std::lock_guard<std::mutex> lk(g->cache_mu);
    const size_t cap = (size_t)opt.msm_cache_max_mb << 20;
    while (!g->cache.empty() && g->cache_bytes + reg->bytes > cap) {          // least recently used goes first
        auto victim = g->cache.begin();
        for (auto it = g->cache.begin(); it != g->cache.end(); ++it)
            if (it->second.last_use < victim->second.last_use) victim = it;
        g->cache_bytes -= victim->second.reg->bytes;
        g->cache.erase(victim);
    }
    if (reg->bytes <= cap) {
        g->cache[key] = Global::CacheEntry{reg, fp, ++g->cache_clock};
        g->cache_bytes += reg->bytes;
    }
    return reg;
}

static int32_t msm_direct(int32_t curve, int group, const uint64_t* bases_xy, const uint8_t* infinity,
                          const uint64_t* scalars, size_t n, uint64_t* out_xy, uint8_t* out_inf) {
    return guarded([&] {
        check_curve_group(curve, group);
        if (n && !bases_xy) ZKM_FAIL(ZKM_ERR_ARG, "null bases");
        if (!out_xy || !out_inf) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
        if (n && !scalars) ZKM_FAIL(ZKM_ERR_ARG, "null scalars");
        const Options opt = current_options();
        if (opt.msm_cache && n >= 1024) {
            std::shared_ptr<BasesReg> reg = cached_registration(curve, group, bases_xy, infinity, n, opt);
            msm_reg_host(reg, 0, scalars, n, out_xy, out_inf);
            return;
        }
        LaneGuard lane(0);
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        const int W = coord_words(curve, group);
        const size_t sbytes = (size_t)fr_words(curve) * 8;
        StreamScope scope(c, c->stream);
        void* d_bases = c->io_bases.get((n ? n : 1) * 2 * W * 8);
        uint8_t* d_inf = nullptr;
        h2d(d_bases, bases_xy, n * 2 * W * 8, c->stream);
        if (infinity) {
            d_inf = (uint8_t*)c->io_inf.get(n ? n : 1);
            h2d(d_inf, infinity, n, c->stream);
        }
        uint64_t* d_scal = (uint64_t*)c->io_scalars.get((n ? n : 1) * sbytes);
        uint64_t* d_out = (uint64_t*)c->io_out.get((2 * W + 1) * 8);
        h2d(d_scal, scalars, n * sbytes, c->stream);
        msm_run(c, curve, group, d_bases, d_inf, d_scal, n, d_out, c->stream);
        uint64_t* h = (uint64_t*)c->pin_in.get((2 * W + 1) * 8);
        ZKM_CUDA(cudaMemcpyAsync(h, d_out, (2 * W + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
        memcpy(out_xy, h, 2 * W * 8);
        *out_inf = rec_flag(h[2 * W]);
    });
}

static int pick_host_call_device() {
    std::lock_guard<std::mutex> lk(g_lane_mu);
    if (!g || g->devs.empty()) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    if (!g->opt.spread_host_calls || g->devs.size() == 1) return 0;
    return (int)(g->rr.fetch_add(1) % g->devs.size());
}

static void free_lanes(std::vector<Context*>& lanes) {
    for (Context* c : lanes) {
        cudaSetDevice(c->device);
        c->ntt_a.release();
        c->ntt_b.release();
        for (auto& b : c->ws) b.release();
        c->io_scalars.release();
        c->io_bases.release();
        c->io_inf.release();
        c->io_out.release();
        c->gather.release();
        c->pin_in.release();
        c->pin_out.release();
        for (auto& e : c->pev)
            if (e) cudaEventDestroy(e);
        if (c->done_ev) cudaEventDestroy(c->done_ev);
        if (c->stream) cudaStreamDestroy(c->stream);
        if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
        for (cudaEvent_t& e : c->feed_ev)
            if (e) {
                cudaEventDestroy(e);
                e = nullptr;
            }
        delete c;
    }
    lanes.clear();
}

static int32_t init_devices(const int32_t* devices, int32_t count) {
    return guarded([&] {
        std::lock_guard<std::mutex> lk(g_init_mu);
        if (count < 1 || count > 16 || !devices) ZKM_FAIL(ZKM_ERR_ARG, "between 1 and 16 devices expected");
        std::vector<int> want(devices, devices + count);
        if (g) {
            if (g->ordinals != want) {
                std::string have;
                for (int d : g->ordinals) have += (have.empty() ? "" : ",") + std::to_string(d);
                ZKM_FAIL(ZKM_ERR_ARG, "already initialised on device(s) %s; call zkm_shutdown() before re-initialising", have.c_str());
            }
            return;
        }
        // Hardware work queues: a proof keeps six streams busy and several proofs are in flight; with the default of 8
        // queues streams share one and wait behind each other's kernels (Groth16 proxy on B200: 389 -> 454 proofs/s with
        // 32).  Only effective if the CUDA runtime has not been initialised by the process yet; the user's setting wins.
        setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0) {
            cudaGetLastError();
            ZKM_FAIL(ZKM_ERR_CUDA, "no usable CUDA device (%s); this library has no CPU fallback",
                     e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        }
        for (int d : want)
            if (d < 0 || d >= ndev) ZKM_FAIL(ZKM_ERR_ARG, "device %d out of range (0..%d)", d, ndev - 1);
        Global* ng = new Global();
        ng->ordinals = want;
        try {
            for (int i = 0; i < count; i++) {
                const int device = want[i];
                ZKM_CUDA(cudaSetDevice(device));
                cudaDeviceProp prop;
                ZKM_CUDA(cudaGetDeviceProperties(&prop, device));
                if (prop.major != 10)
                    ZKM_FAIL(ZKM_ERR_CUDA, "device %d is sm_%d%d; this build carries sm_100a code only", device, prop.major, prop.minor);
                // the MSM gathers 64..192-byte base records at random: fetch 32-byte sectors, not 128-byte lines
                cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 32);
                cudaGetLastError();
                Shared* sh = new Shared();
                sh->device = device;
                sh->index = i;
                sh->sm_count = prop.multiProcessorCount;
                ng->devs.push_back(sh);
                ng->lanes.emplace_back();
                for (int l = 0; l < ZKM_NUM_LANES; l++) {
                    Context* c = new Context(sh);
                    c->lane_id = l;
                    ng->lanes.back().push_back(c);   // owned from here on: freed below if a later step throws
                    ZKM_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
                    ZKM_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
                    c->cur_stream = c->stream;
                }
                ZKM_CUDA(cudaStreamCreateWithFlags(&sh->null_stream, cudaStreamNonBlocking));
                // workspaces come from the default memory pool (DevBuf): keep freed blocks in the process
                cudaMemPool_t pool;
                ZKM_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
                uint64_t keep = UINT64_MAX;
                ZKM_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
            }
            // NVLink peer access between every pair of distinct devices (partial results and scalar slices travel P2P)
            for (int i = 0; i < count; i++)
                for (int j = 0; j < count; j++) {
                    if (want[i] == want[j]) continue;
                    int can = 0;
                    cudaDeviceCanAccessPeer(&can, want[i], want[j]);
                    if (can) {
                        cudaSetDevice(want[i]);
                        cudaDeviceEnablePeerAccess(want[j], 0);
                        // pool memory of device j (lane workspaces: scalar slices, result records) readable / writable from i
                        cudaMemPool_t pool;
                        if (cudaDeviceGetDefaultMemPool(&pool, want[j]) == cudaSuccess) {
                            cudaMemAccessDesc desc;
                            memset(&desc, 0, sizeof(desc));
                            desc.location.type = cudaMemLocationTypeDevice;
                            desc.location.id = want[i];
                            desc.flags = cudaMemAccessFlagsProtReadWrite;
                            cudaMemPoolSetAccess(pool, &desc, 1);
                        }
                    }
                    cudaGetLastError();   // "already enabled" is fine
                }
            ZKM_CUDA(cudaSetDevice(want[0]));
        } catch (...) {
            for (auto& v : ng->lanes) free_lanes(v);
            for (Shared* sh : ng->devs) {
                if (sh->null_stream) cudaStreamDestroy(sh->null_stream);
                delete sh;
            }
            delete ng;
            throw;
        }
        std::lock_guard<std::mutex> ll(g_lane_mu);
        g = ng;
    });
}

// ------------------------------------------------------------------------------------------ Groth16 prover
static std::shared_ptr<G16Key> g16_lookup(uint64_t pk) {
    if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    std::lock_guard<std::mutex> rl(g->reg_mu);
    auto it = g->pks.find(pk);
    if (it == g->pks.end()) ZKM_FAIL(ZKM_ERR_HANDLE, "unknown Groth16 proving key %llu", (unsigned long long)pk);
    return it->second;
}

static uint64_t g16_create(int curve, const uint64_t* handles, const uint64_t* g1_xy, const uint8_t* g1_inf, const uint64_t* g2_xy,
                           const uint8_t* g2_inf) {
    if (!curve_known(curve)) ZKM_FAIL(ZKM_ERR_ARG, "unknown curve id %d", curve);
    if (!handles || !g1_xy || !g1_inf || !g2_xy || !g2_inf) ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
    auto key = std::make_shared<G16Key>();
    key->curve = curve;
    static const char* names[5] = {"h_query", "l_query", "a_query", "b_g1_query", "b_g2_query"};
    for (int i = 0; i < 5; i++) {
        key->reg[i] = lookup(handles[i], 0, 0);
        const int want = i == G16_B2 ? 2 : 1;
        if (key->reg[i]->curve != curve || key->reg[i]->group != want)
            ZKM_FAIL(ZKM_ERR_ARG, "%s: registration of curve %d group %d, expected curve %d group %d", names[i], key->reg[i]->curve,
                     key->reg[i]->group, curve, want);
    }
    key->m = key->reg[G16_A]->n;
    if (key->reg[G16_B1]->n != key->m || key->reg[G16_B2]->n != key->m)
        ZKM_FAIL(ZKM_ERR_ARG, "a_query, b_g1_query and b_g2_query differ in length (%zu, %zu, %zu after entry 0)", key->m,
                 key->reg[G16_B1]->n, key->reg[G16_B2]->n);
    const size_t xy1 = 2 * (size_t)coord_words(curve, 1), xy2 = 2 * (size_t)coord_words(curve, 2);
    const size_t rw1 = xy1 + 1, rw2 = xy2 + 1;
    std::vector<uint64_t> rec(5 * rw1 + 3 * rw2, 0);
    for (int i = 0; i < 5; i++) {
        memcpy(&rec[i * rw1], g1_xy + i * xy1, xy1 * 8);
        rec[i * rw1 + xy1] = g1_inf[i] ? 1 : 0;
    }
    for (int j = 0; j < 3; j++) {
        memcpy(&rec[5 * rw1 + j * rw2], g2_xy + j * xy2, xy2 * 8);
        rec[5 * rw1 + j * rw2 + xy2] = g2_inf[j] ? 1 : 0;
    }
    key->delta1_inf = g1_inf[G16_DELTA] != 0;
    key->delta2_inf = g2_inf[G16_DELTA2] != 0;
    const G16Ops ops = groth16_ops(curve);
    const int ndev = device_count_initialised();
    if (ndev == 0) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    key->dev.resize(ndev);
    for (int d = 0; d < ndev; d++) {
        LaneGuard lane(d);
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        G16Key::Dev& kd = key->dev[d];
        kd.ordinal = c->device;
        StreamScope scope(c, c->stream);
        ZKM_CUDA(malloc_retry((void**)&kd.d_key, rec.size() * 8));
        h2d(kd.d_key, rec.data(), rec.size() * 8, c->stream);
        if (!key->delta1_inf) {
            ZKM_CUDA(malloc_retry((void**)&kd.d_tab1, ops.table_bytes(1)));
            ops.table(c, 1, g1_xy + G16_DELTA * xy1, kd.d_tab1, c->stream);
        }
        if (!key->delta2_inf) {
            ZKM_CUDA(malloc_retry((void**)&kd.d_tab2, ops.table_bytes(2)));
            ops.table(c, 2, g2_xy + G16_DELTA2 * xy2, kd.d_tab2, c->stream);
        }
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
    }
    std::lock_guard<std::mutex> rl(g->reg_mu);
    const uint64_t h = g->next_handle++;
    g->pks[h] = key;
    return h;
}

static void g16_check(const G16Key& k, uint32_t log_n, size_t num_inputs, size_t num_aux) {
    const int adicity = fr_two_adicity(k.curve);
    if ((int)log_n > adicity) ZKM_FAIL(ZKM_ERR_DOMAIN, "log_n %u exceeds the two-adicity %d of Fr", log_n, adicity);
    if (log_n > 28) ZKM_FAIL(ZKM_ERR_ARG, "log_n %u: witness maps above 2^28 are not supported by this build", log_n);
    if (num_inputs + num_aux != k.m)
        ZKM_FAIL(ZKM_ERR_ARG, "num_inputs + num_aux = %zu, but the key's a_query has %zu + 1 entries", num_inputs + num_aux, k.m);
    if (k.reg[G16_L]->n != num_aux) ZKM_FAIL(ZKM_ERR_ARG, "num_aux = %zu, but the key's l_query has %zu entries", num_aux, k.reg[G16_L]->n);
    if (k.reg[G16_H]->n > ((size_t)1 << log_n))
        ZKM_FAIL(ZKM_ERR_ARG, "the key's h_query has %zu entries, more than the domain size 2^%u", k.reg[G16_H]->n, log_n);
}

// host buffers of zkm_groth16_prove: staged through the home lane's pinned and device workspaces
struct G16Host {
    const uint64_t *a, *b, *c, *assignment;
    uint64_t *a_xy, *b_xy, *c_xy;
    uint8_t *a_inf, *b_inf, *c_inf;
};

// One proof enqueued on `caller` (null: the home lane's stream) of device index `home`: witness map (h replaces b),
// into_repr(h), the range check of the assignment, the five MSMs on lanes of their own (the b_g2 one joined only before
// the G2 assembly), the G1 assembly (A, C), the G2 assembly (B).  All lanes are taken at once.
static void g16_prove(const G16Key& k, int home, cudaStream_t caller, uint32_t log_n, size_t num_inputs, size_t num_aux,
                      const uint64_t* r, const uint64_t* s, uint64_t* d_a, uint64_t* d_b, uint64_t* d_c, const uint64_t* d_asg,
                      uint64_t* d_out, const G16Host* host) {
    const int curve = k.curve;
    const size_t S = (size_t)fr_words(curve), m = num_inputs + num_aux, nh = k.reg[G16_H]->n;
    const size_t rw1 = 2 * (size_t)coord_words(curve, 1) + 1, rw2 = 2 * (size_t)coord_words(curve, 2) + 1;
    const G16Ops ops = groth16_ops(curve);
    std::vector<DevItem> items(5);
    const size_t offs[5] = {0, 0, 0, 0, 0}, ns[5] = {nh, num_aux, m, m, m};
    for (int i = 0; i < 5; i++) {
        items[i].reg = k.reg[i];
        items[i].offset = offs[i];
        items[i].n = ns[i];
    }
    const ItemsPlan plan = plan_items(items, home);
    MultiLaneGuard lanes(plan.devs, caller, &plan.keys);
    Context* hc = lanes.c[0];
    ZKM_CUDA(cudaSetDevice(hc->device));
    if (!caller) caller = hc->stream;
    StreamScope scope(hc, caller);
    const size_t vb = (S * 8) << log_n, ab = m * S * 8;
    if (host) {   // one pinned upload of a, b, c and the assignment
        char* pin = (char*)hc->pin_in.get(3 * vb + ab);
        memcpy(pin, host->a, vb);
        memcpy(pin + vb, host->b, vb);
        memcpy(pin + 2 * vb, host->c, vb);
        if (ab) memcpy(pin + 3 * vb, host->assignment, ab);
        char* d = (char*)hc->io_scalars.get(3 * vb + ab + 16);
        h2d(d, pin, 3 * vb + ab, caller);
        d_a = (uint64_t*)d;
        d_b = (uint64_t*)(d + vb);
        d_c = (uint64_t*)(d + 2 * vb);
        d_asg = (const uint64_t*)(d + 3 * vb);
    }
    const size_t r1 = (rw1 * 8 + 15) & ~(size_t)15, r2 = (rw2 * 8 + 15) & ~(size_t)15, ob = (2 * rw1 + rw2) * 8;
    char* w = (char*)hc->io_out.get(4 * r1 + r2 + 16 + (host ? ob : 0));
    uint64_t* rec[5];
    for (int i = 0; i < 5; i++) rec[i] = (uint64_t*)(w + i * r1);   // b_g2 last: its record may be the longer one
    uint32_t* d_flag = (uint32_t*)(w + 4 * r1 + r2);
    if (host) d_out = (uint64_t*)(w + 4 * r1 + r2 + 16);
    ZKM_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(uint32_t), caller));
    witness_map_run(hc, curve, d_a, d_b, d_c, log_n, d_b, caller);
    fr_into_repr_run(hc, curve, d_b, d_b, (uint64_t)nh, caller);
    ops.range(hc, d_asg, m, d_flag, caller);
    const uint64_t* scal[5] = {d_b, d_asg + num_inputs * S, d_asg, d_asg, d_asg};
    for (int i = 0; i < 5; i++) {
        items[i].d_scalars = scal[i];
        items[i].d_out = rec[i];
    }
    // the G2 MSM is the longest: the G1 assembly (two ~SCALAR_BITS doubling chains) runs next to it
    struct Join {
        cudaStream_t s;
        cudaEvent_t e = nullptr;
        void now() {
            if (!e) return;
            cudaError_t rc = cudaStreamWaitEvent(s, e, 0);
            cudaEventDestroy(e);
            e = nullptr;
            ZKM_CUDA(rc);
        }
        ~Join() {
            try { now(); } catch (...) { cudaStreamSynchronize(s); cudaGetLastError(); }
        }
    } g2{caller};
    items[G16_B2].done = &g2.e;
    run_items(items, plan, lanes.c.data(), caller);
    G16Args args;
    memset(&args, 0, sizeof(args));
    const G16Key::Dev& kd = k.dev[home];
    args.key1 = kd.d_key;
    args.key2 = kd.d_key + 5 * rw1;
    for (int i = 0; i < 5; i++) {
        args.rec[i] = rec[i];
        args.rec_words[i] = (int)(i == G16_B2 ? rw2 : rw1);
    }
    args.range_flag = d_flag;
    memcpy(args.r, r, S * 8);
    memcpy(args.s, s, S * 8);
    args.out = d_out;
    ops.assemble(hc, 1, args, kd.d_tab1, caller);
    g2.now();
    ops.assemble(hc, 2, args, kd.d_tab2, caller);
    if (!host) return;
    uint64_t* h = (uint64_t*)hc->pin_out.get(ob);
    ZKM_CUDA(cudaMemcpyAsync(h, d_out, ob, cudaMemcpyDeviceToHost, caller));
    ZKM_CUDA(cudaStreamSynchronize(caller));
    const uint64_t* ra = h;
    const uint64_t* rb = h + rw1;
    const uint64_t* rc = h + rw1 + rw2;
    if (ra[rw1 - 1] == 2 || rb[rw2 - 1] == 2 || rc[rw1 - 1] == 2)
        ZKM_FAIL(ZKM_ERR_SCALAR_RANGE, "an assignment element, r or s is not below the scalar modulus");
    memcpy(host->a_xy, ra, (rw1 - 1) * 8);
    memcpy(host->b_xy, rb, (rw2 - 1) * 8);
    memcpy(host->c_xy, rc, (rw1 - 1) * 8);
    *host->a_inf = ra[rw1 - 1] ? 1 : 0;
    *host->b_inf = rb[rw2 - 1] ? 1 : 0;
    *host->c_inf = rc[rw1 - 1] ? 1 : 0;
}

}  // namespace zkm

using namespace zkm;

extern "C" {

const char* zkm_last_error(void) { return t_err; }
const char* zkm_version(void) { return "zkmember-b200 0.2 (sm_100a)"; }

int32_t zkm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int32_t zkm_init(int32_t device) { return init_devices(&device, 1); }

int32_t zkm_init_mask(uint32_t device_mask) {
    int32_t list[32];
    int32_t count = 0;
    for (int i = 0; i < 32; i++)
        if (device_mask & (1u << i)) list[count++] = i;
    if (count > 16) count = 17;   // rejected below with a clear message
    return init_devices(list, count);
}

int32_t zkm_init_devices(const int32_t* devices, int32_t count) { return init_devices(devices, count); }

int32_t zkm_initialised_devices(void) { return device_count_initialised(); }

void zkm_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_init_mu);
    Global* og;
    {
        std::lock_guard<std::mutex> ll(g_lane_mu);
        og = g;
        g = nullptr;
    }
    if (!og) return;
    for (Shared* sh : og->devs) {
        cudaSetDevice(sh->device);
        cudaDeviceSynchronize();
    }
    for (auto& v : og->lanes) free_lanes(v);
    {
        std::lock_guard<std::mutex> cl(og->cache_mu);
        og->cache.clear();
    }
    {
        std::lock_guard<std::mutex> rl(og->reg_mu);
        og->pks.clear();
        og->bases.clear();          // ~BasesReg frees the device memory
    }
    for (Shared* sh : og->devs) {
        cudaSetDevice(sh->device);
        ntt_release_tables(sh);
        if (sh->null_stream) cudaStreamDestroy(sh->null_stream);
        DevBuf::trim_pool();     // the lanes' workspaces went back to the default pool: return them to the device
        delete sh;
    }
    delete og;
    g_lane_cv.notify_all();
}

int32_t zkm_msm_g1(int32_t curve, const uint64_t* bases_xy, const uint8_t* infinity, const uint64_t* scalars, size_t n,
                   uint64_t* out_xy, uint8_t* out_inf) {
    return msm_direct(curve, 1, bases_xy, infinity, scalars, n, out_xy, out_inf);
}
int32_t zkm_msm_g2(int32_t curve, const uint64_t* bases_xy, const uint8_t* infinity, const uint64_t* scalars, size_t n,
                   uint64_t* out_xy, uint8_t* out_inf) {
    return msm_direct(curve, 2, bases_xy, infinity, scalars, n, out_xy, out_inf);
}

int32_t zkm_bases_register_ex(int32_t curve, int32_t group, const uint64_t* bases_xy, const uint8_t* infinity, size_t n,
                              uint32_t flags, uint64_t* handle_out) {
    return guarded([&] {
        if (!handle_out) ZKM_FAIL(ZKM_ERR_ARG, "null handle_out");
        *handle_out = publish(build_registration(curve, group, bases_xy, infinity, n, flags));
    });
}
int32_t zkm_bases_register(int32_t curve, int32_t group, const uint64_t* bases_xy, const uint8_t* infinity, size_t n,
                           uint64_t* handle_out) {
    return zkm_bases_register_ex(curve, group, bases_xy, infinity, n, 0, handle_out);
}
int32_t zkm_bases_register_device(int32_t curve, int32_t group, const uint64_t* d_bases_xy, const uint8_t* d_infinity,
                                  size_t n, uint64_t* handle_out) {
    return zkm_bases_register_ex(curve, group, d_bases_xy, d_infinity, n, 0, handle_out);
}

int32_t zkm_bases_release(uint64_t handle) {
    return guarded([&] {
        if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
        std::shared_ptr<BasesReg> keep;     // destroyed (device memory freed) outside the registry lock
        {
            std::lock_guard<std::mutex> rl(g->reg_mu);
            auto it = g->bases.find(handle);
            if (it == g->bases.end()) ZKM_FAIL(ZKM_ERR_HANDLE, "unknown bases handle %llu", (unsigned long long)handle);
            keep = std::move(it->second);
            g->bases.erase(it);
        }
    });
}

int32_t zkm_msm_registered(uint64_t handle, size_t offset, const uint64_t* scalars, size_t n, uint64_t* out_xy,
                           uint8_t* out_inf) {
    return guarded([&] { msm_reg_host(lookup(handle, offset, n), offset, scalars, n, out_xy, out_inf); });
}

// skip_leading_zeros_and_convert_to_bigints: number of zero coefficients at the low end
static size_t leading_zero_coeffs(const uint64_t* coeffs, size_t n, size_t S) {
    size_t z = 0;
    while (z < n) {
        uint64_t o = 0;
        for (size_t k = 0; k < S; k++) o |= coeffs[S * z + k];
        if (o) break;
        z++;
    }
    return z;
}

static void kzg_commit_impl(uint64_t handle, const uint64_t* coeffs, size_t n, uint64_t* out_xy, uint8_t* out_inf) {
    if (!out_xy || !out_inf || (n && !coeffs)) ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
    std::shared_ptr<BasesReg> r0 = lookup(handle, 0, 0);
    if (r0->group != 1) ZKM_FAIL(ZKM_ERR_ARG, "KZG powers must be G1 bases");
    const size_t S = (size_t)fr_words(r0->curve);
    const size_t z = leading_zero_coeffs(coeffs, n, S);
    std::shared_ptr<BasesReg> r = lookup(handle, z, n - z);
    msm_reg_host(r, z, coeffs + S * z, n - z, out_xy, out_inf, /*montgomery_coeffs=*/true);
}

int32_t zkm_kzg_commit(uint64_t handle, const uint64_t* coeffs, size_t n, uint64_t* out_xy, uint8_t* out_inf) {
    return guarded([&] { kzg_commit_impl(handle, coeffs, n, out_xy, out_inf); });
}

int32_t zkm_kzg_commit_batch(uint64_t handle, int32_t count, const uint64_t* const* coeffs, const size_t* n, uint64_t* out_xy,
                             uint8_t* out_inf) {
    return guarded([&] {
        if (count < 0 || count > 64) ZKM_FAIL(ZKM_ERR_ARG, "count must be 0..64");
        if (count && (!coeffs || !n || !out_xy || !out_inf)) ZKM_FAIL(ZKM_ERR_ARG, "null argument array");
        std::shared_ptr<BasesReg> r0 = lookup(handle, 0, 0);
        const size_t W2 = 2 * (size_t)coord_words(r0->curve, r0->group);
        std::vector<int32_t> rc((size_t)count, ZKM_OK);
        std::vector<std::string> msg((size_t)count);
        // at most ZKM_NUM_LANES - 2 commitments in flight: each borrows a lane (its workspaces are the memory bound)
        const int width = count < ZKM_NUM_LANES - 2 ? count : ZKM_NUM_LANES - 2;
        std::atomic<int> next{0};
        std::vector<std::thread> th;
        for (int t = 0; t < width; t++)
            th.emplace_back([&] {
                for (int i = next.fetch_add(1); i < count; i = next.fetch_add(1)) {
                    rc[i] = guarded([&] { kzg_commit_impl(handle, coeffs[i], n[i], out_xy + (size_t)i * W2, out_inf + i); });
                    if (rc[i] != ZKM_OK) msg[i] = t_err;
                }
            });
        for (auto& t : th) t.join();
        for (int i = 0; i < count; i++)
            if (rc[i] != ZKM_OK) {
                set_error("polynomial %d: %s", i, msg[i].c_str());
                throw ZkmError{rc[i]};
            }
    });
}

// sum of two affine points given as host (xy, inf): through k_points_sum on the primary device
static void add_two_points(int curve, int group, const uint64_t* a_xy, uint8_t a_inf, const uint64_t* b_xy, uint8_t b_inf,
                           uint64_t* out_xy, uint8_t* out_inf) {
    const size_t W2 = 2 * (size_t)coord_words(curve, group), rb = (W2 + 1) * 8;
    LaneGuard lane(0);
    Context* c = lane.c;
    ZKM_CUDA(cudaSetDevice(c->device));
    StreamScope scope(c, c->stream);
    uint64_t* h = (uint64_t*)c->pin_in.get(3 * rb);
    memcpy(h, a_xy, W2 * 8);
    h[W2] = a_inf ? 1 : 0;
    memcpy(h + W2 + 1, b_xy, W2 * 8);
    h[2 * W2 + 1] = b_inf ? 1 : 0;
    const size_t gofs = (rb + 15) & ~(size_t)15;        // the sum (written with 128-bit stores) sits at the aligned start
    char* d = (char*)c->gather.get(gofs + 2 * rb);
    h2d(d + gofs, h, 2 * rb, c->stream);
    points_sum_run(c, curve, group, (const uint64_t*)(d + gofs), 2, (uint64_t*)d, c->stream);
    ZKM_CUDA(cudaMemcpyAsync(h + 2 * (W2 + 1), d, rb, cudaMemcpyDeviceToHost, c->stream));
    ZKM_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(out_xy, h + 2 * (W2 + 1), W2 * 8);
    *out_inf = rec_flag(h[2 * (W2 + 1) + W2]);
}

int32_t zkm_kzg_commit_hiding(uint64_t handle_g, uint64_t handle_gamma_g, const uint64_t* coeffs, size_t n,
                              const uint64_t* blinding_coeffs, size_t nb, uint64_t* out_xy, uint8_t* out_inf) {
    return guarded([&] {
        if (!out_xy || !out_inf) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
        std::shared_ptr<BasesReg> rg = lookup(handle_g, 0, 0);
        std::shared_ptr<BasesReg> rh = lookup(handle_gamma_g, 0, nb);
        if (rg->curve != rh->curve || rh->group != 1) ZKM_FAIL(ZKM_ERR_ARG, "powers_of_g and powers_of_gamma_g must be G1 bases of one curve");
        const size_t W2 = 2 * (size_t)coord_words(rg->curve, 1);
        std::vector<uint64_t> c_xy(W2), r_xy(W2);
        uint8_t c_inf = 0, r_inf = 0;
        int32_t rc2 = ZKM_OK;
        std::string msg2;
        // the two MSMs run concurrently (separate lanes); upstream: commitment.add_assign_mixed(&random_commitment)
        std::thread t2([&] {
            rc2 = guarded([&] { msm_reg_host(rh, 0, blinding_coeffs, nb, r_xy.data(), &r_inf, true); });
            if (rc2 != ZKM_OK) msg2 = t_err;
        });
        int32_t rc1 = guarded([&] { kzg_commit_impl(handle_g, coeffs, n, c_xy.data(), &c_inf); });
        t2.join();
        if (rc1 != ZKM_OK) throw ZkmError{rc1};
        if (rc2 != ZKM_OK) {
            set_error("hiding term: %s", msg2.c_str());
            throw ZkmError{rc2};
        }
        add_two_points(rg->curve, 1, c_xy.data(), c_inf, r_xy.data(), r_inf, out_xy, out_inf);
    });
}

// witness polynomial of `coeffs` at `point` on the device, then its commitment; returns p(point) through eval_out
static void kzg_open_one(const std::shared_ptr<BasesReg>& r, const uint64_t* coeffs, size_t n, const uint64_t* point,
                         uint64_t* out_xy, uint8_t* out_inf, uint64_t* eval_out) {
    const size_t S = (size_t)fr_words(r->curve), sb = S * 8;
    const size_t W2 = 2 * (size_t)coord_words(r->curve, 1), rb = (W2 + 1) * 8;
    if (n && n - 1 > r->n) ZKM_FAIL(ZKM_ERR_HANDLE, "witness polynomial of %zu coefficients exceeds the %zu registered powers", n - 1, r->n);
    const size_t nq = n ? n - 1 : 0;
    std::vector<Job> jobs = split_jobs(*r, 0, nq);
    const int dev = jobs.empty() ? 0 : jobs[0].part->dev;
    LaneGuard lane(dev);
    Context* c = lane.c;
    ZKM_CUDA(cudaSetDevice(c->device));
    StreamScope scope(c, c->stream);
    char* d = (char*)c->io_scalars.get((n + 2) * sb);
    uint64_t* d_p = (uint64_t*)d;
    uint64_t* d_z = (uint64_t*)(d + n * sb);
    uint64_t* d_ev = (uint64_t*)(d + (n + 1) * sb);
    uint64_t* d_q = (uint64_t*)c->ntt_a.get((n ? n : 1) * sb);
    h2d(d_p, coeffs, n * sb, c->stream);
    h2d(d_z, point, sb, c->stream);
    kzg_quotient_run(c, r->curve, d_p, n, d_z, d_q, d_ev, c->stream);
    uint64_t* h = (uint64_t*)c->pin_out.get(rb + sb);
    if (eval_out) ZKM_CUDA(cudaMemcpyAsync(h + W2 + 1, d_ev, sb, cudaMemcpyDeviceToHost, c->stream));
    uint64_t* d_out = (uint64_t*)c->io_out.get(rb);
    if (jobs.size() <= 1) {
        fr_into_repr_run(c, r->curve, d_q, d_q, (uint64_t)nq, c->stream);          // convert_to_bigints
        if (jobs.empty()) msm_run(c, r->curve, 1, nullptr, nullptr, nullptr, 0, d_out, c->stream);
        else run_part(c, *r, jobs[0], d_q, d_out, c->stream);
        ZKM_CUDA(cudaMemcpyAsync(h, d_out, rb, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
        memcpy(out_xy, h, W2 * 8);
        *out_inf = rec_flag(h[W2]);
    } else {
        // powers sharded over several devices: the quotient (Montgomery) goes back to the host and through the sharded path
        std::vector<uint64_t> q(nq * S);
        ZKM_CUDA(cudaMemcpyAsync(q.data(), d_q, nq * sb, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
        msm_reg_host(r, 0, q.data(), nq, out_xy, out_inf, true);
    }
    if (eval_out) memcpy(eval_out, h + W2 + 1, sb);
}

int32_t zkm_kzg_open(uint64_t handle_g, uint64_t handle_gamma_g, const uint64_t* coeffs, size_t n,
                     const uint64_t* blinding_coeffs, size_t nb, const uint64_t* point, uint64_t* out_w_xy, uint8_t* out_w_inf,
                     uint64_t* out_random_v) {
    return guarded([&] {
        if (!point || !out_w_xy || !out_w_inf || (n && !coeffs)) ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
        std::shared_ptr<BasesReg> rg = lookup(handle_g, 0, 0);
        if (rg->group != 1) ZKM_FAIL(ZKM_ERR_ARG, "KZG powers must be G1 bases");
        const size_t W2 = 2 * (size_t)coord_words(rg->curve, 1);
        if (!handle_gamma_g || nb == 0) {
            kzg_open_one(rg, coeffs, n, point, out_w_xy, out_w_inf, nullptr);
            if (out_random_v) memset(out_random_v, 0, (size_t)fr_words(rg->curve) * 8);
            return;
        }
        if (!blinding_coeffs) ZKM_FAIL(ZKM_ERR_ARG, "null blinding polynomial");
        std::shared_ptr<BasesReg> rh = lookup(handle_gamma_g, 0, 0);
        if (rh->curve != rg->curve || rh->group != 1) ZKM_FAIL(ZKM_ERR_ARG, "powers_of_gamma_g must be G1 bases of the same curve");
        std::vector<uint64_t> w_xy(W2), h_xy(W2);
        uint8_t w_inf = 0, h_inf = 0;
        int32_t rc2 = ZKM_OK;
        std::string msg2;
        std::thread t2([&] {      // hiding witness polynomial + blinding_polynomial.evaluate(point), concurrently
            rc2 = guarded([&] { kzg_open_one(rh, blinding_coeffs, nb, point, h_xy.data(), &h_inf, out_random_v); });
            if (rc2 != ZKM_OK) msg2 = t_err;
        });
        int32_t rc1 = guarded([&] { kzg_open_one(rg, coeffs, n, point, w_xy.data(), &w_inf, nullptr); });
        t2.join();
        if (rc1 != ZKM_OK) throw ZkmError{rc1};
        if (rc2 != ZKM_OK) {
            set_error("hiding witness: %s", msg2.c_str());
            throw ZkmError{rc2};
        }
        add_two_points(rg->curve, 1, w_xy.data(), w_inf, h_xy.data(), h_inf, out_w_xy, out_w_inf);
    });
}

int32_t zkm_msm_registered_device(uint64_t handle, size_t offset, const uint64_t* d_scalars, size_t n, uint64_t* d_out,
                                  void* stream) {
    return guarded([&] {
        if (!d_out || (n && !d_scalars)) ZKM_FAIL(ZKM_ERR_ARG, "null device pointer");
        std::vector<DevItem> items{DevItem{lookup(handle, offset, n), offset, n, d_scalars, d_out}};
        const int home = home_device_of(d_out);
        msm_items_device(items, home, call_stream(home, stream));
    });
}

// `count` MSMs over registered bases issued CONCURRENTLY: one host thread + one lane + the lane's own
// stream per item, all ordered after the current point of `stream` and joined back into it.  This is the
// create_proof pattern (four G1 MSMs and the G2 one, ark-groth16 0.3.0 src/prover.rs): upstream runs them
// back to back; here the G2 MSM and the serial tails of the G1 ones overlap.
int32_t zkm_msm_batch_registered_device(int32_t count, const uint64_t* handles, const size_t* offsets,
                                        const uint64_t* const* d_scalars, const size_t* n, uint64_t* const* d_outs,
                                        void* stream) {
    return guarded([&] {
        if (count < 0 || count > ZKM_NUM_LANES - 2) ZKM_FAIL(ZKM_ERR_ARG, "count must be 0..%d", ZKM_NUM_LANES - 2);
        if (count && (!handles || !offsets || !d_scalars || !n || !d_outs)) ZKM_FAIL(ZKM_ERR_ARG, "null argument array");
        if (count == 0) return;
        std::vector<DevItem> items;
        for (int i = 0; i < count; i++) {
            if (!d_outs[i] || (n[i] && !d_scalars[i])) ZKM_FAIL(ZKM_ERR_ARG, "item %d: null device pointer", i);
            items.push_back(DevItem{lookup(handles[i], offsets[i], n[i]), offsets[i], n[i], d_scalars[i], d_outs[i]});
        }
        const int home = home_device_of(d_outs[0]);
        msm_items_device(items, home, call_stream(home, stream));
    });
}

int32_t zkm_points_sum_device(int32_t curve, int32_t group, const uint64_t* d_points, size_t m, uint64_t* d_out,
                              void* stream) {
    return guarded([&] {
        check_curve_group(curve, group);
        if (!d_out || (m && !d_points)) ZKM_FAIL(ZKM_ERR_ARG, "null device pointer");
        const int home = home_device_of(d_out);
        cudaStream_t s = call_stream(home, stream);
        LaneGuard lane(home, s);
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        points_sum_run(c, curve, group, d_points, m, d_out, s);
    });
}

int32_t zkm_ntt(int32_t curve, uint64_t* data, uint32_t log_n, int32_t inverse, int32_t coset) {
    return guarded([&] {
        if (!curve_known(curve)) ZKM_FAIL(ZKM_ERR_ARG, "unknown curve id %d", curve);
        if (!data) ZKM_FAIL(ZKM_ERR_ARG, "null data");
        const int adicity = fr_two_adicity(curve);
        if ((int)log_n > adicity) ZKM_FAIL(ZKM_ERR_DOMAIN, "log_n %u exceeds the two-adicity %d of Fr", log_n, adicity);
        if (log_n > 30) ZKM_FAIL(ZKM_ERR_ARG, "log_n %u: domains above 2^30 are not supported by this build", log_n);
        LaneGuard lane(pick_host_call_device());
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        const size_t bytes = ((size_t)fr_words(curve) * 8) << log_n;
        StreamScope scope(c, c->stream);
        uint64_t* d_a = (uint64_t*)c->io_scalars.get(bytes);
        uint64_t* d_b = (uint64_t*)c->ntt_b.get(bytes);
        h2d(d_a, data, bytes, c->stream);
        ntt_run(c, curve, d_a, d_b, log_n, inverse != 0, coset != 0, c->stream);
        ZKM_CUDA(cudaMemcpyAsync(data, d_b, bytes, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
    });
}

int32_t zkm_ntt_device(int32_t curve, const uint64_t* d_in, uint64_t* d_out, uint32_t log_n, int32_t inverse,
                       int32_t coset, void* stream) {
    return guarded([&] {
        if (!d_in || !d_out) ZKM_FAIL(ZKM_ERR_ARG, "null device pointer");
        const int home = home_device_of(d_out);
        cudaStream_t s = call_stream(home, stream);
        LaneGuard lane(home, s);
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        StreamScope scope(c, s);
        ntt_run(c, curve, d_in, d_out, log_n, inverse != 0, coset != 0, s);
    });
}

int32_t zkm_fr_into_repr_device(int32_t curve, const uint64_t* d_in, uint64_t* d_out, size_t n, void* stream) {
    return guarded([&] {
        if (n && (!d_in || !d_out)) ZKM_FAIL(ZKM_ERR_ARG, "null device pointer");
        const int home = n ? home_device_of(d_out) : 0;
        cudaStream_t s = call_stream(home, stream);
        LaneGuard lane(home, s);
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        fr_into_repr_run(c, curve, d_in, d_out, (uint64_t)n, s);
    });
}

int32_t zkm_witness_map_device(int32_t curve, uint64_t* d_a, uint64_t* d_b, uint64_t* d_c, uint32_t log_n, uint64_t* d_h,
                               void* stream) {
    return guarded([&] {
        if (!d_a || !d_b || !d_c || !d_h) ZKM_FAIL(ZKM_ERR_ARG, "null device pointer");
        const int home = home_device_of(d_h);
        cudaStream_t s = call_stream(home, stream);
        LaneGuard lane(home, s);
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        StreamScope scope(c, s);
        witness_map_run(c, curve, d_a, d_b, d_c, log_n, d_h, s);
    });
}

int32_t zkm_witness_map(int32_t curve, const uint64_t* a, const uint64_t* b, const uint64_t* cc, uint32_t log_n,
                        uint64_t* h_out) {
    return guarded([&] {
        if (!a || !b || !cc || !h_out) ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
        if (!curve_known(curve)) ZKM_FAIL(ZKM_ERR_ARG, "unknown curve id %d", curve);
        const int adicity = fr_two_adicity(curve);
        if ((int)log_n > adicity) ZKM_FAIL(ZKM_ERR_DOMAIN, "log_n %u exceeds the two-adicity %d of Fr", log_n, adicity);
        if (log_n > 28) ZKM_FAIL(ZKM_ERR_ARG, "log_n %u: witness maps above 2^28 are not supported by this build", log_n);
        LaneGuard lane(pick_host_call_device());
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        const size_t bytes = ((size_t)fr_words(curve) * 8) << log_n;
        StreamScope scope(c, c->stream);
        char* d = (char*)c->io_scalars.get(4 * bytes);
        h2d(d, a, bytes, c->stream);
        h2d(d + bytes, b, bytes, c->stream);
        h2d(d + 2 * bytes, cc, bytes, c->stream);
        witness_map_run(c, curve, (uint64_t*)d, (uint64_t*)(d + bytes), (uint64_t*)(d + 2 * bytes), log_n,
                        (uint64_t*)(d + 3 * bytes), c->stream);
        ZKM_CUDA(cudaMemcpyAsync(h_out, d + 3 * bytes, bytes, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
    });
}

int32_t zkm_domain_constants(int32_t curve, uint32_t log_n, uint64_t* out5x4) {
    return guarded([&] {
        LaneGuard lane(0);
        Context* c = lane.c;
        if (!out5x4) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
        ZKM_CUDA(cudaSetDevice(c->device));
        StreamScope scope(c, c->stream);
        ntt_domain_constants(c, curve, log_n, out5x4);
    });
}

int32_t zkm_set_option(const char* key, int64_t value) {
    return guarded([&] {
        if (!key) ZKM_FAIL(ZKM_ERR_ARG, "null key");
        std::lock_guard<std::mutex> lk(g_lane_mu);      // lanes snapshot the options under the same mutex
        if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
        Options& o = g->opt;
        if (!strcmp(key, "msm_window_bits")) {
            if (value < 0 || value > 24) ZKM_FAIL(ZKM_ERR_ARG, "msm_window_bits must be 0 (auto) or 2..24");
            o.msm_window_bits = (int)value;
        } else if (!strcmp(key, "msm_chunk")) {
            if (value < 0 || value > 1024) ZKM_FAIL(ZKM_ERR_ARG, "msm_chunk must be 0 (auto) or 1..1024");
            o.msm_chunk = (int)value;
        } else if (!strcmp(key, "ntt_max_radix_log")) {
            if (value < 6 || value > 12) ZKM_FAIL(ZKM_ERR_ARG, "ntt_max_radix_log must be 6..12");
            o.ntt_max_radix_log = (int)value;
        } else if (!strcmp(key, "profile")) {
            o.profile = value ? 1 : 0;
        } else if (!strcmp(key, "msm_affine_levels")) {
            if (value < -1 || value > 24) ZKM_FAIL(ZKM_ERR_ARG, "msm_affine_levels must be -1 (auto) or 0..24");
            o.msm_affine_levels = (int)value;
        } else if (!strcmp(key, "msm_pair_m")) {
            if (value < 2 || value > 4096) ZKM_FAIL(ZKM_ERR_ARG, "msm_pair_m must be 2..4096");
            o.msm_pair_m = (int)value;
        } else if (!strcmp(key, "msm_pair_m2")) {
            if (value < 2 || value > 4096) ZKM_FAIL(ZKM_ERR_ARG, "msm_pair_m2 must be 2..4096");
            o.msm_pair_m2 = (int)value;
        } else if (!strcmp(key, "msm_prefetch_fwd") || !strcmp(key, "msm_prefetch_bwd")) {
            if (value < 0 || value > 64) ZKM_FAIL(ZKM_ERR_ARG, "%s must be 0 (off) .. 64 pairs ahead", key);
            (key[13] == 'f' ? o.msm_prefetch_fwd : o.msm_prefetch_bwd) = (int)value;
        } else if (!strcmp(key, "msm_xarr")) {
            o.msm_xarr = value ? 1 : 0;
        } else if (!strcmp(key, "msm_fold")) {
            if (value != 0 && (value < 2 || value > 1024)) ZKM_FAIL(ZKM_ERR_ARG, "msm_fold must be 0 (auto) or 2..1024");
            o.msm_fold = (int)value;
        } else if (!strcmp(key, "msm_precompute")) {
            o.msm_precompute = value ? 1 : 0;
        } else if (!strcmp(key, "msm_cache")) {
            if (value < 0 || value > 2) ZKM_FAIL(ZKM_ERR_ARG, "msm_cache must be 0 (off), 1 (sampled fingerprint) or 2 (full fingerprint)");
            o.msm_cache = (int)value;
        } else if (!strcmp(key, "msm_cache_precompute")) {
            o.msm_cache_precompute = value ? 1 : 0;
        } else if (!strcmp(key, "msm_cache_max_mb")) {
            if (value < 0) ZKM_FAIL(ZKM_ERR_ARG, "msm_cache_max_mb must be >= 0");
            o.msm_cache_max_mb = value;
        } else if (!strcmp(key, "host_wait")) {
            if (value < 0 || value > 2) ZKM_FAIL(ZKM_ERR_ARG, "host_wait must be 0 (auto), 1 (spin) or 2 (block)");
            o.host_wait = (int)value;
        } else if (!strcmp(key, "spread_host_calls")) {
            o.spread_host_calls = value ? 1 : 0;
        } else {
            ZKM_FAIL(ZKM_ERR_ARG, "unknown option '%s'", key);
        }
    });
}

int32_t zkm_msm_cache_clear(void) {
    return guarded([&] {
        if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
        std::map<Global::CacheKey, Global::CacheEntry> old;
        {
            std::lock_guard<std::mutex> lk(g->cache_mu);
            old.swap(g->cache);
            g->cache_bytes = 0;
        }
    });
}

int32_t zkm_msm_cache_stats(uint64_t* out4) {
    return guarded([&] {
        if (!out4) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
        if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
        std::lock_guard<std::mutex> lk(g->cache_mu);
        out4[0] = g->cache_hits;
        out4[1] = g->cache_misses;
        out4[2] = g->cache.size();
        out4[3] = g->cache_bytes;
    });
}

// lane that ran the last profiled MSM (set by msm_run through note_profiled_lane)
static Context* profiled_lane() {
    if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
    Context* c = g->last_prof.load();
    if (!c || !c->pev_valid) ZKM_FAIL(ZKM_ERR_ARG, "no profiled MSM yet (set option \"profile\" to 1 first)");
    return c;
}

int32_t zkm_profile_last_msm(double* ms_out6) {
    return guarded([&] {
        if (!ms_out6) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
        Context* c = profiled_lane();
        ZKM_CUDA(cudaSetDevice(c->device));
        ZKM_CUDA(cudaEventSynchronize(c->pev[6]));
        for (int i = 0; i < 6; i++) {
            float ms = 0.f;
            ZKM_CUDA(cudaEventElapsedTime(&ms, c->pev[i], c->pev[i + 1]));
            ms_out6[i] = ms;
        }
    });
}

int32_t zkm_profile_last_msm_counts(uint64_t* out16) {
    return guarded([&] {
        if (!out16) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
        Context* c = profiled_lane();
        for (int i = 0; i < 16; i++) out16[i] = c->pcount[i];
    });
}

uint64_t zkm_launch_count(int32_t reset) {
    uint64_t v = g_launches.load();
    if (reset) g_launches.store(0);
    return v;
}

int32_t zkm_msm_window_bits(int32_t curve, int32_t group, size_t n) {
    {
        std::lock_guard<std::mutex> lk(g_lane_mu);
        if (g && g->opt.msm_window_bits > 0) return g->opt.msm_window_bits;
    }
    return msm_auto_window_bits(curve, group, n);
}

int32_t zkm_fixed_base_msm(int32_t curve, int32_t group, const uint64_t* base_xy, uint8_t base_inf, const uint64_t* scalars,
                           size_t n, uint64_t* out_xy, uint8_t* out_inf) {
    return guarded([&] {
        check_curve_group(curve, group);
        if (n && (!base_xy || !scalars || !out_xy || !out_inf)) ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
        LaneGuard lane(pick_host_call_device());
        Context* c = lane.c;
        if (n == 0) return;
        ZKM_CUDA(cudaSetDevice(c->device));
        const size_t sbytes = (size_t)fr_words(curve) * 8, xyb = 2 * (size_t)coord_words(curve, group) * 8;
        StreamScope scope(c, c->stream);
        uint64_t* d_scal = (uint64_t*)c->io_scalars.get(n * sbytes);
        uint64_t* d_xy = (uint64_t*)c->io_bases.get(n * xyb);
        uint8_t* d_inf = (uint8_t*)c->io_inf.get(n);
        uint32_t* d_flag = (uint32_t*)c->io_out.get(16);
        ZKM_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(uint32_t), c->stream));
        h2d(d_scal, scalars, n * sbytes, c->stream);
        fixed_base_run(c, curve, group, base_xy, base_inf != 0, d_scal, n, d_xy, d_inf, d_flag, c->stream);
        uint32_t* h_flag = (uint32_t*)c->pin_in.get(16);
        ZKM_CUDA(cudaMemcpyAsync(out_xy, d_xy, n * xyb, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaMemcpyAsync(out_inf, d_inf, n, cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaMemcpyAsync(h_flag, d_flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        ZKM_CUDA(cudaStreamSynchronize(c->stream));
        if (*h_flag) ZKM_FAIL(ZKM_ERR_SCALAR_RANGE, "a scalar-field element is not below the modulus");
    });
}

int32_t zkm_fixed_base_msm_device(int32_t curve, int32_t group, const uint64_t* base_xy, uint8_t base_inf, const uint64_t* d_scalars,
                                  size_t n, uint64_t* d_out_xy, uint8_t* d_out_inf, void* stream) {
    return guarded([&] {
        check_curve_group(curve, group);
        if (n && (!base_xy || !d_scalars || !d_out_xy || !d_out_inf)) ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
        if (((uintptr_t)d_scalars | (uintptr_t)d_out_xy) & 15) ZKM_FAIL(ZKM_ERR_ARG, "device pointers must be 16-byte aligned");
        if (device_count_initialised() == 0) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
        const int home = n ? home_device_of(d_out_xy) : 0;
        cudaStream_t s = call_stream(home, stream);
        LaneGuard lane(home, s);
        Context* c = lane.c;
        if (n == 0) return;
        ZKM_CUDA(cudaSetDevice(c->device));
        StreamScope scope(c, s);
        fixed_base_run(c, curve, group, base_xy, base_inf != 0, d_scalars, n, d_out_xy, d_out_inf, nullptr, s);
    });
}

int32_t zkm_groth16_pk_create(int32_t curve, const uint64_t* handles, const uint64_t* g1_xy, const uint8_t* g1_inf,
                              const uint64_t* g2_xy, const uint8_t* g2_inf, uint64_t* pk_out) {
    return guarded([&] {
        if (!pk_out) ZKM_FAIL(ZKM_ERR_ARG, "null pk_out");
        *pk_out = g16_create(curve, handles, g1_xy, g1_inf, g2_xy, g2_inf);
    });
}

int32_t zkm_groth16_pk_release(uint64_t pk) {
    return guarded([&] {
        if (!g) ZKM_FAIL(ZKM_ERR_NOT_INIT, "zkm_init() has not been called (or failed)");
        std::shared_ptr<G16Key> keep;     // destroyed (device memory freed) outside the registry lock
        std::lock_guard<std::mutex> rl(g->reg_mu);
        auto it = g->pks.find(pk);
        if (it == g->pks.end()) ZKM_FAIL(ZKM_ERR_HANDLE, "unknown Groth16 proving key %llu", (unsigned long long)pk);
        keep = std::move(it->second);
        g->pks.erase(it);
    });
}

int32_t zkm_groth16_prove(uint64_t pk, const uint64_t* a, const uint64_t* b, const uint64_t* c, uint32_t log_n,
                          const uint64_t* assignment, size_t num_inputs, size_t num_aux, const uint64_t* r, const uint64_t* s,
                          uint64_t* out_a_xy, uint8_t* out_a_inf, uint64_t* out_b_xy, uint8_t* out_b_inf, uint64_t* out_c_xy,
                          uint8_t* out_c_inf) {
    return guarded([&] {
        if (!a || !b || !c || !r || !s || (num_inputs + num_aux && !assignment)) ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
        if (!out_a_xy || !out_a_inf || !out_b_xy || !out_b_inf || !out_c_xy || !out_c_inf) ZKM_FAIL(ZKM_ERR_ARG, "null output pointer");
        std::shared_ptr<G16Key> key = g16_lookup(pk);
        g16_check(*key, log_n, num_inputs, num_aux);
        const G16Host host{a, b, c, assignment, out_a_xy, out_b_xy, out_c_xy, out_a_inf, out_b_inf, out_c_inf};
        g16_prove(*key, pick_host_call_device(), nullptr, log_n, num_inputs, num_aux, r, s, nullptr, nullptr, nullptr, nullptr,
                  nullptr, &host);
    });
}

int32_t zkm_groth16_prove_device(uint64_t pk, uint64_t* d_a, uint64_t* d_b, uint64_t* d_c, uint32_t log_n,
                                 const uint64_t* d_assignment, size_t num_inputs, size_t num_aux, const uint64_t* r,
                                 const uint64_t* s, uint64_t* d_out, void* stream) {
    return guarded([&] {
        if (!d_a || !d_b || !d_c || !d_out || !r || !s || (num_inputs + num_aux && !d_assignment))
            ZKM_FAIL(ZKM_ERR_ARG, "null pointer");
        std::shared_ptr<G16Key> key = g16_lookup(pk);
        g16_check(*key, log_n, num_inputs, num_aux);
        const int home = home_device_of(d_out);
        g16_prove(*key, home, call_stream(home, stream), log_n, num_inputs, num_aux, r, s, d_a, d_b, d_c, d_assignment, d_out,
                  nullptr);
    });
}

int32_t zkm_testgen_progression_device(int32_t curve, int32_t group, uint64_t a0, uint64_t d, size_t n,
                                       uint64_t* d_bases_xy, void* stream) {
    return guarded([&] {
        check_curve_group(curve, group);
        if (n && !d_bases_xy) ZKM_FAIL(ZKM_ERR_ARG, "null device pointer");
        const int home = n ? home_device_of(d_bases_xy) : 0;
        cudaStream_t s = call_stream(home, stream);
        LaneGuard lane(home, s);
        Context* c = lane.c;
        ZKM_CUDA(cudaSetDevice(c->device));
        testgen_progression(c, curve, group, a0, d, n, d_bases_xy, s);
    });
}

}  // extern "C"

namespace zkm {
void note_profiled_lane(Context* c) {
    if (g) g->last_prof.store(c);
}
}  // namespace zkm
