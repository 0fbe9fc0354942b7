// pipeline.cu -- the host-buffer pipeline behind the NumPy-level API (vr180_ctx_*, include/vr180_b200.h).
//
// Replaces the body of the reference's apply() / apply_lr() for arrays that live in HOST memory
// (/root/reference/src/vr180_convert/remapper.py:379-398: one radius, ONE map, cv.remap for every image of the call;
// :474-484 + :518: both eyes + np.concatenate): upload -> [get_radius] -> warp -> download for a batch of frames,
// with the copies of neighbouring chunks overlapped on three streams and a ring of kSlots device buffers.
//
// Host buffers that are page-locked (vr180_host_alloc / vr180_host_register) are DMA'd directly.  Pageable buffers
// (plain NumPy arrays) are staged through a pinned ring owned by the context: a small pool of copy threads packs
// chunk k + 1 while the GPU works on chunk k, and a drain thread unpacks finished chunks into the caller's arrays,
// so the pipeline never degrades to the driver's single-threaded pageable memcpy path.
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <cstdlib>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "common.cuh"

namespace vr180 {
void stream_copy_avx2(uint8_t* d, const uint8_t* s, size_t n);  // hostcopy.cpp (g++ -mavx2)
}
using namespace vr180;

namespace {

constexpr int kSlots = 3;
constexpr size_t kChunkBytes = (size_t)192 << 20;  // source + destination bytes per pipeline chunk
constexpr size_t kBandBytes = (size_t)8 << 20;     // rows packed and uploaded as one band of the first chunk
constexpr size_t kCopyUnit = (size_t)1 << 20;      // bytes one copy-thread task moves

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return VR180_OK;
        release();
        const size_t want = bytes + bytes / 8;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            p = nullptr;
            set_cuda_error(e, "cudaMalloc");
            return e == cudaErrorMemoryAllocation ? VR180_ERR_NOMEM : VR180_ERR_CUDA;
        }
        cap = want;
        return VR180_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct PinBuf {  // page-locked host staging
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return VR180_OK;
        release();
        cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
        if (e != cudaSuccess) {
            p = nullptr;
            set_cuda_error(e, "cudaHostAlloc");
            return e == cudaErrorMemoryAllocation ? VR180_ERR_NOMEM : VR180_ERR_CUDA;
        }
        cap = bytes;
        return VR180_OK;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// Copy threads: run(n, fn) executes fn(0) .. fn(n - 1) on the workers and the calling thread, and returns when all
// are done.  Concurrent run() calls (stage-in on the caller's thread, copy-out on the drain thread) share the workers.
class CopyPool {
  public:
    explicit CopyPool(int n_threads) {
        for (int i = 0; i < n_threads; ++i) th_.emplace_back([this] { loop(); });
    }
    ~CopyPool() {
        {
            std::lock_guard<std::mutex> l(m_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto& t : th_) t.join();
    }
    int threads() const { return (int)th_.size(); }
    void run(int n, const std::function<void(int)>& fn) {
        if (n <= 0) return;
        auto job = std::make_shared<Job>();
        job->fn = &fn;
        job->n = n;
        const int helpers = std::min<int>((int)th_.size(), n - 1);
        if (helpers > 0) {
            {
                std::lock_guard<std::mutex> l(m_);
                for (int i = 0; i < helpers; ++i) q_.push_back(job);
            }
            cv_.notify_all();
        }
        work(*job);
        std::unique_lock<std::mutex> l(job->m);
        job->cv.wait(l, [&] { return job->done == job->n; });
    }

  private:
    struct Job {
        const std::function<void(int)>* fn;
        int n;
        std::atomic<int> next{0};
        int done = 0;
        std::mutex m;
        std::condition_variable cv;
    };
    static void work(Job& j) {
        int mine = 0;
        for (;;) {
            const int i = j.next.fetch_add(1, std::memory_order_relaxed);
            if (i >= j.n) break;
            (*j.fn)(i);
            ++mine;
        }
        if (mine) {
            std::lock_guard<std::mutex> l(j.m);
            j.done += mine;
            if (j.done == j.n) j.cv.notify_all();
        }
    }
    void loop() {
        for (;;) {
            std::shared_ptr<Job> j;
            {
                std::unique_lock<std::mutex> l(m_);
                cv_.wait(l, [&] { return stop_ || !q_.empty(); });
                if (stop_ && q_.empty()) return;
                j = q_.front();
                q_.pop_front();
            }
            work(*j);
        }
    }
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<std::shared_ptr<Job>> q_;
    bool stop_ = false;
};

int default_copy_threads() {
    if (const char* e = getenv("VR180_COPY_THREADS")) {
        const int n = atoi(e);
        if (n >= 1) return std::min(n, 64);
    }
    // packing a pageable frame is a plain memcpy (~6-10 GB/s per core); the PCIe link takes ~50 GB/s each way, so a GPU
    // needs ~8 copy threads to be fed from pageable memory.  Half the cores, at most 12.
    const unsigned hw = std::thread::hardware_concurrency();
    return (int)std::max(2u, std::min(12u, hw / 2));
}

bool is_page_locked(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// Large copies into / out of the page-locked ring: streaming stores where the CPU has them (hostcopy.cpp)
void copy_bytes(uint8_t* dst, const uint8_t* src, size_t n) {
    static const bool nt = [] {
        const char* e = getenv("VR180_NT_COPY");
        if (e && atoi(e) == 0) return false;
#if defined(__x86_64__)
        return __builtin_cpu_supports("avx2") != 0;
#else
        return false;
#endif
    }();
    if (nt && n >= ((size_t)8 << 10)) stream_copy_avx2(dst, src, n);
    else memcpy(dst, src, n);
}

// a 2-D byte copy (rows x row_bytes, independent pitches), split into ~kCopyUnit tasks
struct Copy2D {
    uint8_t* dst;
    const uint8_t* src;
    size_t dst_pitch, src_pitch, row_bytes, rows;
};

void run_copies(CopyPool& pool, const std::vector<Copy2D>& copies) {
    struct Unit {
        int c;
        size_t r0, r1;
    };
    std::vector<Unit> units;
    for (int c = 0; c < (int)copies.size(); ++c) {
        const Copy2D& k = copies[c];
        const size_t rows_per = std::max<size_t>(1, kCopyUnit / std::max<size_t>(k.row_bytes, 1));
        for (size_t r = 0; r < k.rows; r += rows_per) units.push_back({c, r, std::min(k.rows, r + rows_per)});
    }
    pool.run((int)units.size(), [&](int i) {
        const Unit& u = units[i];
        const Copy2D& k = copies[u.c];
        if (k.dst_pitch == k.row_bytes && k.src_pitch == k.row_bytes) {
            copy_bytes(k.dst + u.r0 * k.dst_pitch, k.src + u.r0 * k.src_pitch, (u.r1 - u.r0) * k.row_bytes);
        } else {
            for (size_t r = u.r0; r < u.r1; ++r) copy_bytes(k.dst + r * k.dst_pitch, k.src + r * k.src_pitch, k.row_bytes);
        }
    });
}

struct Slot {
    DevBuf src[2], dst, merged;
    PinBuf h_src[2], h_dst;
    cudaEvent_t ev_h2d = nullptr, ev_comp = nullptr, ev_d2h = nullptr;
};

}  // namespace

struct vr180_ctx {
    int device = 0;
    cudaStream_t s_h2d = nullptr, s_comp = nullptr, s_d2h = nullptr;
    Slot slot[kSlots];
    DevBuf maps[2][2], trans, radius;
    // identity of the cached FLOAT2 maps: caller's key + what was actually uploaded
    uint64_t map_key = 0;
    size_t map_elems = 0;
    int map_n = 0;
    const float* map_ptr[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
    std::unique_ptr<CopyPool> pool;
    // drain thread: unpacks finished chunks from the pinned ring into the caller's (pageable) destination
    std::thread drain;
    std::mutex dm;
    std::condition_variable dcv;
    std::deque<std::function<void()>> dq;
    long long drained = 0, queued = 0;
    bool dstop = false;
    std::mutex mu;

    CopyPool& copy_pool(int threads) {
        if (!pool || (threads > 0 && pool->threads() != threads - 1))
            pool.reset(new CopyPool(std::max(0, (threads > 0 ? threads : default_copy_threads()) - 1)));
        return *pool;
    }
    void start_drain() {
        if (drain.joinable()) return;
        drain = std::thread([this] {
            cudaSetDevice(device);
            for (;;) {
                std::function<void()> fn;
                {
                    std::unique_lock<std::mutex> l(dm);
                    dcv.wait(l, [&] { return dstop || !dq.empty(); });
                    if (dq.empty()) return;
                    fn = std::move(dq.front());
                    dq.pop_front();
                }
                fn();
                {
                    std::lock_guard<std::mutex> l(dm);
                    ++drained;
                }
                dcv.notify_all();
            }
        });
    }
    long long push_drain(std::function<void()> fn) {
        long long ticket;
        {
            std::lock_guard<std::mutex> l(dm);
            dq.push_back(std::move(fn));
            ticket = ++queued;
        }
        dcv.notify_all();
        return ticket;
    }
    void wait_drained(long long ticket) {
        std::unique_lock<std::mutex> l(dm);
        dcv.wait(l, [&] { return drained >= ticket; });
    }
    void stop_drain() {
        if (!drain.joinable()) return;
        {
            std::lock_guard<std::mutex> l(dm);
            dstop = true;
        }
        dcv.notify_all();
        drain.join();
    }
};

static void ctx_free(vr180_ctx* c) {
    c->stop_drain();
    for (Slot& s : c->slot) {
        for (int v = 0; v < 2; ++v) {
            s.src[v].release();
            s.h_src[v].release();
        }
        s.dst.release();
        s.merged.release();
        s.h_dst.release();
        if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
        if (s.ev_comp) cudaEventDestroy(s.ev_comp);
        if (s.ev_d2h) cudaEventDestroy(s.ev_d2h);
    }
    for (int v = 0; v < 2; ++v)
        for (int k = 0; k < 2; ++k) c->maps[v][k].release();
    c->trans.release();
    c->radius.release();
    if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
    if (c->s_comp) cudaStreamDestroy(c->s_comp);
    if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
    delete c;
}

extern "C" {

int vr180_ctx_create(int device, vr180_ctx_t** out) {
    if (!out) return VR180_ERR_INVALID_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        return VR180_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) return VR180_ERR_INVALID_ARG;
    DeviceGuard g(device);
    if (!g.ok) return VR180_ERR_CUDA;
    vr180_ctx* c = new (std::nothrow) vr180_ctx();
    if (!c) return VR180_ERR_NOMEM;
    c->device = device;
    auto init = [&]() -> int {
        VR180_CUDA(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
        VR180_CUDA(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
        VR180_CUDA(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
        for (Slot& s : c->slot) {
            VR180_CUDA(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
            VR180_CUDA(cudaEventCreateWithFlags(&s.ev_comp, cudaEventDisableTiming));
            VR180_CUDA(cudaEventCreateWithFlags(&s.ev_d2h, cudaEventDisableTiming));
        }
        return VR180_OK;
    };
    const int rc = init();
    if (rc != VR180_OK) {  // nothing half-built survives a failed create
        ctx_free(c);
        return rc;
    }
    *out = c;
    return VR180_OK;
}

int vr180_ctx_destroy(vr180_ctx_t* c) {
    if (!c) return VR180_OK;
    DeviceGuard g(c->device);
    cudaDeviceSynchronize();
    ctx_free(c);
    return VR180_OK;
}

int vr180_ctx_device(const vr180_ctx_t* c) { return c ? c->device : -1; }

// The body of vr180_ctx_run after argument validation; every failure after the first enqueue returns through the
// caller, which drains all three streams and the drain thread before the job's buffers may be released.
static int ctx_run_locked(vr180_ctx* c, const vr180_host_job_t* job, const double* border_scalar) {
    // C: bytes per pixel (channels x element size); every size below is in bytes
    const int V = job->n_views, F = job->n_frames, C = job->channels * depth_bytes(job->depth);
    const bool scattered = job->src_frames[0] != nullptr;
    const size_t src_row = (size_t)job->src_cols * C, src_pitch = align_up(src_row, 16);
    const size_t src_frame = src_pitch * job->src_rows;
    // Device SBS frame: eye 1 starts at a 16-byte aligned column (a TMA box must start at a 16-byte aligned address;
    // --size 1000x1000 would otherwise push the whole launch to the per-pixel kernel).  The host frame stays dense:
    // the two eyes are then downloaded as two column segments.
    const size_t eye1_col = (V == 2 && ((size_t)job->out_w * C) % 16 != 0) ? align_up((size_t)job->out_w, 16) : (size_t)job->out_w;
    const size_t dst_row = (V == 2 ? eye1_col + job->out_w : (size_t)job->out_w) * C, dst_pitch = align_up(dst_row, 16);
    const size_t dst_frame = dst_pitch * job->out_h;
    // what goes back to the host: the SBS frame, or (merge) the anaglyph of its two halves
    const bool merge = job->merge != 0;
    const size_t out_row = merge ? (size_t)job->out_w * C : dst_row, out_pitch = align_up(out_row, 16);
    const size_t out_frame = out_pitch * job->out_h;
    struct Seg { size_t dev_col, host_col, bytes; };  // column segments (bytes) of a device row that go to the host row
    std::vector<Seg> segs;
    if (!merge && V == 2 && eye1_col != (size_t)job->out_w) {
        segs.push_back({0, 0, (size_t)job->out_w * C});
        segs.push_back({eye1_col * C, (size_t)job->out_w * C, (size_t)job->out_w * C});
    } else {
        segs.push_back({0, 0, merge ? out_row : (size_t)job->out_w * V * C});
    }

    auto src_of = [&](int v, int f) -> const uint8_t* {
        return scattered ? job->src_frames[v][f] : job->src[v] + (size_t)f * job->src_frame_stride[v];
    };
    auto dst_of = [&](int f) -> uint8_t* {
        return job->dst_frames ? job->dst_frames[f] : job->dst + (size_t)f * job->dst_frame_stride;
    };

    // page-locked buffers are DMA'd directly; pageable ones go through the pinned ring
    bool stage_in = job->staging == 1, stage_out = job->staging == 1;
    if (job->staging == 0) {
        for (int v = 0; v < V && !stage_in; ++v)
            for (int f = 0; f < (scattered ? F : 1) && !stage_in; ++f) stage_in = !is_page_locked(src_of(v, f));
        for (int f = 0; f < (job->dst_frames ? F : 1) && !stage_out; ++f) stage_out = !is_page_locked(dst_of(f));
    }

    // frames per chunk: ~kChunkBytes of traffic per chunk, at least two chunks so that copies overlap compute
    const size_t per_frame = src_frame * V + dst_frame + (merge ? out_frame : 0);
    int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)F, kChunkBytes / std::max<size_t>(per_frame, 1)));
    if (F >= 2) chunk = std::min(chunk, (F + 1) / 2);
    const int n_chunks = (F + chunk - 1) / chunk;

    int rc;
    for (int s = 0; s < std::min(kSlots, n_chunks); ++s) {
        Slot& sl = c->slot[s];
        for (int v = 0; v < V; ++v) {
            if ((rc = sl.src[v].reserve(src_frame * chunk)) != VR180_OK) return rc;
            if (stage_in && (rc = sl.h_src[v].reserve(src_frame * chunk)) != VR180_OK) return rc;
        }
        if ((rc = sl.dst.reserve(dst_frame * chunk)) != VR180_OK) return rc;
        if (merge && (rc = sl.merged.reserve(out_frame * chunk)) != VR180_OK) return rc;
        if (stage_out && (rc = sl.h_dst.reserve(out_frame * chunk)) != VR180_OK) return rc;
    }
    if ((rc = c->trans.reserve(sizeof(int32_t) * 2 * V * F)) != VR180_OK) return rc;
    if ((rc = c->radius.reserve(sizeof(double) * F)) != VR180_OK) return rc;
    CopyPool* pool = (stage_in || stage_out) ? &c->copy_pool(job->copy_threads) : nullptr;
    if (stage_out) c->start_drain();

    // maps (FLOAT2): upload once; kept while the caller's cache key AND what it points at are unchanged
    const int n_maps = (V == 2 && !job->share_map) ? 2 : 1;
    if (job->map_kind == VR180_MAPSRC_FLOAT2) {
        const size_t elems = (size_t)job->out_w * job->out_h;
        bool cached = job->maps_cache_key != 0 && job->maps_cache_key == c->map_key && c->map_elems == elems &&
                      c->map_n >= n_maps;
        for (int m = 0; m < n_maps; ++m) {
            if (!job->xmap[m] || !job->ymap[m]) return VR180_ERR_INVALID_ARG;
            cached = cached && c->map_ptr[m][0] == job->xmap[m] && c->map_ptr[m][1] == job->ymap[m];
        }
        if (!cached) {
            c->map_key = 0;
            for (int m = 0; m < n_maps; ++m) {
                if ((rc = c->maps[m][0].reserve(elems * 4)) != VR180_OK) return rc;
                if ((rc = c->maps[m][1].reserve(elems * 4)) != VR180_OK) return rc;
                VR180_CUDA(cudaMemcpyAsync(c->maps[m][0].p, job->xmap[m], elems * 4, cudaMemcpyHostToDevice, c->s_comp));
                VR180_CUDA(cudaMemcpyAsync(c->maps[m][1].p, job->ymap[m], elems * 4, cudaMemcpyHostToDevice, c->s_comp));
                c->map_ptr[m][0] = job->xmap[m];
                c->map_ptr[m][1] = job->ymap[m];
            }
            c->map_key = job->maps_cache_key;
            c->map_elems = elems;
            c->map_n = n_maps;
        }
    } else {
        for (int m = 0; m < n_maps; ++m)
            if ((rc = validate_chain(job->chain[m])) != VR180_OK) return rc;
    }

    long long slot_ticket[kSlots] = {0, 0, 0};  // drain ticket of the chunk that last used the slot's pinned dst
    for (int k = 0; k < n_chunks; ++k) {
        const int s = k % kSlots, f0 = k * chunk, nf = std::min(chunk, F - f0);
        Slot& sl = c->slot[s];
        // --- pack (pageable sources): copy threads fill the slot's pinned buffer while the GPU runs chunk k - 1 --
        // The first chunk has nothing to hide behind (and a single pair -- apply_lr on two arrays -- IS one chunk): it is
        // packed and uploaded in bands of rows, so that the DMA of a band runs while the copy threads pack the next one.
        const bool banded = stage_in && k == 0;
        if (stage_in && !banded) {
            if (k >= kSlots) VR180_CUDA(cudaEventSynchronize(sl.ev_h2d));  // the slot's previous upload has left it
            std::vector<Copy2D> cp;
            for (int v = 0; v < V; ++v)
                for (int f = 0; f < nf; ++f)
                    cp.push_back({(uint8_t*)sl.h_src[v].p + (size_t)f * src_frame, src_of(v, f0 + f), src_pitch,
                                  (size_t)job->src_pitch[v], src_row, (size_t)job->src_rows});
            run_copies(*pool, cp);
        }
        // --- upload -------------------------------------------------------------------------------------
        if (k >= kSlots) VR180_CUDA(cudaStreamWaitEvent(c->s_h2d, sl.ev_comp, 0));  // slot's previous compute done
        if (banded) {
            const size_t band_rows = std::max<size_t>(1, kBandBytes / std::max<size_t>(src_pitch, 1));
            for (int v = 0; v < V; ++v)
                for (int f = 0; f < nf; ++f)
                    for (size_t r0 = 0; r0 < (size_t)job->src_rows; r0 += band_rows) {
                        const size_t nr = std::min(band_rows, (size_t)job->src_rows - r0);
                        uint8_t* hp = (uint8_t*)sl.h_src[v].p + (size_t)f * src_frame + r0 * src_pitch;
                        run_copies(*pool, {{hp, src_of(v, f0 + f) + r0 * (size_t)job->src_pitch[v], src_pitch,
                                            (size_t)job->src_pitch[v], src_row, nr}});
                        VR180_CUDA(cudaMemcpyAsync((uint8_t*)sl.src[v].p + (size_t)f * src_frame + r0 * src_pitch, hp,
                                                   nr * src_pitch, cudaMemcpyHostToDevice, c->s_h2d));
                    }
        }
        for (int v = 0; v < V && !banded; ++v) {
            uint8_t* dp = (uint8_t*)sl.src[v].p;
            if (stage_in) {
                VR180_CUDA(cudaMemcpyAsync(dp, sl.h_src[v].p, src_frame * nf, cudaMemcpyHostToDevice, c->s_h2d));
                continue;
            }
            const size_t hp_pitch = (size_t)job->src_pitch[v];
            const bool dense_frames = !scattered && (size_t)job->src_frame_stride[v] == hp_pitch * job->src_rows;
            if (dense_frames && hp_pitch == src_pitch) {  // 1-D copy: one DMA descriptor per view and chunk
                VR180_CUDA(cudaMemcpyAsync(dp, src_of(v, f0), src_frame * nf, cudaMemcpyHostToDevice, c->s_h2d));
            } else if (dense_frames) {
                VR180_CUDA(cudaMemcpy2DAsync(dp, src_pitch, src_of(v, f0), hp_pitch, src_row, (size_t)job->src_rows * nf,
                                             cudaMemcpyHostToDevice, c->s_h2d));
            } else {
                for (int f = 0; f < nf; ++f) {
                    if (hp_pitch == src_pitch)
                        VR180_CUDA(cudaMemcpyAsync(dp + f * src_frame, src_of(v, f0 + f), src_frame, cudaMemcpyHostToDevice,
                                                   c->s_h2d));
                    else
                        VR180_CUDA(cudaMemcpy2DAsync(dp + f * src_frame, src_pitch, src_of(v, f0 + f), hp_pitch, src_row,
                                                     job->src_rows, cudaMemcpyHostToDevice, c->s_h2d));
                }
            }
        }
        VR180_CUDA(cudaEventRecord(sl.ev_h2d, c->s_h2d));
        // --- compute ------------------------------------------------------------------------------------
        VR180_CUDA(cudaStreamWaitEvent(c->s_comp, sl.ev_h2d, 0));
        if (k >= kSlots) VR180_CUDA(cudaStreamWaitEvent(c->s_comp, sl.ev_d2h, 0));  // slot's previous download done
        vr180_remap_params_t p;
        memset(&p, 0, sizeof(p));
        p.n_views = V;
        p.n_frames = nf;
        p.share_map = (V == 2 && job->share_map) ? 1 : 0;
        p.out_w = job->out_w;
        p.out_h = job->out_h;
        p.interpolation = job->interpolation;
        p.border_mode = job->border_mode;
        memcpy(p.border_value, job->border_value, 4);
        p.dst = (uint8_t*)sl.dst.p;
        p.dst_pitch = (int64_t)dst_pitch;
        p.dst_frame_stride = (int64_t)dst_frame;
        double* rad = (double*)c->radius.p + f0;
        for (int v = 0; v < V; ++v) {
            vr180_view_t& vw = p.view[v];
            vw.src.data = (const uint8_t*)sl.src[v].p;
            vw.src.rows = job->src_rows;
            vw.src.cols = job->src_cols;
            vw.src.channels = job->channels;
            vw.src.depth = job->depth;
            vw.src.pitch = (int64_t)src_pitch;
            vw.src.frame_stride = (int64_t)src_frame;
            vw.dst_x_offset = v ? (int)eye1_col : 0;
            const int m = (n_maps == 2) ? v : 0;
            vw.map.kind = job->map_kind;
            if (job->map_kind == VR180_MAPSRC_ANALYTIC) {
                vw.map.chain = job->chain[m];
                vw.map.radius_dev = job->radius_mode == 1 ? rad : nullptr;
            } else {
                vw.map.xmap = (const float*)c->maps[m][0].p;
                vw.map.ymap = (const float*)c->maps[m][1].p;
                vw.map.map_pitch = job->out_w;
            }
        }
        if (job->radius_mode == 1 || job->transitions_out) {
            vr180_image_t im[2] = {p.view[0].src, p.view[1].src};
            rc = launch_get_radius(im, V, nf, job->threshold, (int32_t*)c->trans.p + (size_t)2 * V * f0, rad, c->s_comp);
            if (rc != VR180_OK) return rc;
        }
        rc = launch_remap(&p, border_scalar, c->s_comp);
        if (rc != VR180_OK) return rc;
        if (merge) {
            rc = launch_anaglyph((const uint8_t*)sl.dst.p, (int64_t)dst_pitch, (int64_t)dst_frame, job->out_w, (int)eye1_col,
                                 job->out_h, nf, (uint8_t*)sl.merged.p, (int64_t)out_pitch, (int64_t)out_frame, c->s_comp);
            if (rc != VR180_OK) return rc;
        }
        const uint8_t* d_out = (const uint8_t*)(merge ? sl.merged.p : sl.dst.p);
        VR180_CUDA(cudaEventRecord(sl.ev_comp, c->s_comp));
        // --- download -----------------------------------------------------------------------------------
        VR180_CUDA(cudaStreamWaitEvent(c->s_d2h, sl.ev_comp, 0));
        if (stage_out) {
            if (slot_ticket[s]) c->wait_drained(slot_ticket[s]);  // the slot's pinned dst has been unpacked
            VR180_CUDA(cudaMemcpyAsync(sl.h_dst.p, d_out, out_frame * nf, cudaMemcpyDeviceToHost, c->s_d2h));
            VR180_CUDA(cudaEventRecord(sl.ev_d2h, c->s_d2h));
            std::vector<Copy2D> cp;
            for (int f = 0; f < nf; ++f)
                for (const Seg& g : segs)
                    cp.push_back({dst_of(f0 + f) + g.host_col, (const uint8_t*)sl.h_dst.p + (size_t)f * out_frame + g.dev_col,
                                  (size_t)job->dst_pitch, out_pitch, g.bytes, (size_t)job->out_h});
            cudaEvent_t ev = sl.ev_d2h;
            slot_ticket[s] = c->push_drain([pool, ev, cp] {
                cudaEventSynchronize(ev);
                run_copies(*pool, cp);
            });
            continue;
        }
        const size_t hd_pitch = (size_t)job->dst_pitch;
        const bool dense_out = !job->dst_frames && (size_t)job->dst_frame_stride == hd_pitch * job->out_h;
        if (dense_out && hd_pitch == out_pitch && segs.size() == 1) {
            VR180_CUDA(cudaMemcpyAsync(dst_of(f0), d_out, out_frame * nf, cudaMemcpyDeviceToHost, c->s_d2h));
        } else if (dense_out) {
            for (const Seg& g : segs)
                VR180_CUDA(cudaMemcpy2DAsync(dst_of(f0) + g.host_col, hd_pitch, d_out + g.dev_col, out_pitch, g.bytes,
                                             (size_t)job->out_h * nf, cudaMemcpyDeviceToHost, c->s_d2h));
        } else {
            for (int f = 0; f < nf; ++f) {
                if (hd_pitch == out_pitch && segs.size() == 1)
                    VR180_CUDA(cudaMemcpyAsync(dst_of(f0 + f), d_out + f * out_frame, out_frame, cudaMemcpyDeviceToHost,
                                               c->s_d2h));
                else
                    for (const Seg& g : segs)
                        VR180_CUDA(cudaMemcpy2DAsync(dst_of(f0 + f) + g.host_col, hd_pitch, d_out + f * out_frame + g.dev_col,
                                                     out_pitch, g.bytes, job->out_h, cudaMemcpyDeviceToHost, c->s_d2h));
            }
        }
        VR180_CUDA(cudaEventRecord(sl.ev_d2h, c->s_d2h));
    }
    if (job->transitions_out || job->radius_out) {
        VR180_CUDA(cudaStreamWaitEvent(c->s_d2h, c->slot[(n_chunks - 1) % kSlots].ev_comp, 0));
        if (job->transitions_out)
            VR180_CUDA(cudaMemcpyAsync(job->transitions_out, c->trans.p, sizeof(int32_t) * 2 * V * F,
                                       cudaMemcpyDeviceToHost, c->s_d2h));
        if (job->radius_out && job->radius_mode == 1)
            VR180_CUDA(cudaMemcpyAsync(job->radius_out, c->radius.p, sizeof(double) * F, cudaMemcpyDeviceToHost, c->s_d2h));
    }
    return VR180_OK;
}

int vr180_ctx_run(vr180_ctx_t* c, const vr180_host_job_t* job) { return vr180_ctx_run_ex(c, job, nullptr); }

int vr180_ctx_run_ex(vr180_ctx_t* c, const vr180_host_job_t* job, const double border_scalar[4]) {
    if (!c || !job || (!job->dst && !job->dst_frames)) return VR180_ERR_INVALID_ARG;
    const int V = job->n_views, F = job->n_frames, ch = job->channels;
    if (V < 1 || V > 2 || F < 0 || job->src_rows <= 0 || job->src_cols <= 0 || job->out_w <= 0 || job->out_h <= 0)
        return VR180_ERR_INVALID_ARG;
    if (ch != 1 && ch != 3 && ch != 4) return VR180_ERR_UNSUPPORTED;
    if (job->depth != VR180_DEPTH_8U && job->depth != VR180_DEPTH_16U) return VR180_ERR_UNSUPPORTED;
    if (job->merge && job->depth != VR180_DEPTH_8U) return VR180_ERR_UNSUPPORTED;  // the anaglyph is 8-bit
    const int C = ch * depth_bytes(job->depth);  // bytes per pixel
    const bool scattered = job->src_frames[0] != nullptr;
    for (int v = 0; v < V; ++v) {
        if (scattered ? !job->src_frames[v] : !job->src[v]) return VR180_ERR_INVALID_ARG;
        if ((size_t)job->src_pitch[v] < (size_t)job->src_cols * C) return VR180_ERR_INVALID_ARG;
        for (int f = 0; scattered && f < F; ++f)
            if (!job->src_frames[v][f]) return VR180_ERR_INVALID_ARG;
    }
    for (int f = 0; job->dst_frames && f < F; ++f)
        if (!job->dst_frames[f]) return VR180_ERR_INVALID_ARG;
    if (job->merge && (V != 2 || ch != 3)) return VR180_ERR_INVALID_ARG;
    if ((size_t)job->dst_pitch < (size_t)job->out_w * (job->merge ? 1 : V) * C) return VR180_ERR_INVALID_ARG;
    if (job->map_kind != VR180_MAPSRC_ANALYTIC && job->map_kind != VR180_MAPSRC_FLOAT2) return VR180_ERR_UNSUPPORTED;
    if (job->radius_mode == 1 && job->map_kind != VR180_MAPSRC_ANALYTIC) return VR180_ERR_UNSUPPORTED;
    if (job->staging < 0 || job->staging > 2 || job->copy_threads < 0) return VR180_ERR_INVALID_ARG;
    if (F == 0) return VR180_OK;

    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    if (!g.ok) return VR180_ERR_CUDA;
    const int rc = ctx_run_locked(c, job, border_scalar);
    // One exit for success and failure alike: nothing of this job may still be in flight when the caller gets its
    // buffers back (copies and kernels of earlier chunks read job->src / write job->dst asynchronously).
    const cudaError_t e0 = cudaStreamSynchronize(c->s_h2d), e1 = cudaStreamSynchronize(c->s_comp),
                      e2 = cudaStreamSynchronize(c->s_d2h);
    {
        std::unique_lock<std::mutex> l(c->dm);
        c->dcv.wait(l, [&] { return c->drained >= c->queued; });
    }
    if (rc != VR180_OK) {
        cudaGetLastError();
        return rc;
    }
    for (cudaError_t e : {e0, e1, e2})
        if (e != cudaSuccess) {
            set_cuda_error(e, "cudaStreamSynchronize");
            return VR180_ERR_CUDA;
        }
    return VR180_OK;
}

/* Test hook: the copy threads' byte mover (streaming stores for large copies, hostcopy.cpp) on caller buffers. */
int vr180_debug_host_copy(void* dst, const void* src, size_t bytes) {
    if ((!dst || !src) && bytes) return VR180_ERR_INVALID_ARG;
    copy_bytes(static_cast<uint8_t*>(dst), static_cast<const uint8_t*>(src), bytes);
    return VR180_OK;
}

/* Measurement utility for bench.py's e2e.copy_ceiling: page-locked host <-> device copies of `bytes` each way with NO
   kernel in between -- upload alone, download alone, and both at once on two streams (what the pipeline above
   overlaps).  out_gbs[0..3] = {H2D alone, D2H alone, H2D while both run, D2H while both run} in GB/s (1e9). */
int vr180_debug_copy_ceiling(int device, size_t bytes, int reps, double* out_gbs) {
    if (!out_gbs || bytes == 0 || reps < 1) return VR180_ERR_INVALID_ARG;
    DeviceGuard g(device);
    if (!g.ok) return VR180_ERR_CUDA;
    void *h_up = nullptr, *h_down = nullptr, *d_up = nullptr, *d_down = nullptr;
    cudaStream_t s0 = nullptr, s1 = nullptr;
    cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
    auto body = [&]() -> int {
        VR180_CUDA(cudaHostAlloc(&h_up, bytes, cudaHostAllocPortable));
        VR180_CUDA(cudaHostAlloc(&h_down, bytes, cudaHostAllocPortable));
        memset(h_up, 1, bytes);
        memset(h_down, 2, bytes);
        VR180_CUDA(cudaMalloc(&d_up, bytes));
        VR180_CUDA(cudaMalloc(&d_down, bytes));
        VR180_CUDA(cudaStreamCreateWithFlags(&s0, cudaStreamNonBlocking));
        VR180_CUDA(cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking));
        for (auto& ev : e) VR180_CUDA(cudaEventCreate(&ev));
        auto timed = [&](bool up, bool down, float* ms_up, float* ms_down) -> int {
            for (int warm = 0; warm < 2; ++warm) {
                if (warm == 1) {
                    if (up) VR180_CUDA(cudaEventRecord(e[0], s0));
                    if (down) VR180_CUDA(cudaEventRecord(e[2], s1));
                }
                for (int r = 0; r < (warm ? reps : 1); ++r) {
                    if (up) VR180_CUDA(cudaMemcpyAsync(d_up, h_up, bytes, cudaMemcpyHostToDevice, s0));
                    if (down) VR180_CUDA(cudaMemcpyAsync(h_down, d_down, bytes, cudaMemcpyDeviceToHost, s1));
                }
                if (warm == 1) {
                    if (up) VR180_CUDA(cudaEventRecord(e[1], s0));
                    if (down) VR180_CUDA(cudaEventRecord(e[3], s1));
                }
                VR180_CUDA(cudaStreamSynchronize(s0));
                VR180_CUDA(cudaStreamSynchronize(s1));
            }
            if (up) VR180_CUDA(cudaEventElapsedTime(ms_up, e[0], e[1]));
            if (down) VR180_CUDA(cudaEventElapsedTime(ms_down, e[2], e[3]));
            return VR180_OK;
        };
        float a = 0, b = 0, cu = 0, cd = 0, dummy = 0;
        int rc;
        if ((rc = timed(true, false, &a, &dummy)) != VR180_OK) return rc;
        if ((rc = timed(false, true, &dummy, &b)) != VR180_OK) return rc;
        if ((rc = timed(true, true, &cu, &cd)) != VR180_OK) return rc;
        const double gb = (double)bytes * reps / 1e9;
        out_gbs[0] = gb / (a / 1e3);
        out_gbs[1] = gb / (b / 1e3);
        out_gbs[2] = gb / (cu / 1e3);
        out_gbs[3] = gb / (cd / 1e3);
        return VR180_OK;
    };
    const int rc = body();
    for (auto& ev : e)
        if (ev) cudaEventDestroy(ev);
    if (s0) cudaStreamDestroy(s0);
    if (s1) cudaStreamDestroy(s1);
    if (d_up) cudaFree(d_up);
    if (d_down) cudaFree(d_down);
    if (h_up) cudaFreeHost(h_up);
    if (h_down) cudaFreeHost(h_down);
    return rc;
}

}  // extern "C"
