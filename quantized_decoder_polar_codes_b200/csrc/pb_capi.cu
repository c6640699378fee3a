// libpolar_b200.so -- C ABI (include/polar_b200.h) over the sm_100a decoder kernels.
// Host side: validates the constructor arguments the reference classes take, packs the lookup tables to
// bytes, replays the reference's data-independent tree walk once into a linear schedule, uploads
// everything, and launches the kernels.  No CPU decode path exists here: without a CUDA device every
// entry point fails with PD_ECUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <limits>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include "../../include/polar_b200.h"
#include "pb_internal.h"
#include "pb_generic.cuh"
#include "pb_scl_lut.cuh"
#include "pb_path_warp.cuh"
#include "pb_path_cta.cuh"
#ifndef PB_HOST_EMU   // (tools/emu emulates the decode kernels only)
#include "pb_sim.cuh"
#include "pb_enc.cuh"
#endif

using namespace pb;

// dispatchers over the kernel objects (pb_kernels.cu)
namespace pb {
const void *scl_fn_l3_plain(bool ca);
const void *scl_fn_l3_fast(bool ca);
const void *scl_fn_l01(int logL, bool ca, bool fast);
const void *scl_fn_l2(bool ca, bool fast);
const void *path_fn_lut(int logL);
const void *path_fn_float(int logL);
const void *path_fn_uniform(int logL);
const void *path_fn_lloyd(int logL);
// pb_lutgen.cu (its own object: the compile-time-unrolled pairwise sums take minutes to build)
constexpr int kOptlsMaxM = 1024;
cudaError_t launch_optls(int n_problems, size_t smem, const double *density, const double *quanta, const int32_t *M, long long stride, int K,
                         double *out_density, double *out_quanta, int32_t *out_lut, double *T, int32_t *lm, long long t_stride, long long lm_stride);
cudaError_t launch_mmi_table(int P, int M, int W, int mode, const double *p1, const double *p2, const double *l1, const double *l2,
                             double c1, double c2, double *out1, double *out2);
cudaError_t launch_mmi_dp(int P, int M, int K, int W, const double *T, int32_t *lm, int32_t *Az);
const void *fast_kernel_fn(int logL, bool ca, bool fast) {
    if (logL >= 3) return fast ? scl_fn_l3_fast(ca) : scl_fn_l3_plain(ca);
    if (logL == 2) return scl_fn_l2(ca, fast);
    return scl_fn_l01(logL, ca, fast);
}
const void *path_kernel_fn(int dom, int logL) {
    switch (dom) {
    case DOM_LUT: return path_fn_lut(logL);
    case DOM_FLOAT: return path_fn_float(logL);
    case DOM_UNIFORM: return path_fn_uniform(logL);
    default: return path_fn_lloyd(logL);
    }
}
}  // namespace pb

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};

// SM count of the current device (grid sizing of the streaming kernels), cached
int current_sm_count() {
    static std::atomic<int> cache[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    int v = cache[dev].load();
    if (v == 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        cache[dev].store(v);
    }
    return v;
}

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess) return fail(PD_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(e_));    \
    } while (0)

bool is_lut(int k) { return k >= PD_SCLUT && k <= PD_CAFASTSCLLUT; }
bool is_list(int k) {
    return k == PD_SCL || k == PD_FASTSCL || k == PD_CASCL || k == PD_SCLLUT || k == PD_FASTSCLLUT ||
           k == PD_CASCLLUT || k == PD_CAFASTSCLLUT || k == PD_SCL_UNIFORM || k == PD_SCL_LLOYD || k == PD_BD_CASCL;
}
bool is_fast(int k) {
    return k == PD_FASTSC || k == PD_FASTSCL || k == PD_FASTSCLUT || k == PD_FASTSCLLUT || k == PD_CAFASTSCLLUT || k == PD_BD_DMETRIC;
}
bool is_ca(int k) { return k == PD_CASCL || k == PD_CASCLLUT || k == PD_CAFASTSCLLUT || k == PD_BD_CASCL; }
int domain_of(int k) {
    if (is_lut(k)) return DOM_LUT;
    if (k == PD_SC_UNIFORM || k == PD_SCL_UNIFORM) return DOM_UNIFORM;
    if (k == PD_SC_LLOYD || k == PD_SCL_LLOYD) return DOM_LLOYD;
    return DOM_FLOAT;
}

struct StreamSlot {
    cudaStream_t stream = nullptr;
    void *d_in = nullptr;
    uint8_t *d_out = nullptr;
    char *ws = nullptr;
    size_t in_cap = 0, out_cap = 0, ws_cap = 0;
    // pd_decode with pageable / int32 host buffers: pinned staging areas and the event that says the chunk's result is in h_out
    char *h_in = nullptr, *h_out = nullptr;
    size_t h_in_cap = 0, h_out_cap = 0;
    cudaEvent_t done = nullptr;
};

}  // namespace

// ---- host-side staging of pd_decode ------------------------------------------------------------------------------
// A small persistent pool: pd_decode converts / copies the caller's (pageable, possibly int32) buffers to and from pinned
// staging memory with all host cores while the previous chunk is on the GPU.
namespace {
class HostPool {
public:
    static HostPool &get() { static HostPool p; return p; }
    int size() const { return (int)workers_.size() + 1; }
    // runs fn(part) for part = 0 .. parts-1 on the pool (the caller takes part too) and waits
    void run(int parts, const std::function<void(int)> &fn) {
        if (parts <= 1 || workers_.empty()) { for (int i = 0; i < parts; ++i) fn(i); return; }
        {
            std::lock_guard<std::mutex> lk(m_);
            fn_ = &fn; parts_ = parts; next_ = 0; done_ = 0; ++gen_;
        }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(m_);
        cv_done_.wait(lk, [&] { return done_ == parts_; });
        fn_ = nullptr;
    }
private:
    HostPool() {
        int n = (int)std::thread::hardware_concurrency();
        if (const char *e = getenv("POLAR_B200_HOST_THREADS")) n = atoi(e);
        n = std::max(1, std::min(n, 32));
        for (int i = 1; i < n; ++i) workers_.emplace_back([this] { loop(); });
    }
    ~HostPool() {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; ++gen_; }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
    }
    void work() {
        for (;;) {
            int i;
            { std::lock_guard<std::mutex> lk(m_); if (!fn_ || next_ >= parts_) return; i = next_++; }
            (*fn_)(i);
            { std::lock_guard<std::mutex> lk(m_); if (++done_ == parts_) cv_done_.notify_all(); }
        }
    }
    void loop() {
        unsigned long long seen = 0;
        for (;;) {
            { std::unique_lock<std::mutex> lk(m_); cv_.wait(lk, [&] { return gen_ != seen; }); seen = gen_; if (stop_) return; }
            work();
        }
    }
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_, cv_done_;
    const std::function<void(int)> *fn_ = nullptr;
    int parts_ = 0, next_ = 0, done_ = 0;
    unsigned long long gen_ = 0;
    bool stop_ = false;
};

// n int32 symbols -> bytes; returns false if a value does not fit a byte (the kernels then never see it)
bool narrow_i32_to_u8(const int32_t *src, uint8_t *dst, size_t n) {
    uint32_t bad = 0;
    size_t i = 0;
#if defined(__SSE2__)
    const bool nt = (reinterpret_cast<uintptr_t>(dst) & 15u) == 0;
    __m128i acc = _mm_setzero_si128();
    for (; i + 16 <= n; i += 16) {
        const __m128i a0 = _mm_loadu_si128((const __m128i *)(src + i)), a1 = _mm_loadu_si128((const __m128i *)(src + i + 4));
        const __m128i a2 = _mm_loadu_si128((const __m128i *)(src + i + 8)), a3 = _mm_loadu_si128((const __m128i *)(src + i + 12));
        acc = _mm_or_si128(acc, _mm_or_si128(_mm_or_si128(a0, a1), _mm_or_si128(a2, a3)));
        const __m128i r = _mm_packus_epi16(_mm_packs_epi32(a0, a1), _mm_packs_epi32(a2, a3));
        if (nt) _mm_stream_si128((__m128i *)(dst + i), r);     // pinned staging area: written once, read by the copy engine
        else _mm_storeu_si128((__m128i *)(dst + i), r);
    }
    if (nt) _mm_sfence();
    alignas(16) uint32_t lanes[4];
    _mm_store_si128((__m128i *)lanes, acc);
    bad = lanes[0] | lanes[1] | lanes[2] | lanes[3];
#endif
    for (; i < n; ++i) { bad |= (uint32_t)src[i]; dst[i] = (uint8_t)src[i]; }
    return (bad & 0xffffff00u) == 0;
}

// n float64 symbols -> bytes (the probability-domain drivers keep their symbols in float64 arrays; the reference's pybind
// layer casts them to int by truncation); false if a value does not fit a byte
bool narrow_f64_to_u8(const double *src, uint8_t *dst, size_t n) {
    uint32_t bad = 0;
    size_t i = 0;
#if defined(__SSE2__)
    const bool nt = (reinterpret_cast<uintptr_t>(dst) & 15u) == 0;
    __m128i acc = _mm_setzero_si128();
    for (; i + 16 <= n; i += 16) {
        __m128i q[4];
        for (int k = 0; k < 4; ++k) {
            const __m128i lo = _mm_cvttpd_epi32(_mm_loadu_pd(src + i + 4 * k)), hi = _mm_cvttpd_epi32(_mm_loadu_pd(src + i + 4 * k + 2));
            q[k] = _mm_unpacklo_epi64(lo, hi);
        }
        acc = _mm_or_si128(acc, _mm_or_si128(_mm_or_si128(q[0], q[1]), _mm_or_si128(q[2], q[3])));
        const __m128i r = _mm_packus_epi16(_mm_packs_epi32(q[0], q[1]), _mm_packs_epi32(q[2], q[3]));
        if (nt) _mm_stream_si128((__m128i *)(dst + i), r);
        else _mm_storeu_si128((__m128i *)(dst + i), r);
    }
    if (nt) _mm_sfence();
    alignas(16) uint32_t lanes[4];
    _mm_store_si128((__m128i *)lanes, acc);
    bad = lanes[0] | lanes[1] | lanes[2] | lanes[3];
#endif
    for (; i < n; ++i) {
        const double v = src[i];
        const int32_t t = (v > -1.0 && v < 256.0) ? (int32_t)v : -1;
        bad |= (uint32_t)t;
        dst[i] = (uint8_t)t;
    }
    return (bad & 0xffffff00u) == 0;
}

bool is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}
}  // namespace

// Deep copy of the constructor arguments: pd_set_devices clones the decoder onto other GPUs from it.
struct ConfigCopy {
    pd_config c{};
    std::vector<int32_t> frozen, node_type, crc_loc, lut_pool, f_npos, g_npos, f_qa, f_qb, g_qa, g_qb;
    std::vector<int64_t> f_off, g_off, llr_off;
    std::vector<double> llr_pool, r_f, r_g, bf, bg, rf, rg;
    void take(const pd_config *src) {
        c = *src;
        const size_t N = (size_t)src->N;
        auto cp = [](auto &vec, const auto *ptr, size_t n, const auto *&field) {
            if (ptr && n) { vec.assign(ptr, ptr + n); field = vec.data(); } else { vec.clear(); field = nullptr; }
        };
        cp(frozen, src->frozen_bits, N, c.frozen_bits);
        cp(node_type, src->node_type, 2 * N - 1, c.node_type);
        cp(crc_loc, src->crc_loc, (size_t)std::max(0, src->crc_loc_len), c.crc_loc);
        cp(lut_pool, src->lut_pool, (size_t)std::max<int64_t>(0, src->lut_pool_len), c.lut_pool);
        cp(f_off, src->f_off, N - 1, c.f_off); cp(g_off, src->g_off, N - 1, c.g_off);
        cp(f_npos, src->f_npos, N - 1, c.f_npos); cp(g_npos, src->g_npos, N - 1, c.g_npos);
        cp(f_qa, src->f_qa, N - 1, c.f_qa); cp(f_qb, src->f_qb, N - 1, c.f_qb);
        cp(g_qa, src->g_qa, N - 1, c.g_qa); cp(g_qb, src->g_qb, N - 1, c.g_qb);
        const size_t rows = src->llr_off ? (size_t)src->llr_levels * N : 0;
        cp(llr_off, src->llr_off, rows ? rows + 1 : 0, c.llr_off);
        cp(llr_pool, src->llr_pool, rows ? (size_t)src->llr_off[rows] : 0, c.llr_pool);
        cp(r_f, src->decoder_r_f, N - 1, c.decoder_r_f); cp(r_g, src->decoder_r_g, N - 1, c.decoder_r_g);
        cp(bf, src->boundaries_f, (N - 1) * (size_t)std::max(0, src->n_boundaries), c.boundaries_f);
        cp(bg, src->boundaries_g, (N - 1) * (size_t)std::max(0, src->n_boundaries), c.boundaries_g);
        cp(rf, src->reconstruction_f, (N - 1) * (size_t)std::max(0, src->n_reconstruction), c.reconstruction_f);
        cp(rg, src->reconstruction_g, (N - 1) * (size_t)std::max(0, src->n_reconstruction), c.reconstruction_g);
    }
};

struct pd_decoder {
    Dev dev{};
    int device = 0;
    int sm_count = 0;
    std::vector<void *> allocs;
    std::vector<Step> steps;
    int64_t elem_ops = 0, n_sorts = 0;
    // generic kernel launch geometry
    int threads = 32;
    size_t ws_bytes = 0;      // per-CTA workspace
    int use_smem = 0;
    int ctas_per_sm = 1;
    // specialised kernel
    FastPlan fast{};
    PathPlan path{};          // warp-level schedule interpreter (all classes, L power of two)
    CtaPlan cta{};            // CTA-level schedule interpreter: the list sizes 64, 128, 256, and nothing else runs them
    cudaEvent_t fork_ev = nullptr, join_ev[2] = {nullptr, nullptr};   // pd_decode_device: split of large batches
    cudaStream_t side[2] = {nullptr, nullptr};
    int force = 0;            // POLAR_B200_FORCE_GENERIC: 1 = CTA-per-frame generic kernel, 2 = path_warp (L <= 32 only:
                              // L > 32 always runs path_cta)
    const char *kernel_name = "generic";
    int *d_err = nullptr;             // device view of the mapped error flag
    volatile int *h_err = nullptr;   // host view
    double *dbg_pm = nullptr;
    int32_t *dbg_win = nullptr;
    char *ws_user = nullptr;  // workspace for pd_decode_device (global-memory variant)
    size_t ws_user_cap = 0;
    StreamSlot slot[2];
    int64_t chunk_frames = 0;
    // pd_decode, tiny calls (the reference drivers decode one frame per call): a mapped pinned staging area the kernel
    // reads and writes directly -- no copy engine round trips
    char *h_small = nullptr, *d_small = nullptr;
    // pd_set_devices: the batch of a pd_decode call is dealt chunk by chunk to `units` (this decoder and its clones on other
    // GPUs of the box); empty = this decoder alone
    ConfigCopy cfg;
    std::vector<pd_decoder *> clones;     // owned
    std::vector<pd_decoder *> units;      // not owned: this and / or clones, in the order of the device list
};
constexpr size_t kSmallIn = 64 << 10, kSmallOut = 16 << 10;   // bytes of input / output served by the mapped path

namespace {

template <typename T>
int upload(pd_decoder *D, const std::vector<T> &h, const T **out) {
    void *p = nullptr;
    size_t bytes = std::max<size_t>(h.size() * sizeof(T), 16);
    CUDA_TRY(cudaMalloc(&p, bytes));
    D->allocs.push_back(p);
    if (!h.empty()) CUDA_TRY(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = reinterpret_cast<const T *>(p);
    return PD_OK;
}

bool special_type(int kind, int t) {
    if (!is_fast(kind)) return false;
    if (t < 0) return false;
    return is_list(kind) ? t <= 2 : t <= 3;   // list variants expand SPC nodes (SURVEY App. B6)
}

struct Builder {
    const pd_config *cfg;
    int N, n, kind;
    std::vector<Step> steps;
    int64_t elem_ops = 0, n_sorts = 0;
    int r1_tmax = 0;
    void walk(int d, uint32_t node) {
        if (d == n) {
            steps.push_back(Step{OP_LEAF, (uint8_t)d, (uint8_t)(cfg->frozen_bits[node] == 1), 0, node});
            if (is_list(kind) && cfg->frozen_bits[node] != 1) n_sorts++;
            return;
        }
        int p = (1 << d) + (int)node - 1;
        if (is_fast(kind)) {
            int t = cfg->node_type[p];
            if (special_type(kind, t)) {
                static const uint8_t ops[4] = {OP_R0, OP_R1, OP_REP, OP_SPC};
                steps.push_back(Step{ops[t], (uint8_t)d, 0, 0, node});
                int temp = N >> d;
                if (is_list(kind)) {
                    if (t == 1) { r1_tmax = std::max(r1_tmax, temp); n_sorts += std::min(cfg->L - 1, temp); }
                    if (t == 2) n_sorts++;
                }
                return;
            }
        }
        steps.push_back(Step{OP_F, (uint8_t)d, 0, 0, node});
        elem_ops += N >> (d + 1);
        walk(d + 1, 2 * node);
        steps.push_back(Step{OP_G, (uint8_t)d, 0, 0, node});
        elem_ops += N >> (d + 1);
        walk(d + 1, 2 * node + 1);
        steps.push_back(Step{OP_C, (uint8_t)d, 0, 0, node});
    }
};

int build_lut(pd_decoder *D, const pd_config *c) {
    const int N = c->N, n = D->dev.n, kind = c->kind;
    if (!c->lut_pool || !c->f_off || !c->g_off || !c->f_npos || !c->g_npos || !c->f_qa || !c->f_qb || !c->g_qa ||
        !c->g_qb || !c->llr_pool || !c->llr_off)
        return fail(PD_EINVAL, "LUT decoder needs LUT_f, LUT_g and virtual_channel_llr");
    if (c->llr_levels < n) return fail(PD_EINVAL, "virtual_channel_llr has %d levels, need >= %d", c->llr_levels, n);
    auto llr_len = [&](int level, int pos) -> int64_t {
        int64_t r = (int64_t)level * N + pos;
        return c->llr_off[r + 1] - c->llr_off[r];
    };
    // bound that the values of child (cd,cn), element j, must respect
    auto consumer_bound = [&](int cd, uint32_t cn, int j) -> int64_t {
        int ct = N >> cd;
        if (cd == n) return llr_len(n - 1, (int)cn);
        int cp = (1 << cd) + (int)cn - 1;
        if (is_fast(kind) && special_type(kind, c->node_type[cp])) return llr_len(cd - 1, (int)(cn * (uint32_t)ct) + j);
        int half = ct / 2;
        return j < half ? std::min(c->f_qa[cp], c->g_qa[cp]) : std::min(c->f_qb[cp], c->g_qb[cp]);
    };
    std::vector<NodeTab> tabs(N - 1);
    std::vector<uint8_t> pool;
    pool.reserve(1 << 20);
    for (int d = 0; d < n; ++d) {
        for (uint32_t node = 0; node < (1u << d); ++node) {
            int p = (1 << d) + (int)node - 1;
            int ct = N >> (d + 1);
            NodeTab &tb = tabs[p];
            for (int isg = 0; isg < 2; ++isg) {
                int qa = isg ? c->g_qa[p] : c->f_qa[p], qb = isg ? c->g_qb[p] : c->f_qb[p];
                int npos = isg ? c->g_npos[p] : c->f_npos[p];
                int64_t off = isg ? c->g_off[p] : c->f_off[p];
                int planes = isg ? 2 : 1;
                if (qa < 1 || qb < 1 || qa > 256 || qb > 256) return fail(PD_EINVAL, "node %d: table dims %dx%d unsupported (1..256)", p, qa, qb);
                if (npos != 1 && npos < ct) return fail(PD_EINVAL, "node %d: %d per-position tables, need 1 or >= %d", p, npos, ct);
                int64_t per = (int64_t)planes * qa * qb;
                if (off < 0 || off + per * (npos == 1 ? 1 : ct) > c->lut_pool_len) return fail(PD_EINVAL, "node %d: table outside lut_pool", p);
                int stored = (npos == 1) ? 1 : ct;
                // per-position tables that are all equal collapse to one (every generator of the reference emits that)
                if (stored > 1) {
                    bool same = true;
                    for (int j = 1; j < stored && same; ++j)
                        same = memcmp(c->lut_pool + off, c->lut_pool + off + per * j, (size_t)per * sizeof(int32_t)) == 0;
                    if (same) stored = 1;
                }
                uint32_t base = (uint32_t)pool.size();
                uint32_t cn = 2 * node + (uint32_t)isg;
                for (int j = 0; j < stored; ++j) {
                    int64_t bound = std::numeric_limits<int64_t>::max();
                    if (stored == 1) for (int jj = 0; jj < ct; ++jj) bound = std::min(bound, consumer_bound(d + 1, cn, jj));
                    else bound = consumer_bound(d + 1, cn, j);
                    const int32_t *src = c->lut_pool + off + per * j;
                    for (int64_t e = 0; e < per; ++e) {
                        int32_t v = src[e];
                        if (v < 0 || v >= bound || v > 255)
                            return fail(PD_EINVAL, "LUT_%s[%d]: entry %d is outside the consumer alphabet [0,%lld)", isg ? "g" : "f", p, v, (long long)std::min<int64_t>(bound, 256));
                        pool.push_back((uint8_t)v);
                    }
                }
                if (isg) { tb.g_off = base; tb.g_sz = (uint32_t)(qa * qb); tb.g_qb = (uint16_t)qb; tb.g_pstride = stored == 1 ? 0 : (uint32_t)per; }
                else { tb.f_off = base; tb.f_sz = (uint32_t)(qa * qb); tb.f_qb = (uint16_t)qb; tb.f_pstride = stored == 1 ? 0 : (uint32_t)per; }
            }
        }
    }
    D->dev.root_qa = std::min(c->f_qa[0], c->g_qa[0]);
    D->dev.root_qb = std::min(c->f_qb[0], c->g_qb[0]);
    int64_t rows = (int64_t)c->llr_levels * N;
    int64_t total = c->llr_off[rows];
    if (total > (int64_t)0x7fffffff) return fail(PD_EINVAL, "virtual_channel_llr too large");
    std::vector<uint32_t> loff(rows);
    for (int64_t r = 0; r < rows; ++r) {
        if (c->llr_off[r + 1] < c->llr_off[r]) return fail(PD_EINVAL, "llr_off not monotone");
        loff[r] = (uint32_t)c->llr_off[r];
    }
    std::vector<double> llr(c->llr_pool, c->llr_pool + total);
    int rc;
    if ((rc = upload(D, pool, &D->dev.lut))) return rc;
    if ((rc = upload(D, tabs, &D->dev.tabs))) return rc;
    if ((rc = upload(D, llr, &D->dev.llr))) return rc;
    if ((rc = upload(D, loff, &D->dev.llr_off))) return rc;
    {
        const bool fastk = is_fast(kind);
        const int max_special = !fastk ? -1 : (is_list(kind) ? 2 : 3);
        plan_fast_lut(D->dev, true, c->node_type, max_special, tabs, pool, llr, loff, c->llr_off, c->frozen_bits, D->dev.crc_taps, &D->fast);
    }
    return PD_OK;
}

// kernel instantiations live in pb_kernels.cu (one object per family, compiled in parallel)
const void *generic_fn_for(const pd_decoder *D) {
    return pb::generic_kernel_fn(D->dev.domain, D->dev.list != 0, D->threads == 32);
}

int generic_grid(const pd_decoder *D, int64_t B) {
    int64_t g = (int64_t)D->sm_count * D->ctas_per_sm;
    return (int)std::max<int64_t>(1, std::min<int64_t>(g, B));
}

int launch_generic(pd_decoder *D, const void *d_in, int dtype, int64_t B, uint8_t *d_out, cudaStream_t s, char *ws) {
    int grid = generic_grid(D, B);
    size_t smem = D->use_smem ? D->ws_bytes : 0;
    long long Bll = B;
    void *args[] = {(void *)&D->dev, (void *)&d_in, (void *)&dtype, (void *)&d_out, (void *)&Bll, (void *)&ws, (void *)&D->ws_bytes,
                    (void *)&D->use_smem, (void *)&D->d_err, (void *)&D->dbg_pm, (void *)&D->dbg_win};
    CUDA_TRY(cudaLaunchKernel(generic_fn_for(D), dim3(grid), dim3(D->threads), args, smem, s));
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return PD_OK;
}

int plan_generic(pd_decoder *D) {
    const Dev &d = D->dev;
    int L = d.list ? d.L : 1;
    size_t vsz = d.domain == DOM_LUT ? 1 : 8;
    size_t ws = (((size_t)L * d.N * vsz + 15) & ~(size_t)15) + (size_t)L * d.r1_tmax * (8 + 4) + (size_t)L * 3 * d.N + (size_t)2 * L * d.r1_tmax + d.N;
    ws = (ws + 15) & ~(size_t)15;
    D->ws_bytes = ws;
    int64_t work = (int64_t)L * d.N / 2;
    int th = 32;
    while (th < 256 && th * 8 < work) th *= 2;
    D->threads = th;
    D->use_smem = ws <= 96 * 1024;
    const void *fn = generic_fn_for(D);
    // (the attribute belongs to the kernel function, which every decoder of the same domain shares: always the cap, never
    //  this decoder's own size -- a smaller decoder created later must not shrink it under a live larger one)
    if (D->use_smem) CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    int occ = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, th, D->use_smem ? ws : 0));
    if (occ < 1) return fail(PD_ECUDA, "generic kernel does not fit on the device (ws=%zu)", ws);
    D->ctas_per_sm = occ;
    return PD_OK;
}

size_t ws_need(const pd_decoder *D, int dtype, const void *d_in, int64_t B);
bool want_fast(const pd_decoder *D, int dtype, const void *d_in) {
    if (D->fast.ok && dtype != PD_F64 && D->force == 0 && (reinterpret_cast<uintptr_t>(d_in) & 15u) != 0) {
        static std::atomic<bool> told{false};
        if (!told.exchange(true) && !getenv("POLAR_B200_QUIET"))
            fprintf(stderr, "[polar_b200] note: input pointer %p is not 16-byte aligned: this call runs on the slower 'path_warp' / 'generic' kernel\n", d_in);
        return false;
    }
    return D->fast.ok && dtype != PD_F64 && D->force == 0;
}
bool want_path(const pd_decoder *D, int dtype, const void *d_in) {
    return !want_fast(D, dtype, d_in) && D->path.ok && D->force != 1;
}

int launch(pd_decoder *D, const void *d_in, int dtype, int64_t B, uint8_t *d_out, cudaStream_t s, char *ws) {
    if (B <= 0) return PD_OK;
    if (D->cta.ok) {
        int rc = launch_path_cta(D->dev, D->cta, d_in, dtype, B, d_out, s, ws, D->d_err, D->dbg_pm, D->dbg_win, D->sm_count);
        g_launches++;
        if (rc != 0) return fail(PD_ECUDA, "path_cta launch failed: %s", cudaGetErrorString((cudaError_t)rc));
        return PD_OK;
    }
    if (want_fast(D, dtype, d_in)) {
        int rc = launch_fast_lut(D->dev, D->fast, d_in, dtype, B, d_out, s, reinterpret_cast<uint32_t *>(ws), D->d_err, D->dbg_pm, D->dbg_win, D->sm_count);
        g_launches++;
        if (rc != 0) return fail(PD_ECUDA, "fast kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
        return PD_OK;
    }
    if (want_path(D, dtype, d_in)) {
        int rc = launch_path_warp(D->dev, D->path, d_in, dtype, B, d_out, s, ws, D->d_err, D->dbg_pm, D->dbg_win, D->sm_count);
        g_launches++;
        if (rc != 0) return fail(PD_ECUDA, "path_warp launch failed: %s", cudaGetErrorString((cudaError_t)rc));
        return PD_OK;
    }
    return launch_generic(D, d_in, dtype, B, d_out, s, ws);
}

// bytes of global workspace the kernel chosen for this call needs
size_t ws_need(const pd_decoder *D, int dtype, const void *d_in, int64_t B) {
    if (D->cta.ok) return D->cta.ws_bytes_per_cta * (size_t)path_cta_grid(D->cta, B, D->sm_count);
    if (want_fast(D, dtype, d_in)) return pb::kWsHeadWords * 4 + D->fast.ws_bytes_per_cta * (size_t)fast_grid(D->fast, B, D->sm_count);
    if (want_path(D, dtype, d_in)) return D->path.ws_bytes_per_cta * (size_t)path_grid(D->path, B, D->sm_count);
    return D->use_smem ? 0 : D->ws_bytes * (size_t)generic_grid(D, B);
}

// frames one full wave of the chosen (persistent) kernel holds in flight; 0 for the CTA-per-frame generic kernel
int64_t wave_frames(const pd_decoder *D, int dtype, const void *d_in) {
    if (D->cta.ok) return (int64_t)D->sm_count * D->cta.ctas_per_sm;   // one frame per CTA
    if (want_fast(D, dtype, d_in)) return (int64_t)D->sm_count * D->fast.ctas_per_sm * D->fast.p.warps * (32 >> D->fast.logL);
    if (want_path(D, dtype, d_in)) return (int64_t)D->sm_count * D->path.ctas_per_sm * (32 >> D->path.logL);
    return 0;
}

size_t dtype_size(int t) { return t == PD_U8 ? 1 : t == PD_I32 ? 4 : 8; }

int check_dtype(const pd_decoder *D, int t, bool host_call = false) {
    if (D->dev.domain == DOM_LUT) {
        if (t == PD_F64 && host_call) return PD_OK;       // float64-typed symbols: narrowed to bytes on the host (pd_decode)
        if (t != PD_U8 && t != PD_I32) return fail(PD_EINVAL, "LUT decoders take PD_U8 or PD_I32 symbols (pd_decode also PD_F64-typed symbols)");
    } else if (t != PD_F64) {
        return fail(PD_EINVAL, "float/uniform/Lloyd decoders take PD_F64 LLRs");
    }
    return PD_OK;
}

}  // namespace

extern "C" {

const char *pd_last_error(void) { return g_err.c_str(); }
const char *pd_version(void) { return "polar_b200 0.1 (sm_100a)"; }
int64_t pd_launch_count(void) { return g_launches.load(); }

void pd_destroy(pd_decoder *D) {
    if (!D) return;
    for (pd_decoder *c : D->clones) pd_destroy(c);
    D->clones.clear();
    cudaSetDevice(D->device);
    for (auto &sl : D->slot) {
        if (sl.stream) { cudaStreamSynchronize(sl.stream); cudaStreamDestroy(sl.stream); }
        cudaFree(sl.d_in); cudaFree(sl.d_out); cudaFree(sl.ws);
        if (sl.h_in) cudaFreeHost(sl.h_in);
        if (sl.h_out) cudaFreeHost(sl.h_out);
        if (sl.done) cudaEventDestroy(sl.done);
    }
    cudaFree(D->ws_user);
    if (D->h_err) cudaFreeHost((void *)D->h_err);
    if (D->h_small) cudaFreeHost(D->h_small);
    for (int i = 0; i < 2; ++i) { if (D->side[i]) { cudaStreamSynchronize(D->side[i]); cudaStreamDestroy(D->side[i]); } if (D->join_ev[i]) cudaEventDestroy(D->join_ev[i]); }
    if (D->fork_ev) cudaEventDestroy(D->fork_ev);
    for (void *p : D->allocs) cudaFree(p);
    free_fast_plan(&D->fast);
    delete D;
}

int pd_create(const pd_config *c, pd_decoder **out) {
    if (!c || !out) return fail(PD_EINVAL, "null argument");
    *out = nullptr;
    const int kind = c->kind, N = c->N;
    if (kind < 0 || kind >= PD_KIND_COUNT) return fail(PD_EINVAL, "unknown decoder kind %d", kind);
    if (N < 2 || N > (1 << kMaxLog) || (N & (N - 1))) return fail(PD_EINVAL, "N=%d must be a power of two in [2,%d]", N, 1 << kMaxLog);
    if (!c->frozen_bits) return fail(PD_EINVAL, "frozen_bits missing");
    int n = 0;
    while ((1 << n) < N) n++;
    const bool list = is_list(kind), fastk = is_fast(kind), ca = is_ca(kind);
    if (list) {   // 1..32 on the warp kernels; 64, 128 and 256 on path_cta, which keeps partial sums as 32-bit words per path
        const bool big = c->L == 64 || c->L == 128 || c->L == 256;
        if (c->L < 1 || (c->L > kMaxL && !big) || (big && (N < 32 || kind == PD_BD_CASCL)))
            return fail(PD_EINVAL, "L=%d: list sizes are 1..%d, or 64, 128 or 256 with N >= 32 (here N=%d; blind-detection CA-SCL: 1..%d only)",
                        c->L, kMaxL, N, kMaxL);
    }
    std::vector<int32_t> info_pos;
    for (int i = 0; i < N; ++i) if (c->frozen_bits[i] == 0) info_pos.push_back(i);
    if ((int)info_pos.size() != c->K) return fail(PD_EINVAL, "K=%d but frozen_bits has %zu non-frozen positions", c->K, info_pos.size());
    if (c->K < 1) return fail(PD_EINVAL, "K must be >= 1");
    if (fastk) {
        if (!c->node_type) return fail(PD_EINVAL, "node_type missing");
        if (special_type(kind, c->node_type[0])) return fail(PD_EINVAL, "degenerate code: the root itself is a special node (the reference reads level -1 here)");
    }
    int crc_n = 0, crc_check = 0;
    uint32_t taps = 0;
    if (ca) {
        if (c->A < 1 || c->A > c->K) return fail(PD_EINVAL, "A=%d must be in [1,K]", c->A);
        std::vector<int> poly;
        if (kind == PD_CASCL || kind == PD_BD_CASCL) {   // honours the ctor polynomial, compares crc_n bits (PD/src/CASCLDecoder.cpp:49-53,222; CASCLWithRNTI.cpp:48-56,228-233)
            crc_n = c->crc_n;
            if (crc_n < 1 || crc_n > 32) return fail(PD_EINVAL, "crc_n=%d unsupported (1..32)", crc_n);
            poly.assign(crc_n + 1, 0);
            for (int i = 0; i < c->crc_loc_len; ++i) {
                if (c->crc_loc[i] < 0 || c->crc_loc[i] > crc_n) return fail(PD_EINVAL, "crc_p entry out of range");
                poly[c->crc_loc[i]] = 1;
            }
            crc_check = crc_n;
        } else {                  // hard-coded CRC-24, compares K-A bits (PD/include/CASCLLUTDecoder.h:33-34, CASCLLUTDecoder.cpp:280)
            static const int loc[13] = {24, 23, 21, 20, 17, 15, 13, 12, 8, 4, 2, 1, 0};
            crc_n = 24;
            poly.assign(25, 0);
            for (int l : loc) poly[l] = 1;
            crc_check = c->K - c->A;
            if (crc_check > 24) return fail(PD_EINVAL, "K-A=%d > 24: the reference reads past its 24 check bits", crc_check);
        }
        if (c->A + crc_check > c->K) return fail(PD_EINVAL, "A + checked CRC bits exceeds K");
        for (int k = 0; k < crc_n; ++k) if (poly[1 + k]) taps |= 1u << (crc_n - 1 - k);
    }

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PD_ECUDA, "no CUDA device: libpolar_b200 has no CPU path");
    if (c->device < 0 || c->device >= ndev) return fail(PD_EINVAL, "device %d out of range", c->device);
    CUDA_TRY(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, c->device));
    if (prop.major != 10) return fail(PD_ECUDA, "device %d is sm_%d%d; this library is built for sm_100a only", c->device, prop.major, prop.minor);

    pd_decoder *D = new pd_decoder();
    D->device = c->device;
    D->sm_count = prop.multiProcessorCount;
    Dev &d = D->dev;
    d.kind = kind; d.N = N; d.n = n; d.K = c->K; d.A = c->A; d.L = list ? c->L : 1;
    d.Kout = ca ? c->A : c->K;
    d.domain = domain_of(kind); d.list = list; d.fast = fastk; d.ca = ca;
    d.pm_init = (kind == PD_SCL || kind == PD_CASCL || kind == PD_SCL_UNIFORM || kind == PD_SCL_LLOYD) ? 1e300 : std::numeric_limits<double>::infinity();
    if (kind == PD_BD_CASCL) d.pm_init = 1e30;   // CASCLWithRNTI.cpp:82
    d.bd = kind == PD_BD_DMETRIC ? 1 : kind == PD_BD_CASCL ? 2 : 0;
    d.crc_n = crc_n; d.crc_check = crc_check; d.crc_taps = taps;

    Builder b{c, N, n, kind};
    b.walk(0, 0);
    D->steps = b.steps;
    D->elem_ops = b.elem_ops; D->n_sorts = b.n_sorts;
    d.r1_tmax = b.r1_tmax;
    d.n_steps = (int)b.steps.size();
    int rc = PD_OK;
    auto bail = [&](int code) { pd_destroy(D); return code; };
    if ((rc = upload(D, b.steps, &d.steps))) return bail(rc);
    if ((rc = upload(D, info_pos, &d.info_pos))) return bail(rc);

    if (d.domain == DOM_LUT) {
        if ((rc = build_lut(D, c))) return bail(rc);
    } else if (d.domain == DOM_UNIFORM) {
        if (!c->decoder_r_f || !c->decoder_r_g) return bail(fail(PD_EINVAL, "decoder_r_f / decoder_r_g missing"));
        std::vector<double> rf(c->decoder_r_f, c->decoder_r_f + N - 1), rg(c->decoder_r_g, c->decoder_r_g + N - 1);
        for (int i = 0; i < N - 1; ++i)
            if (!(rf[i] > 0) || !(rg[i] > 0) || !std::isfinite(rf[i]) || !std::isfinite(rg[i]))
                return bail(fail(PD_EINVAL, "decoder_r_f / decoder_r_g[%d] must be finite and > 0", i));
        if (c->v < 2) return bail(fail(PD_EINVAL, "v=%d must be >= 2", c->v));
        if ((rc = upload(D, rf, &d.r_f)) || (rc = upload(D, rg, &d.r_g))) return bail(rc);
        d.mf_mul = double(c->v / 2 - 0.5);
        d.mg_mul = double(c->v / 2 - 1);
    } else if (d.domain == DOM_LLOYD) {
        if (!c->boundaries_f || !c->boundaries_g || !c->reconstruction_f || !c->reconstruction_g) return bail(fail(PD_EINVAL, "Lloyd tables missing"));
        if (c->n_boundaries < 1 || c->n_reconstruction < 1) return bail(fail(PD_EINVAL, "Lloyd table widths missing"));
        // bisect() returns reconstruction[lo-1] with lo in [0, n_boundaries] (PD/src/utils.cpp:12-24): the reference reads
        // out of bounds unless the first boundary is below every input and there is a cell per boundary gap
        if (c->n_reconstruction < c->n_boundaries - 1) return bail(fail(PD_EINVAL, "Lloyd tables: %d reconstruction values for %d boundaries (need >= boundaries-1)", c->n_reconstruction, c->n_boundaries));
        for (int t = 0; t < 2; ++t) {
            const double *bd = t ? c->boundaries_g : c->boundaries_f;
            for (int p = 0; p < N - 1; ++p) {
                const double *row = bd + (size_t)p * c->n_boundaries;
                for (int k = 0; k < c->n_boundaries; ++k) {
                    if (row[k] != row[k]) return bail(fail(PD_EINVAL, "boundaries_%s[%d][%d] is NaN", t ? "g" : "f", p, k));
                    if (k && row[k] < row[k - 1]) return bail(fail(PD_EINVAL, "boundaries_%s[%d] must ascend", t ? "g" : "f", p));
                }
                if (!(row[0] <= -1e290)) return bail(fail(PD_EINVAL, "boundaries_%s[%d][0] must be the -1e300 sentinel of LloydQuantizer.py:64 (a value below it reads reconstruction[-1] in the reference)", t ? "g" : "f", p));
                if (c->n_reconstruction < c->n_boundaries && !(row[c->n_boundaries - 1] >= 1e290)) return bail(fail(PD_EINVAL, "boundaries_%s[%d]: last boundary must be the +1e300 sentinel when there are fewer reconstruction values than boundaries", t ? "g" : "f", p));
            }
        }
        size_t nbs = (size_t)(N - 1) * c->n_boundaries, nrs = (size_t)(N - 1) * c->n_reconstruction;
        std::vector<double> bf(c->boundaries_f, c->boundaries_f + nbs), bg(c->boundaries_g, c->boundaries_g + nbs);
        std::vector<double> rf(c->reconstruction_f, c->reconstruction_f + nrs), rg(c->reconstruction_g, c->reconstruction_g + nrs);
        if ((rc = upload(D, bf, &d.bnd_f)) || (rc = upload(D, bg, &d.bnd_g)) || (rc = upload(D, rf, &d.rec_f)) || (rc = upload(D, rg, &d.rec_g))) return bail(rc);
        d.nb = c->n_boundaries; d.nr = c->n_reconstruction;
    }
    {   // error flag in mapped pinned host memory: the kernels write it (over PCIe) only when a symbol is out of range,
        // the host reads it without a device->host copy
        void *hp = nullptr, *dp = nullptr;
        if (cudaHostAlloc(&hp, sizeof(int), cudaHostAllocMapped) != cudaSuccess || cudaHostGetDevicePointer(&dp, hp, 0) != cudaSuccess)
            return bail(fail(PD_ECUDA, "cudaHostAlloc (mapped) failed"));
        D->h_err = (volatile int *)hp;
        *D->h_err = 0;
        D->d_err = (int *)dp;
    }
    if (d.L > kMaxL) {   // path_cta only: the generic kernel's control block and path_warp's lanes stop at 32 paths
        if (const char *why = plan_path_cta(D->dev, &D->cta)) return bail(fail(PD_ECUDA, "path_cta (N=%d, L=%d): %s", N, d.L, why));
        D->kernel_name = "path_cta";
    } else {
        if ((rc = plan_generic(D))) return bail(rc);
        plan_path_warp(D->dev, &D->path);
        if (const char *e = getenv("POLAR_B200_FORCE_GENERIC")) D->force = atoi(e);
        D->kernel_name = (D->fast.ok && D->force == 0) ? D->fast.name : (D->path.ok && D->force != 1) ? "path_warp" : "generic";
    }
    // a LUT class that falls off the nibble kernel runs 3-100x slower: say so once per reason (POLAR_B200_QUIET=1 silences it)
    if (d.domain == DOM_LUT && !D->fast.ok && D->force == 0 && *D->fast.why && !getenv("POLAR_B200_QUIET")) {
        static std::mutex mu;
        static std::vector<std::string> seen;
        std::lock_guard<std::mutex> lk(mu);
        const std::string key = std::string(D->fast.why) + "/" + D->kernel_name;
        if (std::find(seen.begin(), seen.end(), key) == seen.end()) {
            seen.push_back(key);
            fprintf(stderr, "[polar_b200] note: this LUT decoder (N=%d, L=%d) runs on the '%s' kernel, not 'scl_lut_warp': %s\n",
                    N, d.list ? d.L : 1, D->kernel_name, D->fast.why);
        }
    }
    size_t in_frame = (size_t)N * (d.domain == DOM_LUT ? 4 : 8);
    D->chunk_frames = std::max<int64_t>(1024, (int64_t)((32u << 20) / in_frame));
    D->cfg.take(c);
    *out = D;
    return PD_OK;
}

int pd_set_devices(pd_decoder *D, int32_t n, const int32_t *ids) {
    if (!D || n < 0 || (n > 0 && !ids)) return fail(PD_EINVAL, "null argument");
    for (pd_decoder *c : D->clones) pd_destroy(c);
    D->clones.clear();
    D->units.clear();
    if (n == 0) return PD_OK;
    if (n > 64) return fail(PD_EINVAL, "at most 64 devices");
    bool self_used = false;
    for (int i = 0; i < n; ++i) {
        if (ids[i] == D->device && !self_used) { D->units.push_back(D); self_used = true; continue; }
        pd_config c = D->cfg.c;
        c.device = ids[i];
        pd_decoder *clone = nullptr;
        const int rc = pd_create(&c, &clone);
        if (rc != PD_OK) {
            for (pd_decoder *q : D->clones) pd_destroy(q);
            D->clones.clear();
            D->units.clear();
            return rc;
        }
        clone->force = D->force;
        D->clones.push_back(clone);
        D->units.push_back(clone);
    }
    CUDA_TRY(cudaSetDevice(D->device));
    return PD_OK;
}
int32_t pd_device_count(const pd_decoder *D) { return D ? (int32_t)std::max<size_t>(1, D->units.size()) : 0; }

int pd_counters_allreduce(pd_decoder *D, unsigned long long *const *dev_counters, int32_t n) {
    // sums the n per-device counter pairs {bit errors, block errors} (pd_count_errors) and writes the total back to each of
    // them.  One process drives all GPUs here, so 16 bytes per device travel through the host; the one-process-per-GPU
    // front-end (bench.py, simulate.py under torchrun) all-reduces the same two words with NCCL over NVLink instead.
    if (!D || !dev_counters || n < 1 || n != pd_device_count(D)) return fail(PD_EINVAL, "need one counter buffer per device of the decoder");
    unsigned long long tot[2] = {0, 0}, v[2];
    for (int i = 0; i < n; ++i) {
        const pd_decoder *u = D->units.empty() ? D : D->units[i];
        CUDA_TRY(cudaSetDevice(u->device));
        CUDA_TRY(cudaMemcpy(v, dev_counters[i], sizeof v, cudaMemcpyDeviceToHost));
        tot[0] += v[0]; tot[1] += v[1];
    }
    for (int i = 0; i < n; ++i) {
        const pd_decoder *u = D->units.empty() ? D : D->units[i];
        CUDA_TRY(cudaSetDevice(u->device));
        CUDA_TRY(cudaMemcpy(dev_counters[i], tot, sizeof tot, cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaSetDevice(D->device));
    return PD_OK;
}

int pd_out_len(const pd_decoder *D) { return D ? D->dev.Kout : 0; }
int64_t pd_wave_frames(const pd_decoder *D, int in_dtype) { return D ? wave_frames(D, in_dtype, nullptr) : 0; }
int pd_code_len(const pd_decoder *D) { return D ? D->dev.N : 0; }
const char *pd_kernel_name(const pd_decoder *D) { return D ? D->kernel_name : ""; }
const char *pd_kernel_note(const pd_decoder *D) { return (D && !D->fast.ok && D->dev.domain == DOM_LUT) ? D->fast.why : ""; }

int pd_schedule_stats(const pd_decoder *D, int64_t *n_steps, int64_t *elem_ops, int64_t *n_sorts) {
    if (!D) return fail(PD_EINVAL, "null decoder");
    if (n_steps) *n_steps = (int64_t)D->steps.size();
    if (elem_ops) *elem_ops = D->elem_ops;
    if (n_sorts) *n_sorts = D->n_sorts;
    return PD_OK;
}

int pd_set_debug_outputs(pd_decoder *D, double *dev_pm, int32_t *dev_winner) {
    if (!D) return fail(PD_EINVAL, "null decoder");
    D->dbg_pm = dev_pm;
    D->dbg_win = dev_winner;
    return PD_OK;
}

int pd_decode_device(pd_decoder *D, const void *dev_in, int in_dtype, int64_t B, uint8_t *dev_out, void *cuda_stream) {
    if (!D || (B > 0 && (!dev_in || !dev_out))) return fail(PD_EINVAL, "null argument");
    int rc = check_dtype(D, in_dtype);
    if (rc) return rc;
    if (B <= 0) return PD_OK;
    CUDA_TRY(cudaSetDevice(D->device));
    cudaStream_t s = (cudaStream_t)cuda_stream;
    // One launch per call for the plain scl_lut_warp kernels: their warps take frame groups from a counter, so the launch
    // has no tail, and one value workspace (72 MB at N=1024, L=8) stays L2-resident.
    // The other persistent kernels (path_warp, with its static schedule, and the Fast-SSC variants of scl_lut_warp, which
    // are instruction-fetch bound and run 30 % faster when the warps of an SM start their walks together) get their batch in
    // pieces of ONE wave, issued alternately on two internal streams forked from / joined to the caller's stream with
    // events: the CTAs of piece k+1 move into the slots that the CTAs of piece k vacate, so nothing idles between pieces.
    // POLAR_B200_FORCE_SPLIT=0/1 overrides, POLAR_B200_PIECE_WAVES sets the piece size.
    const size_t esz = dtype_size(in_dtype), N = D->dev.N, Ko = D->dev.Kout;
    const int64_t wave = wave_frames(D, in_dtype, dev_in);
    static const int force_split = getenv("POLAR_B200_FORCE_SPLIT") ? atoi(getenv("POLAR_B200_FORCE_SPLIT")) : -1;
    static const int piece_waves = getenv("POLAR_B200_PIECE_WAVES") ? std::max(1, atoi(getenv("POLAR_B200_PIECE_WAVES"))) : 1;
    const bool dynamic_kernel = want_fast(D, in_dtype, dev_in) && !D->fast.fastk;
    const bool split = force_split == 0 ? false
                                        : ((force_split == 1 || !dynamic_kernel) && wave > 0 && B >= 2 * wave * piece_waves && ((N * esz) % 16 == 0));
    const int64_t per = split ? wave * piece_waves : B;
    const int pieces = split ? (int)((B + per - 1) / per) : 1;
    // workspace: one region per concurrently running piece
    const size_t need1 = ws_need(D, in_dtype, dev_in, per);
    const size_t need = need1 * (split ? 2 : 1);
    if (need > D->ws_user_cap) {
        CUDA_TRY(cudaDeviceSynchronize());
        cudaFree(D->ws_user);
        D->ws_user = nullptr; D->ws_user_cap = 0;
        CUDA_TRY(cudaMalloc((void **)&D->ws_user, need));
        D->ws_user_cap = need;
    }
    if (!split) return launch(D, dev_in, in_dtype, B, dev_out, s, D->ws_user);
    if (!D->fork_ev) {
        CUDA_TRY(cudaEventCreateWithFlags(&D->fork_ev, cudaEventDisableTiming));
        for (int i = 0; i < 2; ++i) {
            CUDA_TRY(cudaEventCreateWithFlags(&D->join_ev[i], cudaEventDisableTiming));
            CUDA_TRY(cudaStreamCreateWithFlags(&D->side[i], cudaStreamNonBlocking));
        }
    }
    CUDA_TRY(cudaEventRecord(D->fork_ev, s));
    for (int i = 0; i < 2; ++i) CUDA_TRY(cudaStreamWaitEvent(D->side[i], D->fork_ev, 0));
    // Both pieces in flight use a full grid and their own value workspace (2 x 52 MB at N=1024, L=8): together with the
    // streaming input / output that exceeds the 126 MB L2, so part of the workspace is written back and re-read (ncu,
    // --cache-control none: 5.2 KB of DRAM traffic per frame vs 1.5 KB algorithmic = 65 GB/s, 1 % of the HBM peak).
    for (int pc = 0; pc < pieces; ++pc) {
        const int64_t f0 = (int64_t)pc * per, nb = std::min<int64_t>(per, B - f0);
        if (nb <= 0) break;
        const int w = pc & 1;
        if ((rc = launch(D, (const char *)dev_in + (size_t)f0 * N * esz, in_dtype, nb, dev_out + (size_t)f0 * Ko, D->side[w],
                         D->ws_user ? D->ws_user + (size_t)w * need1 : nullptr)))
            return rc;
    }
    for (int i = 0; i < 2; ++i) {
        CUDA_TRY(cudaEventRecord(D->join_ev[i], D->side[i]));
        CUDA_TRY(cudaStreamWaitEvent(s, D->join_ev[i], 0));
    }
    return PD_OK;
}

int pd_check(pd_decoder *D, void *cuda_stream) {
    if (!D) return fail(PD_EINVAL, "null decoder");
    CUDA_TRY(cudaSetDevice(D->device));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)cuda_stream));
    if (*D->h_err) {
        *D->h_err = 0;
        return fail(PD_ERANGE, "an input symbol is outside the root lookup table (valid: [0,%d) for the first half, [0,%d) for the second)", D->dev.root_qa, D->dev.root_qb);
    }
    return PD_OK;
}

// ---- blind-detection kinds ------------------------------------------------------------------------
int pd_decode_bd_device(pd_decoder *D, const double *dev_llr, int64_t B, const int32_t *dev_rnti, int32_t rnti_len,
                        uint8_t *dev_bits, double *dev_metric, uint8_t *dev_pass, void *cuda_stream) {
    if (!D || (B > 0 && (!dev_llr || !dev_metric))) return fail(PD_EINVAL, "null argument");
    if (D->dev.bd == 0) return fail(PD_EINVAL, "pd_decode_bd: the decoder is not a PD_BD_* kind");
    if (D->dev.bd == 2) {
        if (B > 0 && (!dev_bits || !dev_pass)) return fail(PD_EINVAL, "null argument");
        if (rnti_len < 0 || rnti_len > D->dev.crc_n || (rnti_len > 0 && !dev_rnti)) return fail(PD_EINVAL, "RNTI length %d must be in [0,crc_n=%d]", rnti_len, D->dev.crc_n);
    }
    if (B <= 0) return PD_OK;
    CUDA_TRY(cudaSetDevice(D->device));
    cudaStream_t s = (cudaStream_t)cuda_stream;
    const size_t need = ws_need(D, PD_F64, dev_llr, B);
    if (need > D->ws_user_cap) {
        CUDA_TRY(cudaDeviceSynchronize());
        cudaFree(D->ws_user);
        D->ws_user = nullptr; D->ws_user_cap = 0;
        CUDA_TRY(cudaMalloc((void **)&D->ws_user, need));
        D->ws_user_cap = need;
    }
    // per-call pointers ride in the descriptor, which every launch copies by value
    Dev &d = D->dev;
    d.bd_rnti = dev_rnti; d.bd_rnti_len = d.bd == 2 ? rnti_len : 0; d.bd_metric = dev_metric; d.bd_pass = dev_pass;
    const int rc = launch(D, dev_llr, PD_F64, B, d.bd == 2 ? dev_bits : nullptr, s, D->ws_user);
    d.bd_rnti = nullptr; d.bd_rnti_len = 0; d.bd_metric = nullptr; d.bd_pass = nullptr;
    return rc;
}

int pd_decode_bd(pd_decoder *D, const double *llr, int64_t B, const int32_t *rnti, int32_t rnti_len,
                 uint8_t *out_bits, double *out_metric, uint8_t *out_pass) {
    if (!D || (B > 0 && (!llr || !out_metric))) return fail(PD_EINVAL, "null argument");
    if (D->dev.bd == 0) return fail(PD_EINVAL, "pd_decode_bd: the decoder is not a PD_BD_* kind");
    const bool ca = D->dev.bd == 2;
    if (ca && B > 0 && (!out_bits || !out_pass)) return fail(PD_EINVAL, "null argument");
    if (ca && (rnti_len < 0 || rnti_len > D->dev.crc_n || (rnti_len > 0 && !rnti))) return fail(PD_EINVAL, "RNTI length %d must be in [0,crc_n=%d]", rnti_len, D->dev.crc_n);
    if (B <= 0) return PD_OK;
    CUDA_TRY(cudaSetDevice(D->device));
    const size_t N = D->dev.N, Ko = D->dev.Kout;
    const int64_t chunk = std::min<int64_t>(B, std::max<int64_t>(1024, (int64_t)((32u << 20) / (N * 8))));
    double *d_in = nullptr, *d_metric = nullptr;
    uint8_t *d_bits = nullptr, *d_pass = nullptr;
    int32_t *d_rnti = nullptr;
    int rc = PD_OK;
    auto cleanup = [&]() { cudaFree(d_in); cudaFree(d_metric); cudaFree(d_bits); cudaFree(d_pass); cudaFree(d_rnti); };
    if (cudaMalloc((void **)&d_in, (size_t)chunk * N * 8) != cudaSuccess || cudaMalloc((void **)&d_metric, (size_t)chunk * 8) != cudaSuccess ||
        cudaMalloc((void **)&d_bits, std::max<size_t>((size_t)chunk * Ko, 16)) != cudaSuccess || cudaMalloc((void **)&d_pass, (size_t)chunk) != cudaSuccess ||
        cudaMalloc((void **)&d_rnti, std::max<size_t>((size_t)rnti_len * 4, 16)) != cudaSuccess) {
        cleanup();
        cudaGetLastError();
        return fail(PD_ENOMEM, "cudaMalloc failed");
    }
    cudaStream_t s = nullptr;
    if (ca && rnti_len > 0 && cudaMemcpyAsync(d_rnti, rnti, (size_t)rnti_len * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) rc = fail(PD_ECUDA, "H2D copy failed");
    for (int64_t f0 = 0; f0 < B && rc == PD_OK; f0 += chunk) {
        const int64_t nb = std::min<int64_t>(chunk, B - f0);
        if (cudaMemcpyAsync(d_in, llr + (size_t)f0 * N, (size_t)nb * N * 8, cudaMemcpyHostToDevice, s) != cudaSuccess) { rc = fail(PD_ECUDA, "H2D copy failed"); break; }
        if ((rc = pd_decode_bd_device(D, d_in, nb, d_rnti, rnti_len, d_bits, d_metric, d_pass, s))) break;
        bool ok = cudaMemcpyAsync(out_metric + f0, d_metric, (size_t)nb * 8, cudaMemcpyDeviceToHost, s) == cudaSuccess;
        if (ca) {
            ok = ok && cudaMemcpyAsync(out_bits + (size_t)f0 * Ko, d_bits, (size_t)nb * Ko, cudaMemcpyDeviceToHost, s) == cudaSuccess;
            ok = ok && cudaMemcpyAsync(out_pass + f0, d_pass, (size_t)nb, cudaMemcpyDeviceToHost, s) == cudaSuccess;
        }
        if (!ok) { rc = fail(PD_ECUDA, "D2H copy failed"); break; }
        rc = pd_check(D, s);
    }
    cleanup();
    return rc;
}

int pd_decode(pd_decoder *D, const void *host_in, int in_dtype, int64_t B, uint8_t *host_out) {
    if (!D || (B > 0 && (!host_in || !host_out))) return fail(PD_EINVAL, "null argument");
    int rc = check_dtype(D, in_dtype, true);
    if (rc) return rc;
    if (B <= 0) return PD_OK;
    CUDA_TRY(cudaSetDevice(D->device));
    const size_t esz = dtype_size(in_dtype), N = D->dev.N, Ko = D->dev.Kout;
    const bool f64_symbols = in_dtype == PD_F64 && D->dev.domain == DOM_LUT;
    if (B * N * esz <= kSmallIn && B * Ko <= kSmallOut && !getenv("POLAR_B200_NO_MAPPED_IO")) {
        StreamSlot &sl = D->slot[0];
        if (!sl.stream) CUDA_TRY(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
        if (!D->h_small) {
            void *hp = nullptr, *dp = nullptr;
            CUDA_TRY(cudaHostAlloc(&hp, kSmallIn + kSmallOut, cudaHostAllocMapped));
            if (cudaHostGetDevicePointer(&dp, hp, 0) != cudaSuccess) { cudaFreeHost(hp); return fail(PD_ECUDA, "cudaHostGetDevicePointer failed"); }
            D->h_small = (char *)hp; D->d_small = (char *)dp;
        }
        const int small_dtype = f64_symbols ? PD_U8 : in_dtype;
        const size_t wsn = std::max(ws_need(D, small_dtype, D->d_small, B), (size_t)16);
        if (sl.ws_cap < wsn) { cudaFree(sl.ws); sl.ws = nullptr; sl.ws_cap = 0; CUDA_TRY(cudaMalloc((void **)&sl.ws, wsn)); sl.ws_cap = wsn; }
        if (f64_symbols) {
            if (!narrow_f64_to_u8((const double *)host_in, (uint8_t *)D->h_small, (size_t)B * N)) return fail(PD_ERANGE, "input symbol outside 0..255");
        } else {
            memcpy(D->h_small, host_in, (size_t)B * N * esz);
        }
        if ((rc = launch(D, D->d_small, small_dtype, B, reinterpret_cast<uint8_t *>(D->d_small + kSmallIn), sl.stream, sl.ws))) return rc;
        if ((rc = pd_check(D, sl.stream))) return rc;
        memcpy(host_out, D->h_small + kSmallIn, (size_t)B * Ko);
        return PD_OK;
    }
    // pipeline chunk: ~16 MB of symbols, a whole number of kernel waves when the kernel is persistent.  Chunks are dealt
    // round-robin to the decoder's units (pd_set_devices: this GPU and clones on others; default: this GPU alone), two
    // stream slots per unit, so that the copies of one chunk hide behind the kernel of another.
    std::vector<pd_decoder *> units = D->units.empty() ? std::vector<pd_decoder *>{D} : D->units;
    const int U = (int)units.size();
    const bool narrow = (in_dtype == PD_I32 && D->fast.ok && D->force == 0) || f64_symbols;   // int32 / float64-typed symbols travel as bytes
    const size_t dsz = narrow ? 1 : esz;                                        // element size on the device
    const int dev_dtype = narrow ? PD_U8 : in_dtype;
    int64_t chunk = std::max<int64_t>(8192, (int64_t)((16u << 20) / (N * dsz)));
    if (const int64_t wave = wave_frames(D, dev_dtype, nullptr)) chunk = std::max<int64_t>(1, (chunk + wave / 2) / wave) * wave;
    if (const char *e = getenv("POLAR_B200_CHUNK_FRAMES")) chunk = std::max(1, atoi(e));      // (tests: force many small chunks)
    chunk = std::min<int64_t>(B, chunk);
    // the caller's buffers go through pinned staging memory unless they are pinned already (pd_host_alloc / cudaHostRegister):
    // a cudaMemcpyAsync from pageable memory is neither asynchronous nor fast
    const bool stage_in = narrow || !is_pinned(host_in), stage_out = !is_pinned(host_out);
    for (pd_decoder *u : units) {
        CUDA_TRY(cudaSetDevice(u->device));
        for (auto &sl : u->slot) {
            if (!sl.stream) CUDA_TRY(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
            if (!sl.done) CUDA_TRY(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
            size_t in_need = (size_t)chunk * N * dsz, out_need = (size_t)chunk * Ko;
            if (sl.in_cap < in_need) { cudaFree(sl.d_in); sl.d_in = nullptr; sl.in_cap = 0; CUDA_TRY(cudaMalloc(&sl.d_in, in_need)); sl.in_cap = in_need; }
            if (sl.out_cap < out_need) { cudaFree(sl.d_out); sl.d_out = nullptr; sl.out_cap = 0; CUDA_TRY(cudaMalloc((void **)&sl.d_out, out_need)); sl.out_cap = out_need; }
            if (stage_in && sl.h_in_cap < in_need) { if (sl.h_in) cudaFreeHost(sl.h_in); sl.h_in = nullptr; sl.h_in_cap = 0; CUDA_TRY(cudaHostAlloc((void **)&sl.h_in, in_need, cudaHostAllocPortable)); sl.h_in_cap = in_need; }
            if (stage_out && sl.h_out_cap < out_need) { if (sl.h_out) cudaFreeHost(sl.h_out); sl.h_out = nullptr; sl.h_out_cap = 0; CUDA_TRY(cudaHostAlloc((void **)&sl.h_out, out_need, cudaHostAllocPortable)); sl.h_out_cap = out_need; }
            // our own staging buffers are cudaMalloc'ed (256-B aligned), so the kernel choice depends on the dtype only
            size_t wsn = std::max(ws_need(u, dev_dtype, nullptr, chunk), (size_t)16);
            if (sl.ws_cap < wsn) { cudaFree(sl.ws); sl.ws = nullptr; sl.ws_cap = 0; CUDA_TRY(cudaMalloc((void **)&sl.ws, wsn)); sl.ws_cap = wsn; }
        }
    }
    static const bool trace = getenv("POLAR_B200_TRACE") != nullptr;
#define PD_TRACE(...) do { if (trace) { fprintf(stderr, "[pd_decode] " __VA_ARGS__); fputc('\n', stderr); fflush(stderr); } } while (0)
    PD_TRACE("B=%lld chunk=%lld units=%d narrow=%d stage_in=%d stage_out=%d", (long long)B, (long long)chunk, U, (int)narrow, (int)stage_in, (int)stage_out);
    HostPool &pool = HostPool::get();
    const int parts = pool.size();
    PD_TRACE("pool of %d threads", parts);
    std::atomic<int> bad_value{0};
    const int n_slots = 2 * U;
    std::vector<int64_t> pend_f0(n_slots, -1), pend_nb(n_slots, 0);
    // waits for the chunk that occupies slot w (unit w % U, its slot w / U) and copies its result to the caller's output
    auto drain = [&](int w) -> int {
        if (pend_f0[w] < 0) return PD_OK;
        pd_decoder *u = units[w % U];
        StreamSlot &sl = u->slot[w / U];
        CUDA_TRY(cudaSetDevice(u->device));
        PD_TRACE("drain slot %d: wait", w);
        CUDA_TRY(cudaEventSynchronize(sl.done));     // the chunk's copies are done: both pinned areas of the slot are free again
        PD_TRACE("drain slot %d: done", w);
        if (stage_out) {
            const size_t bytes = (size_t)pend_nb[w] * Ko, per = (bytes / parts + 63) & ~(size_t)63;
            uint8_t *dst = host_out + (size_t)pend_f0[w] * Ko;
            const char *src = sl.h_out;
            pool.run(parts, [&](int i) {
                const size_t o = (size_t)i * per;
                if (o < bytes) memcpy(dst + o, src + o, std::min(per, bytes - o));
            });
        }
        pend_f0[w] = -1;
        return PD_OK;
    };
    int which = 0;
    for (int64_t f0 = 0; f0 < B; f0 += chunk, which = (which + 1) % n_slots) {
        pd_decoder *u = units[which % U];
        StreamSlot &sl = u->slot[which / U];
        const int64_t nb = std::min<int64_t>(chunk, B - f0);
        if ((rc = drain(which))) return rc;          // the slot's previous chunk
        CUDA_TRY(cudaSetDevice(u->device));
        const void *h2d_src = (const char *)host_in + (size_t)f0 * N * esz;
        if (stage_in) {
            const size_t elems = (size_t)nb * N, per = ((elems / parts) + 63) & ~(size_t)63;
            const char *src = (const char *)h2d_src;
            char *dst = sl.h_in;
            pool.run(parts, [&](int i) {
                const size_t o = (size_t)i * per;
                if (o >= elems) return;
                const size_t n = std::min(per, elems - o);
                if (f64_symbols) { if (!narrow_f64_to_u8((const double *)src + o, (uint8_t *)dst + o, n)) bad_value = 1; }
                else if (narrow) { if (!narrow_i32_to_u8((const int32_t *)src + o, (uint8_t *)dst + o, n)) bad_value = 1; }
                else memcpy(dst + o * esz, src + o * esz, n * esz);
            });
            h2d_src = sl.h_in;
        }
        PD_TRACE("chunk at %lld (%lld frames) staged -> slot %d", (long long)f0, (long long)nb, which);
        CUDA_TRY(cudaMemcpyAsync(sl.d_in, h2d_src, (size_t)nb * N * dsz, cudaMemcpyHostToDevice, sl.stream));
        if ((rc = launch(u, sl.d_in, dev_dtype, nb, sl.d_out, sl.stream, sl.ws))) return rc;
        PD_TRACE("chunk at %lld launched", (long long)f0);
        CUDA_TRY(cudaMemcpyAsync(stage_out ? (void *)sl.h_out : (void *)(host_out + (size_t)f0 * Ko), sl.d_out, (size_t)nb * Ko, cudaMemcpyDeviceToHost, sl.stream));
        CUDA_TRY(cudaEventRecord(sl.done, sl.stream));
        pend_f0[which] = f0; pend_nb[which] = nb;
    }
    for (int k = 0; k < n_slots; ++k, which = (which + 1) % n_slots)
        if ((rc = drain(which))) return rc;
    PD_TRACE("all chunks drained");
    rc = PD_OK;
    for (pd_decoder *u : units) {
        CUDA_TRY(cudaSetDevice(u->device));
        for (auto &sl : u->slot) {
            const int r2 = pd_check(u, sl.stream);
            if (r2 != PD_OK && rc == PD_OK) rc = r2;
        }
    }
    CUDA_TRY(cudaSetDevice(D->device));
    if (rc == PD_OK && bad_value.load())
        return fail(PD_ERANGE, "an input symbol is outside the root lookup table (valid: [0,%d) for the first half, [0,%d) for the second)", D->dev.root_qa, D->dev.root_qb);
    return rc;
}

#ifndef PB_HOST_EMU
// ---- simulation-mode error counters -------------------------------------------------------------
// `lpf` lanes per frame (a power of two, 32 / lpf frames per warp): the lanes read the two rows with 16-byte loads (rows of a
// multiple of 16 bytes at 16-byte aligned bases: lpf = len / 16 rounded up to a power of two, at most 32; else byte by
// byte, lane-strided, a warp per frame) -- HBM-bound, 2 * len bytes per frame.
__device__ __forceinline__ unsigned nonzero_bytes(uint32_t x) {
    return (unsigned)__popc((((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u);
}
__global__ void count_errors_kernel(const uint8_t *__restrict__ a, const uint8_t *__restrict__ b, long long B, int len, int lpf, int vec,
                                    unsigned long long *counters) {
    const int lane = threadIdx.x & 31, li = lane & (lpf - 1), sub = lane / lpf, fpw = 32 / lpf;
    const unsigned gmask = (lpf == 32 ? 0xffffffffu : ((1u << lpf) - 1u)) << (sub * lpf);
    const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    unsigned long long bits = 0, blocks = 0;
    for (long long base = warp * fpw; base < B; base += n_warps * fpw) {
        const long long f = base + sub;
        unsigned e = 0;
        if (f < B) {
            const uint8_t *pa = a + (size_t)f * len, *pb = b + (size_t)f * len;
            if (vec) {
                for (int k = li * 16; k < len; k += lpf * 16) {
                    const uint4 x = __ldcs(reinterpret_cast<const uint4 *>(pa + k)), y = __ldcs(reinterpret_cast<const uint4 *>(pb + k));
                    e += nonzero_bytes(x.x ^ y.x) + nonzero_bytes(x.y ^ y.y) + nonzero_bytes(x.z ^ y.z) + nonzero_bytes(x.w ^ y.w);
                }
            } else {
                for (int k = li; k < len; k += lpf) e += (pa[k] != pb[k]);
            }
        }
        bits += e;
        if ((__ballot_sync(0xffffffffu, e != 0) & gmask) != 0u && li == 0) blocks++;
    }
    for (int o = 16; o > 0; o >>= 1) {
        bits += __shfl_down_sync(0xffffffffu, bits, o);
        blocks += __shfl_down_sync(0xffffffffu, blocks, o);
    }
    if (lane == 0) {
        if (bits) atomicAdd(&counters[0], bits);
        if (blocks) atomicAdd(&counters[1], blocks);
    }
}

int pd_count_errors(const uint8_t *dev_decoded, const uint8_t *dev_truth, int64_t B, int32_t len,
                    unsigned long long *dev_counters, void *cuda_stream) {
    if (B <= 0) return PD_OK;
    if (!dev_decoded || !dev_truth || !dev_counters || len < 1) return fail(PD_EINVAL, "null argument");
    const int vec = (len % 16 == 0) && (reinterpret_cast<uintptr_t>(dev_decoded) % 16 == 0) && (reinterpret_cast<uintptr_t>(dev_truth) % 16 == 0);
    int lpf = 32;
    if (vec) { lpf = 1; while (lpf < 32 && lpf * 16 < len) lpf *= 2; }
    const int threads = 256, fpb = (threads / 32) * (32 / lpf);      // frames per block and iteration
    const int grid = (int)std::min<int64_t>((B + fpb - 1) / fpb, (int64_t)current_sm_count() * 8);
    count_errors_kernel<<<grid, threads, 0, (cudaStream_t)cuda_stream>>>(dev_decoded, dev_truth, B, len, lpf, vec, dev_counters);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return PD_OK;
}

// ---- on-device frame generator -------------------------------------------------------------------
}  // extern "C"
struct pd_sim {
    SimDev dev{};
    int device = 0;
    const EncWord *enc_tab = nullptr;   // N <= 1024: per-word deposit description of the register encoder
    std::vector<void *> allocs;
};
extern "C" {

void pd_sim_destroy(pd_sim *S) {
    if (!S) return;
    cudaSetDevice(S->device);
    for (void *p : S->allocs) cudaFree(p);
    delete S;
}

// copies `bytes` host bytes into a new device buffer owned by S (freed by pd_sim_destroy)
static int sim_upload(pd_sim *S, const void *h, size_t bytes, const void **dst) {
    void *p = nullptr;
    if (cudaMalloc(&p, std::max<size_t>(bytes, 16)) != cudaSuccess) return fail(PD_ECUDA, "cudaMalloc failed");
    S->allocs.push_back(p);
    if (bytes && cudaMemcpy(p, h, bytes, cudaMemcpyHostToDevice) != cudaSuccess) return fail(PD_ECUDA, "cudaMemcpy failed");
    *dst = p;
    return PD_OK;
}

int pd_sim_create(const pd_sim_config *c, pd_sim **out) {
    if (!c || !out || !c->frozen_bits) return fail(PD_EINVAL, "null argument");
    *out = nullptr;
    const int N = c->N;
    if (N < 32 || N > (1 << kMaxLog) || (N & (N - 1))) return fail(PD_EINVAL, "N=%d must be a power of two in [32,%d]", N, 1 << kMaxLog);
    std::vector<int32_t> info_pos;
    for (int i = 0; i < N; ++i) if (c->frozen_bits[i] == 0) info_pos.push_back(i);
    if ((int)info_pos.size() != c->K) return fail(PD_EINVAL, "K=%d but frozen_bits has %zu non-frozen positions", c->K, info_pos.size());
    if (c->crc_n < 0 || c->crc_n > 32) return fail(PD_EINVAL, "crc_n must be in [0,32]");
    if (c->A < 1 || c->A + c->crc_n != c->K) return fail(PD_EINVAL, "need K == A + crc_n");
    if (c->edges && (c->n_edges < 2 || !c->chan_lut || c->q_channel < 1 || c->q_channel > 256)) return fail(PD_EINVAL, "bad channel quantizer");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PD_ECUDA, "no CUDA device");
    if (c->device < 0 || c->device >= ndev) return fail(PD_EINVAL, "device %d out of range", c->device);
    CUDA_TRY(cudaSetDevice(c->device));
    pd_sim *S = new pd_sim();
    S->device = c->device;
    SimDev &d = S->dev;
    d.N = N; d.K = c->K; d.A = c->A; d.crc_n = c->crc_n;
    int rc;
    if ((rc = sim_upload(S, info_pos.data(), info_pos.size() * 4, (const void **)&d.info_pos))) { pd_sim_destroy(S); return rc; }
    std::vector<uint32_t> rem(c->A, 0);
    if (c->crc_n > 0) {
        std::vector<int> poly(c->crc_n + 1, 0);
        for (int i = 0; i < c->crc_loc_len; ++i) {
            if (c->crc_loc[i] < 0 || c->crc_loc[i] > c->crc_n) { pd_sim_destroy(S); return fail(PD_EINVAL, "crc_p entry out of range"); }
            poly[c->crc_loc[i]] = 1;
        }
        uint32_t taps = 0;
        for (int k = 0; k < c->crc_n; ++k) if (poly[1 + k]) taps |= 1u << (c->crc_n - 1 - k);
        const uint32_t msb = 1u << (c->crc_n - 1), mask = c->crc_n >= 32 ? 0xffffffffu : ((1u << c->crc_n) - 1u);
        for (int k = 0; k < c->A; ++k) {
            uint32_t reg = 0;
            for (int i = k; i < c->A; ++i) {
                uint32_t top = ((reg & msb) ? 1u : 0u) ^ (i == k ? 1u : 0u);
                reg = (reg << 1) & mask;
                if (top) reg ^= taps;
            }
            rem[k] = reg;
        }
    }
    if ((rc = sim_upload(S, rem.data(), rem.size() * 4, (const void **)&d.crc_rem))) { pd_sim_destroy(S); return rc; }
    if (N <= 1024) {
        std::vector<EncWord> tab(32);
        memset(tab.data(), 0, tab.size() * sizeof(EncWord));
        uint32_t before = 0;
        for (int w = 0; w < N / 32; ++w) {
            uint32_t m = 0;
            for (int b = 0; b < 32; ++b) if (c->frozen_bits[32 * w + b] == 0) m |= 1u << b;
            tab[w].mask = m;
            tab[w].kstart = before;
            enc_expand_masks(m, tab[w].mv);
            before += (uint32_t)__builtin_popcount(m);
        }
        if ((rc = sim_upload(S, tab.data(), tab.size() * sizeof(EncWord), (const void **)&S->enc_tab))) { pd_sim_destroy(S); return rc; }
    }
    if (c->edges) {
        if ((rc = sim_upload(S, c->edges, (size_t)c->n_edges * 8, (const void **)&d.edges)) ||
            (rc = sim_upload(S, c->chan_lut, (size_t)(c->n_edges - 1), (const void **)&d.chan_lut))) { pd_sim_destroy(S); return rc; }
        d.n_edges = c->n_edges;
        d.q_channel = c->q_channel;
        d.mode = PD_SIM_LLR_QUANT;
    } else {
        d.mode = PD_SIM_LLR;
    }
    *out = S;
    return PD_OK;
}

int pd_sim_set_channel(pd_sim *S, const pd_sim_channel *ch) {
    if (!S || !ch) return fail(PD_EINVAL, "null argument");
    SimDev d = S->dev;
    d.edges = nullptr; d.n_edges = 0; d.chan_lut = nullptr; d.q_channel = 0;
    d.r = d.bound = d.sat = 0.0;
    d.mode = ch->mode;
    const bool llr_quant = ch->mode == PD_SIM_LLR_QUANT, y_quant = ch->mode == PD_SIM_Y_QUANT;
    if (llr_quant || y_quant) {
        if (!ch->edges) return fail(PD_EINVAL, "edges is NULL");
        if (ch->n_edges < 2) return fail(PD_EINVAL, "n_edges=%d: need at least 2 edges", ch->n_edges);
        if (ch->q_channel < 1 || ch->q_channel > 256) return fail(PD_EINVAL, "q_channel=%d must be in [1,256]", ch->q_channel);
        for (int i = 0; i < ch->n_edges; ++i)
            if (std::isnan(ch->edges[i]) || (i > 0 && !(ch->edges[i] >= ch->edges[i - 1])))
                return fail(PD_EINVAL, "edges must be ascending and not NaN (edge %d)", i);
        if (y_quant && ch->n_edges != ch->q_channel + 1)
            return fail(PD_EINVAL, "PD_SIM_Y_QUANT needs n_edges == q_channel + 1 (got n_edges=%d, q_channel=%d)", ch->n_edges, ch->q_channel);
        if (llr_quant) {
            if (!ch->chan_lut) return fail(PD_EINVAL, "chan_lut is NULL");
            for (int i = 0; i < ch->n_edges - 1; ++i)
                if (ch->chan_lut[i] >= ch->q_channel) return fail(PD_EINVAL, "chan_lut[%d]=%d is not below q_channel=%d", i, ch->chan_lut[i], ch->q_channel);
        }
        d.n_edges = ch->n_edges;
        d.q_channel = ch->q_channel;
    } else if (ch->mode == PD_SIM_LLR_UNIFORM) {
        if (!(ch->r > 0) || !std::isfinite(ch->r)) return fail(PD_EINVAL, "r=%g must be finite and > 0", ch->r);
        if (ch->v < 2) return fail(PD_EINVAL, "v=%d must be >= 2", ch->v);
        d.r = ch->r;
        d.bound = ((double)(ch->v / 2) - 0.5) * ch->r;   // M = (v//2 - 0.5)*r and M - 0.5*r, numpy's operation order
        d.sat = d.bound - 0.5 * ch->r;
    } else if (ch->mode != PD_SIM_LLR) {
        return fail(PD_EINVAL, "unknown channel mode %d", ch->mode);
    }
    CUDA_TRY(cudaSetDevice(S->device));
    int rc;
    if (d.n_edges && (rc = sim_upload(S, ch->edges, (size_t)d.n_edges * 8, (const void **)&d.edges))) return rc;
    if (llr_quant && (rc = sim_upload(S, ch->chan_lut, (size_t)(d.n_edges - 1), (const void **)&d.chan_lut))) return rc;
    S->dev = d;
    return PD_OK;
}

int pd_sim_generate(pd_sim *S, double sigma, int64_t B, uint64_t seed, uint64_t first_frame, uint8_t *dev_msg, void *dev_out, void *cuda_stream) {
    if (!S || (B > 0 && (!dev_msg || !dev_out))) return fail(PD_EINVAL, "null argument");
    if (!(sigma > 0)) return fail(PD_EINVAL, "sigma must be > 0");
    if (B <= 0) return PD_OK;
    CUDA_TRY(cudaSetDevice(S->device));
    const int threads = 128, wpb = threads / 32;
    const size_t smem = (size_t)wpb * (S->dev.N / 32) * 4;
    const int grid = (int)std::min<int64_t>((B + wpb - 1) / wpb, (int64_t)current_sm_count() * 16);
    sim_generate_kernel<<<grid, threads, smem, (cudaStream_t)cuda_stream>>>(S->dev, sigma, B, seed, first_frame, dev_msg, dev_out);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return PD_OK;
}

static int enc_lengths(const pd_sim *S, int mode, int *in_len, int *out_len) {
    switch (mode) {
    case PD_ENC_POLAR: *in_len = S->dev.K; *out_len = S->dev.N; return PD_OK;
    case PD_ENC_CRC: *in_len = S->dev.A; *out_len = S->dev.K; break;
    case PD_ENC_CRC_POLAR: *in_len = S->dev.A; *out_len = S->dev.N; break;
    default: return fail(PD_EINVAL, "unknown encoder mode %d", mode);
    }
    if (S->dev.crc_n <= 0) return fail(PD_EINVAL, "this pd_sim was created without a CRC (crc_n = 0)");
    return PD_OK;
}

int pd_sim_encode_device(pd_sim *S, int mode, const uint8_t *dev_in, int64_t B, uint8_t *dev_out, void *cuda_stream) {
    if (!S || (B > 0 && (!dev_in || !dev_out))) return fail(PD_EINVAL, "null argument");
    int in_len = 0, out_len = 0, rc;
    if ((rc = enc_lengths(S, mode, &in_len, &out_len))) return rc;
    if (B <= 0) return PD_OK;
    CUDA_TRY(cudaSetDevice(S->device));
    const int threads = 256, wpb = threads / 32;
    const size_t smem = (size_t)wpb * (S->dev.N / 32) * 4;
    const int grid = (int)std::min<int64_t>((B + wpb - 1) / wpb, (int64_t)current_sm_count() * 8);
    const int vec_ok = ((reinterpret_cast<uintptr_t>(dev_in) & 3) == 0 && (reinterpret_cast<uintptr_t>(dev_out) & 15) == 0) ? 1 : 0;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (mode == PD_ENC_CRC) encode_kernel<ENC_CRC><<<grid, threads, smem, st>>>(S->dev, dev_in, dev_out, B, vec_ok);
    else if (S->enc_tab && mode == PD_ENC_POLAR) encode_words_kernel<ENC_POLAR><<<grid, threads, 0, st>>>(S->dev, S->enc_tab, dev_in, dev_out, B, vec_ok);
    else if (S->enc_tab) encode_words_kernel<ENC_CRC_POLAR><<<grid, threads, 0, st>>>(S->dev, S->enc_tab, dev_in, dev_out, B, vec_ok);
    else if (mode == PD_ENC_POLAR) encode_kernel<ENC_POLAR><<<grid, threads, smem, st>>>(S->dev, dev_in, dev_out, B, vec_ok);
    else encode_kernel<ENC_CRC_POLAR><<<grid, threads, smem, st>>>(S->dev, dev_in, dev_out, B, vec_ok);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return PD_OK;
}

int pd_sim_encode(pd_sim *S, int mode, const uint8_t *in, int64_t B, uint8_t *out) {
    if (!S || (B > 0 && (!in || !out))) return fail(PD_EINVAL, "null argument");
    int in_len = 0, out_len = 0, rc;
    if ((rc = enc_lengths(S, mode, &in_len, &out_len))) return rc;
    if (B <= 0) return PD_OK;
    CUDA_TRY(cudaSetDevice(S->device));
    // bounded staging: chunks of <= 32 MiB of output
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(B, ((int64_t)32 << 20) / out_len));
    uint8_t *d_in = nullptr, *d_out = nullptr;
    if (cudaMalloc(&d_in, (size_t)chunk * in_len) != cudaSuccess) return fail(PD_ENOMEM, "cudaMalloc failed");
    if (cudaMalloc(&d_out, (size_t)chunk * out_len) != cudaSuccess) { cudaFree(d_in); return fail(PD_ENOMEM, "cudaMalloc failed"); }
    rc = PD_OK;
    for (int64_t f0 = 0; f0 < B && rc == PD_OK; f0 += chunk) {
        const int64_t b = std::min(chunk, B - f0);
        if (cudaMemcpyAsync(d_in, in + (size_t)f0 * in_len, (size_t)b * in_len, cudaMemcpyHostToDevice, 0) != cudaSuccess) { rc = fail(PD_ECUDA, "H2D copy failed"); break; }
        if ((rc = pd_sim_encode_device(S, mode, d_in, b, d_out, nullptr))) break;
        if (cudaMemcpyAsync(out + (size_t)f0 * out_len, d_out, (size_t)b * out_len, cudaMemcpyDeviceToHost, 0) != cudaSuccess) { rc = fail(PD_ECUDA, "D2H copy failed"); break; }
        if (cudaStreamSynchronize(0) != cudaSuccess) { rc = fail(PD_ECUDA, "encode failed: %s", cudaGetErrorString(cudaGetLastError())); break; }
    }
    cudaFree(d_in);
    cudaFree(d_out);
    return rc;
}

// ---- lookup-table design: batched minimum-distortion quantizer -----------------------------------------
int pd_optls_quantize(const double *density, const double *quanta, const int32_t *M, int64_t stride, int32_t P, int32_t K,
                      double *out_density, double *out_quanta, int32_t *out_lut, int32_t device) {
    if (P <= 0) return PD_OK;
    if (!density || !quanta || !M || !out_density || !out_quanta || !out_lut) return fail(PD_EINVAL, "null argument");
    if (K < 2 || K > 64) return fail(PD_EINVAL, "K=%d must be in [2,64]", K);
    int maxM = 0;
    for (int p = 0; p < P; ++p) {
        if (M[p] <= K || M[p] > kOptlsMaxM || M[p] > stride) return fail(PD_EINVAL, "problem %d: M=%d must be in (K,%d] and <= stride", p, M[p], kOptlsMaxM);
        for (int i = 1; i < M[p]; ++i)
            if (!(quanta[(size_t)p * stride + i] > quanta[(size_t)p * stride + i - 1])) return fail(PD_EINVAL, "problem %d: quanta must be strictly ascending (pass np.unique output)", p);
        maxM = std::max(maxM, M[p]);
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PD_ECUDA, "no CUDA device: libpolar_b200 has no CPU path");
    if (device < 0 || device >= ndev) return fail(PD_EINVAL, "device %d out of range", device);
    CUDA_TRY(cudaSetDevice(device));
    const int W = maxM - K + 1;
    const long long t_stride = (long long)maxM * W, lm_stride = (long long)(K + 1) * W;
    const int chunk = (int)std::max<long long>(1, std::min<long long>(P, (256ll << 20) / (t_stride * 8)));   // <= 256 MiB of tables in flight
    double *d_d = nullptr, *d_q = nullptr, *d_od = nullptr, *d_oq = nullptr, *d_T = nullptr;
    int32_t *d_M = nullptr, *d_lut = nullptr, *d_lm = nullptr;
    auto cleanup = [&]() { cudaFree(d_d); cudaFree(d_q); cudaFree(d_od); cudaFree(d_oq); cudaFree(d_T); cudaFree(d_M); cudaFree(d_lut); cudaFree(d_lm); };
    if (cudaMalloc((void **)&d_d, (size_t)chunk * stride * 8) != cudaSuccess || cudaMalloc((void **)&d_q, (size_t)chunk * stride * 8) != cudaSuccess ||
        cudaMalloc((void **)&d_od, (size_t)chunk * K * 8) != cudaSuccess || cudaMalloc((void **)&d_oq, (size_t)chunk * K * 8) != cudaSuccess ||
        cudaMalloc((void **)&d_T, (size_t)chunk * t_stride * 8) != cudaSuccess || cudaMalloc((void **)&d_M, (size_t)chunk * 4) != cudaSuccess ||
        cudaMalloc((void **)&d_lut, (size_t)chunk * stride * 4) != cudaSuccess || cudaMalloc((void **)&d_lm, (size_t)chunk * lm_stride * 4) != cudaSuccess) {
        cleanup();
        cudaGetLastError();
        return fail(PD_ENOMEM, "cudaMalloc failed");
    }
    int rc = PD_OK;
    const size_t smem = (size_t)(2 * maxM + 2 * W) * sizeof(double);
    for (int p0 = 0; p0 < P && rc == PD_OK; p0 += chunk) {
        const int np = std::min(chunk, P - p0);
        bool ok = cudaMemcpy(d_d, density + (size_t)p0 * stride, (size_t)np * stride * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
                  cudaMemcpy(d_q, quanta + (size_t)p0 * stride, (size_t)np * stride * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
                  cudaMemcpy(d_M, M + p0, (size_t)np * 4, cudaMemcpyHostToDevice) == cudaSuccess;
        if (!ok) { rc = fail(PD_ECUDA, "H2D copy failed"); break; }
        const cudaError_t le = launch_optls(np, smem, d_d, d_q, d_M, stride, K, d_od, d_oq, d_lut, d_T, d_lm, t_stride, lm_stride);
        g_launches++;
        ok = le == cudaSuccess &&
             cudaMemcpy(out_density + (size_t)p0 * K, d_od, (size_t)np * K * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
             cudaMemcpy(out_quanta + (size_t)p0 * K, d_oq, (size_t)np * K * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
             cudaMemcpy(out_lut + (size_t)p0 * stride, d_lut, (size_t)np * stride * 4, cudaMemcpyDeviceToHost) == cudaSuccess;
        if (!ok) rc = fail(PD_ECUDA, "optls kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    cleanup();
    return rc;
}

// ---- lookup-table design, probability domain: the two device passes of the MMI quantizer (see pb_lutgen.cuh) --------
}  // extern "C"
namespace {
struct DevBufs {
    std::vector<void *> v;
    ~DevBufs() { for (void *p : v) cudaFree(p); }
    template <class T> T *get(size_t n) {
        void *p = nullptr;
        if (cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 16)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        v.push_back(p);
        return reinterpret_cast<T *>(p);
    }
};
int mmi_check(const void *a, const void *b, int32_t P, int32_t M, int32_t K, int32_t device) {
    if (!a || !b) return fail(PD_EINVAL, "null argument");
    if (K < 2 || K > 64 || M < K || M > kOptlsMaxM) return fail(PD_EINVAL, "need 2 <= K <= 64 and K <= M <= %d (K=%d, M=%d)", kOptlsMaxM, K, M);
    if ((long long)P * M * (M - K + 1) > (1ll << 27)) return fail(PD_EINVAL, "too many problems in one call (P*M*(M-K+1) <= 2^27)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PD_ECUDA, "no CUDA device: libpolar_b200 has no CPU path");
    if (device < 0 || device >= ndev) return fail(PD_EINVAL, "device %d out of range", device);
    CUDA_TRY(cudaSetDevice(device));
    return PD_OK;
}
}  // namespace
extern "C" {

int pd_mmi_slice_sums(const double *p1, const double *p2, int32_t P, int32_t M, int32_t K, double *sum1, double *sum2, int32_t device) {
    if (P <= 0) return PD_OK;
    int rc = mmi_check(p1, p2, P, M, K, device);
    if (rc) return rc;
    if (!sum1 || !sum2) return fail(PD_EINVAL, "null argument");
    const int W = M - K + 1;
    const size_t nin = (size_t)P * M, nt = (size_t)P * M * W;
    DevBufs b;
    double *d1 = b.get<double>(nin), *d2 = b.get<double>(nin), *o1 = b.get<double>(nt), *o2 = b.get<double>(nt);
    if (!d1 || !d2 || !o1 || !o2) return fail(PD_ENOMEM, "cudaMalloc failed");
    CUDA_TRY(cudaMemcpy(d1, p1, nin * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d2, p2, nin * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(launch_mmi_table(P, M, W, 0, d1, d2, nullptr, nullptr, 0., 0., o1, o2));
    g_launches++;
    CUDA_TRY(cudaMemcpy(sum1, o1, nt * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(sum2, o2, nt * 8, cudaMemcpyDeviceToHost));
    return PD_OK;
}

int pd_mmi_design(const double *p1, const double *p2, const double *l1, const double *l2, double c1, double c2,
                  int32_t P, int32_t M, int32_t K, int32_t *Az, int32_t device) {
    if (P <= 0) return PD_OK;
    int rc = mmi_check(p1, p2, P, M, K, device);
    if (rc) return rc;
    if (!l1 || !l2 || !Az) return fail(PD_EINVAL, "null argument");
    const int W = M - K + 1;
    const size_t nin = (size_t)P * M, nt = (size_t)P * M * W;
    DevBufs b;
    double *d1 = b.get<double>(nin), *d2 = b.get<double>(nin), *e1 = b.get<double>(nt), *e2 = b.get<double>(nt), *T = b.get<double>(nt);
    int32_t *lm = b.get<int32_t>((size_t)P * (K + 1) * W), *dAz = b.get<int32_t>((size_t)P * (K + 1));
    if (!d1 || !d2 || !e1 || !e2 || !T || !lm || !dAz) return fail(PD_ENOMEM, "cudaMalloc failed");
    CUDA_TRY(cudaMemcpy(d1, p1, nin * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d2, p2, nin * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(e1, l1, nt * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(e2, l2, nt * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(launch_mmi_table(P, M, W, 1, d1, d2, e1, e2, c1, c2, T, nullptr));
    CUDA_TRY(launch_mmi_dp(P, M, K, W, T, lm, dAz));
    g_launches += 2;
    CUDA_TRY(cudaMemcpy(Az, dAz, (size_t)P * (K + 1) * 4, cudaMemcpyDeviceToHost));
    return PD_OK;
}

#endif   // PB_HOST_EMU

void *pd_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { fail(PD_ENOMEM, "cudaHostAlloc(%zu) failed", bytes); return nullptr; }
    return p;
}
void pd_host_free(void *p) { if (p) cudaFreeHost(p); }

}  // extern "C"
