// libpolar_b200 built for the host emulator (see shim/cuda_runtime.h): the C ABI + the four decode kernel families as plain
// C++, threads as fibers.  Development tooling only; built into tools/emu/build/, never into the package.
#include <cuda_runtime.h>   // resolves to shim/cuda_runtime.h (-I order)

namespace pb_emu {
State &st() { static State s; return s; }
std::map<const void *, std::function<void(void **)>> &registry() { static std::map<const void *, std::function<void(void **)>> r; return r; }

extern "C" void pb_emu_switch(void **from_sp, void *to_sp);
asm(R"(
.text
.globl pb_emu_switch
.type pb_emu_switch,@function
pb_emu_switch:
    pushq %rbp
    pushq %rbx
    pushq %r12
    pushq %r13
    pushq %r14
    pushq %r15
    movq %rsp, (%rdi)
    movq %rsi, %rsp
    popq %r15
    popq %r14
    popq %r13
    popq %r12
    popq %rbx
    popq %rbp
    ret
)");

static void set_ids(State &s, int t) {
    s.cur = t;
    s.tid.x = (unsigned)t; s.tid.y = s.tid.z = 0;
}
// switch from the running fiber (or the scheduler when from < 0) to the next live fiber after it
static void run_next(int from) {
    State &s = st();
    int t = from;
    for (int k = 0; k < s.nthreads; ++k) {
        t = (t + 1) % s.nthreads;
        if (!s.done[t]) {
            void **save = from < 0 ? &s.main_sp : &s.sp[from];
            if (t == from) return;
            set_ids(s, t);
            pb_emu_switch(save, s.sp[t]);
            if (from >= 0) set_ids(st(), from);
            return;
        }
    }
    if (from >= 0) {   // last fiber finished: back to the scheduler
        void *dummy;
        pb_emu_switch(&dummy, s.main_sp);
    }
}
void yield() { run_next(st().cur); }

static void fiber_entry() {
    State &s = st();
    s.body();
    State &s2 = st();
    s2.done[s2.cur] = 1;
    s2.live--;
    run_next(s2.cur);
    abort();   // unreachable
}

void launch(const std::function<void()> &body, dim3 grid, dim3 block, size_t smem) {
    State &s = st();
    const int nt = (int)block.x;
    constexpr size_t kStack = 512 << 10;
    static std::vector<char *> stacks;
    while ((int)stacks.size() < nt) stacks.push_back((char *)aligned_alloc(64, kStack));
    static char *smem_buf = nullptr;
    static size_t smem_cap = 0;
    if (smem + 64 > smem_cap) { free(smem_buf); smem_cap = smem + 4096; smem_buf = (char *)aligned_alloc(128, (smem_cap + 127) & ~(size_t)127); }
    s.gdim.x = grid.x; s.gdim.y = s.gdim.z = 1;
    s.bdim.x = block.x; s.bdim.y = s.bdim.z = 1;
    s.body = body;
    for (unsigned b = 0; b < grid.x; ++b) {
        s.bid.x = b; s.bid.y = s.bid.z = 0;
        s.nthreads = nt;
        s.sp.assign(nt, nullptr);
        s.done.assign(nt, 0);
        s.warps.assign((nt + 31) / 32, WarpState());
        s.ncoll.assign(nt, 0u);
        s.blk_arrived = 0; s.blk_gen = 0;
        s.smem = smem_buf;
        memset(smem_buf, 0xcd, smem);   // poison: shared memory is not zero-initialised on the device either
        s.live = nt;
        for (int t = 0; t < nt; ++t) {
            uintptr_t top = ((uintptr_t)stacks[t] + kStack) & ~(uintptr_t)15;
            void **sp = (void **)(top - 8 * 8);
            for (int i = 0; i < 6; ++i) sp[i] = nullptr;
            sp[6] = (void *)&fiber_entry;
            sp[7] = nullptr;
            s.sp[t] = sp;
        }
        run_next(-1);
        if (s.live != 0) { fprintf(stderr, "pb_emu: deadlock (%d threads never finished)\n", s.live); abort(); }
    }
}
}  // namespace pb_emu

#define PB_TU_SCL
#define PB_TU_PATH
#define PB_TU_PATH_CTA
#include "pb_capi.cu"

namespace pb {
const void *scl_fn_l3_plain(bool ca) { return fast_kernel_fn_l<3, false>(ca); }
const void *scl_fn_l3_fast(bool ca) { return fast_kernel_fn_l<3, true>(ca); }
const void *scl_fn_l01(int logL, bool ca, bool fast) {
    if (logL == 0) return fast ? fast_kernel_fn_l<0, true>(false) : fast_kernel_fn_l<0, false>(false);
    return fast ? fast_kernel_fn_l<1, true>(ca) : fast_kernel_fn_l<1, false>(ca);
}
const void *scl_fn_l2(bool ca, bool fast) { return fast ? fast_kernel_fn_l<2, true>(ca) : fast_kernel_fn_l<2, false>(ca); }
const void *path_fn_lut(int logL) { return path_kernel_fn_d<DOM_LUT>(logL); }
const void *path_fn_float(int logL) { return path_kernel_fn_d<DOM_FLOAT>(logL); }
const void *path_fn_uniform(int logL) { return path_kernel_fn_d<DOM_UNIFORM>(logL); }
const void *path_fn_lloyd(int logL) { return path_kernel_fn_d<DOM_LLOYD>(logL); }
const void *path_cta_kernel_fn(int dom, int logL) { return path_cta_kernel_fn_all(dom, logL); }
template <int DOM, bool LIST>
static const void *generic_fn(bool warp) {
    return warp ? PB_KFN(generic_decode_kernel<DOM, LIST, true>) : PB_KFN(generic_decode_kernel<DOM, LIST, false>);
}
const void *generic_kernel_fn(int dom, bool l, bool w) {
    switch (dom) {
    case DOM_LUT: return l ? generic_fn<DOM_LUT, true>(w) : generic_fn<DOM_LUT, false>(w);
    case DOM_FLOAT: return l ? generic_fn<DOM_FLOAT, true>(w) : generic_fn<DOM_FLOAT, false>(w);
    case DOM_UNIFORM: return l ? generic_fn<DOM_UNIFORM, true>(w) : generic_fn<DOM_UNIFORM, false>(w);
    default: return l ? generic_fn<DOM_LLOYD, true>(w) : generic_fn<DOM_LLOYD, false>(w);
    }
}
}  // namespace pb

// The compiled scl_lut_warp walk of a decoder (the `_handle` of a pybind decoder): hist[type * 32 + depth] = number of
// ops of that type at that depth (types < 16), plus n_ops and n_chunks.  Returns -1 when the decoder is not on scl_lut_warp.
extern "C" int pb_emu_fast_plan(const pd_decoder *dec, int *hist, int *n_ops, int *n_chunks) {
    if (!dec->fast.ok) return -1;
    memset(hist, 0, 16 * 32 * sizeof(int));
    for (const uint2 &o : dec->fast.ops) hist[(o.x & 15u) * 32 + ((o.x >> 8) & 31u)]++;
    *n_ops = dec->fast.p.n_ops;
    *n_chunks = dec->fast.p.n_chunks;
    return 0;
}

// The plan of a decoder on scl_lut_warp in full: its op entries (x, y pairs) into ops[2 * ops_cap], the value-level
// layout (voff[kMaxLog + 2] and gl), and the uploaded stream, head copies included, into stream[stream_cap] with its
// length in words in *stream_words.  Returns the number of ops, or -1 when the decoder is not on scl_lut_warp.
extern "C" int pb_emu_fast_plan_detail(const pd_decoder *dec, uint32_t *ops, int ops_cap, int *voff, int *gl,
                                       uint32_t *stream, long long stream_cap, long long *stream_words) {
    if (!dec->fast.ok) return -1;
    const std::vector<uint2> &o = dec->fast.ops;
    for (int i = 0; i < (int)o.size() && i < ops_cap; ++i) { ops[2 * i] = o[i].x; ops[2 * i + 1] = o[i].y; }
    for (int d = 0; d < pb::kMaxLog + 2; ++d) voff[d] = dec->fast.p.voff[d];
    *gl = dec->fast.p.gl;
    const long long words = ((long long)dec->fast.p.n_chunks + pb::kRingChunks - 1) * 128;
    *stream_words = words;
    memcpy(stream, dec->fast.p.stream, (size_t)std::min(words, stream_cap) * 4);
    return (int)o.size();
}

// The fork counters of scl_lut_warp, once per warp: forks seen and identity exits taken since the last reset.
extern "C" void pb_emu_fork_counts(unsigned long long *seen, unsigned long long *taken, int reset) {
    *seen = pb::emu_fork::seen();
    *taken = pb::emu_fork::taken();
    if (reset) pb::emu_fork::seen() = pb::emu_fork::taken() = 0;
}

// entry points of the real library that the emulator does not provide (the pybind module links them)
extern "C" {
int pd_count_errors(const uint8_t *, const uint8_t *, int64_t, int32_t, unsigned long long *, void *) { return PD_ECUDA; }
int pd_sim_create(const pd_sim_config *, pd_sim **) { return PD_ECUDA; }
void pd_sim_destroy(pd_sim *) {}
int pd_sim_generate(pd_sim *, double, int64_t, uint64_t, uint64_t, uint8_t *, void *, void *) { return PD_ECUDA; }
int pd_sim_set_channel(pd_sim *, const pd_sim_channel *) { return PD_ECUDA; }
int pd_sim_encode(pd_sim *, int, const uint8_t *, int64_t, uint8_t *) { return PD_ECUDA; }
int pd_sim_encode_device(pd_sim *, int, const uint8_t *, int64_t, uint8_t *, void *) { return PD_ECUDA; }
int pd_mmi_slice_sums(const double *, const double *, int32_t, int32_t, int32_t, double *, double *, int32_t) { return PD_ECUDA; }
int pd_mmi_design(const double *, const double *, const double *, const double *, double, double, int32_t, int32_t, int32_t, int32_t *, int32_t) { return PD_ECUDA; }
int pd_optls_quantize(const double *, const double *, const int32_t *, int64_t, int32_t, int32_t, double *, double *, int32_t *, int32_t) { return PD_ECUDA; }
}
