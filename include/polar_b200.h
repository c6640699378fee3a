/*
 * polar_b200.h -- C ABI of libpolar_b200.so: the B200 (sm_100a) batched polar decoders.
 *
 * This is the drop-in boundary for the decode() hot path of the reference's `PolarDecoder` pybind11
 * module.  The reference has no C ABI of its own (SURVEY.md 8b): its boundary is the pybind11 classes
 * registered in PolarDecoder/PolarDecoder/_cpp/_libPolarDecoder.cpp:29-50.  Each entry point below states
 * which reference interface it replaces ("PD/" = PolarDecoder/PolarDecoder/_cpp/).  The pybind11 module
 * shipped in this repo (quantized_decoder_polar_codes_b200/csrc/pb_pybind.cpp) re-creates those 15 classes
 * on top of this header; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Plain pointers and sizes only; no torch / pybind types.  All functions return a pd_status; the text of
 * the last error on the calling thread is available from pd_last_error().
 */
#ifndef POLAR_B200_H
#define POLAR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* One value per reference class; replaces the 15 py::class_ registrations (PD/py_interface/py_*.cpp). */
typedef enum pd_kind {
    PD_SC = 0,             /* SCDecoder                  PD/src/SCDecoder.cpp:14-89 */
    PD_FASTSC = 1,         /* FastSCDecoder              PD/src/FastSCDecoder.cpp:21-173 */
    PD_SCL = 2,            /* SCLDecoder                 PD/src/SCLDecoder.cpp:38-175 */
    PD_FASTSCL = 3,        /* FastSCLDecoder             PD/src/FastSCLDecoder.cpp:49-423 */
    PD_CASCL = 4,          /* CASCLDecoder               PD/src/CASCLDecoder.cpp:74-249 */
    PD_SCLUT = 5,          /* SCLUTDecoder               PD/src/SCLUTDecoder.cpp:21-124 */
    PD_FASTSCLUT = 6,      /* FastSCLUTDecoder           PD/src/FastSCLUT.cpp:27-206 */
    PD_SCLLUT = 7,         /* SCLLUTDecoder              PD/src/SCLLUTDecoder.cpp:47-253 */
    PD_FASTSCLLUT = 8,     /* FastSCLLUTDecoder          PD/src/FastSCLLUTDecoder.cpp:57-408 */
    PD_CASCLLUT = 9,       /* CASCLLUTDecoder            PD/src/CASCLLUTDecoder.cpp:65-303 */
    PD_CAFASTSCLLUT = 10,  /* CAFastSCLLUTDecoder        PD/src/CAFastSCLLUTDecoder.cpp:60-454 */
    PD_SC_UNIFORM = 11,    /* SCUniformQuantizedDecoder  PD/src/SCUniformQuantizedDecoder.cpp:20-99 */
    PD_SCL_UNIFORM = 12,   /* SCLUniformQuantizedDecoder PD/src/SCLUniformQuantizedDecoder.cpp:43-184 */
    PD_SC_LLOYD = 13,      /* SCLloydQuantizedDecoder    PD/src/SCLloydQuantizedDecoder.cpp:22-101 */
    PD_SCL_LLOYD = 14,     /* SCLLloydQuantizedDecoder   PD/src/SCLLloydQuantizedDecoder.cpp:46-187 */
    /* blind-detection helpers of the reference's PolarEncoder/PolarBD package (SURVEY 8f row f4) */
    PD_BD_DMETRIC = 15,    /* DMetricCalculator          PolarEncoder/PolarBD/_cpp/src/DMetric.cpp:25-176 (Fast-SSC walk + metric) */
    PD_BD_CASCL = 16,      /* PolarBD CASCLDecoder       PolarEncoder/PolarBD/_cpp/src/CASCLWithRNTI.cpp:74-252 (RNTI-scrambled CRC) */
    PD_KIND_COUNT = 17
} pd_kind;

typedef enum pd_dtype {
    PD_U8 = 0,   /* channel symbols, one byte each (LUT family; the compact streaming format)       */
    PD_I32 = 1,  /* channel symbols as the reference's py::array_t<int> (LUT family)                */
    PD_F64 = 2   /* channel LLRs as the reference's py::array_t<double> (float/uniform/Lloyd family); pd_decode (host buffers)
                    also takes float64-TYPED SYMBOLS for the LUT family -- the probability-domain driver keeps them so,
                    mainQuantizedDecoder_ProbabilityDomain.py:174-179 -- and truncates them to bytes like the reference's cast */
} pd_dtype;

typedef enum pd_status {
    PD_OK = 0,
    PD_EINVAL = 1,   /* bad argument / inconsistent tables (the reference: undefined behaviour)  */
    PD_ECUDA = 2,    /* CUDA runtime error or no usable sm_100 device                           */
    PD_ERANGE = 3,   /* an input symbol is outside the root table (the reference: out-of-bounds read) */
    PD_ENOMEM = 4
} pd_status;

/*
 * Constructor arguments, i.e. what the reference's py::init<...> signatures carry
 * (PD/py_interface/py_*.cpp; SURVEY.md 8b), with the nested Python lists flattened:
 *
 *   LUT_f[node][pos][a][b]      -> lut_pool[f_off[node] + (pos*f_qa[node] + a)*f_qb[node] + b]
 *   LUT_g[node][pos][u][a][b]   -> lut_pool[g_off[node] + ((pos*2+u)*g_qa[node] + a)*g_qb[node] + b]
 *        node = heap id (1<<depth)+index-1 in [0,N-1); f_npos/g_npos[node] = number of per-position tables
 *        stored for the node: 1 (one table shared by all positions -- what every generator of the reference
 *        emits, SURVEY App. A.4) or N>>(depth+1).
 *   virtual_channel_llr[level][pos][sym] -> llr_pool[llr_off[level*N+pos] + sym]; llr_off has
 *        llr_levels*N+1 entries so row lengths are known.
 * Unused members are NULL / 0.  All arrays are copied; the caller may free them after pd_create returns.
 */
typedef struct pd_config {
    int32_t kind;                 /* pd_kind */
    int32_t N, K, A, L;           /* A: CA kinds only; L: list kinds only, 1..32, or 64, 128, 256 with N >= 32 (those three
                                     run on "path_cta"; PD_BD_CASCL takes 1..32 only).  Other values: PD_EINVAL */
    int32_t device;               /* CUDA device ordinal */
    const int32_t *frozen_bits;   /* [N], 1 = frozen (indicator mask, mainFPDecoder.py:49,58) */
    const int32_t *node_type;     /* [2N-1] Fast kinds: -1 ordinary, 0 R0, 1 R1, 2 REP, 3 SPC (IdentifyNodes.py) */
    int32_t crc_n;                /* CASCL only: generator degree and its set exponent positions    */
    const int32_t *crc_loc;       /*   (crc_p of PD/py_interface/py_CASCLDecoder.cpp:9-11)           */
    int32_t crc_loc_len;
    const int32_t *lut_pool;
    int64_t lut_pool_len;
    const int64_t *f_off, *g_off;                 /* [N-1] */
    const int32_t *f_npos, *g_npos;               /* [N-1] */
    const int32_t *f_qa, *f_qb, *g_qa, *g_qb;     /* [N-1] */
    const double *llr_pool;
    const int64_t *llr_off;                       /* [llr_levels*N + 1] */
    int32_t llr_levels;
    const double *decoder_r_f, *decoder_r_g;      /* [N-1] uniform kinds */
    int32_t v;                                    /* uniform + Lloyd kinds */
    const double *boundaries_f, *boundaries_g;    /* [N-1][n_boundaries] Lloyd kinds */
    const double *reconstruction_f, *reconstruction_g; /* [N-1][n_reconstruction] */
    int32_t n_boundaries, n_reconstruction;
} pd_config;

typedef struct pd_decoder pd_decoder; /* opaque; owns device copies of all tables + the compiled schedule */

/* Replaces `T(N, K, ...)` of each reference class: validates, packs the tables, compiles the tree walk
 * into a device schedule, uploads everything to `cfg->device`. */
int pd_create(const pd_config *cfg, pd_decoder **out);
void pd_destroy(pd_decoder *dec);

/* Number of bytes written per frame: K, or A for the CRC-aided kinds (PD/src/SCLLUTDecoder.cpp:245,
 * CASCLLUTDecoder.cpp:290). */
int pd_out_len(const pd_decoder *dec);
int pd_code_len(const pd_decoder *dec);
/* Frames that one full wave of the (persistent) decode kernel holds in flight on the decoder's GPU: SMs x resident warps x
 * frames per warp (path_cta, L >= 64: SMs x resident CTAs, one frame per CTA); 0 for the CTA-per-frame generic kernel.  The scl_lut_warp kernels hand frame groups to their warps from a
 * counter, so any batch size runs without a tail in one launch; the statically scheduled kernels (fp64 family, Fast-SSC
 * variants) get large batches as overlapping one-wave launches, and there a multiple of this number has no tail. */
int64_t pd_wave_frames(const pd_decoder *dec, int in_dtype);

/* Replaces `T::decode(array)` (e.g. SCLLUT::decode, PD/src/SCLLUTDecoder.cpp:47) for a batch of B frames.
 * host_in: [B][N] of `in_dtype`, C-contiguous; host_out: [B][pd_out_len] uint8.  Blocking: pipelines
 * host->device copies, the decode kernel and device->host copies in chunks, then synchronizes.
 * Decoding is stateless across calls like the reference's; a decoder object must not be used from two
 * threads at once. */
int pd_decode(pd_decoder *dec, const void *host_in, int in_dtype, int64_t B, uint8_t *host_out);

/* In-library multi-GPU (SURVEY 8b/8e): after pd_set_devices(dec, n, ids) every pd_decode call deals its batch, chunk by chunk,
 * to the n CUDA devices `ids` of the box -- the tables and the compiled schedule are cloned onto each of them, frames are
 * independent, so there is no data-path exchange at all.  n = 0 goes back to the decoder's own device.  An id may repeat
 * (two pipelines on one GPU).  pd_decode_device / pd_check / pd_wave_frames keep referring to the decoder's own device.
 * pd_counters_allreduce sums the per-device {bit errors, block errors} pairs of pd_count_errors over the decoder's devices and
 * writes the total back to each (dev_counters[i] lives on device i of the list). */
int pd_set_devices(pd_decoder *dec, int32_t n, const int32_t *device_ids);
int32_t pd_device_count(const pd_decoder *dec);
int pd_counters_allreduce(pd_decoder *dec, unsigned long long *const *dev_counters, int32_t n);

/* Same with device-resident buffers; asynchronous on `cuda_stream` (a cudaStream_t, NULL = default stream).
 * Input symbol range errors are reported by the next pd_check(). */
int pd_decode_device(pd_decoder *dec, const void *dev_in, int in_dtype, int64_t B, uint8_t *dev_out,
                     void *cuda_stream);
/* Synchronizes `cuda_stream` and returns PD_ERANGE if any frame decoded since the last check carried an
 * out-of-range symbol, PD_ECUDA on a CUDA error. */
int pd_check(pd_decoder *dec, void *cuda_stream);

/* Optional debug taps (tests of the float family compare path metrics with the oracle): after this call
 * every pd_decode_device also writes the final path metrics [B][L] (slot order) and the winning slot [B].
 * Pass NULLs to switch off. */
int pd_set_debug_outputs(pd_decoder *dec, double *dev_pm, int32_t *dev_winner);

/* Simulation-mode counters (the BER/BLER bookkeeping of the drivers' frame loop,
 * mainQuantizedDecoder_LLRDomain.py:181-192): adds #bit errors and #block errors of dev_decoded vs
 * dev_truth ([B][len] each) to dev_counters[0], dev_counters[1] (device uint64).  These two words are what
 * the multi-GPU front-end all-reduces over NCCL. */
int pd_count_errors(const uint8_t *dev_decoded, const uint8_t *dev_truth, int64_t B, int32_t len,
                    unsigned long long *dev_counters, void *cuda_stream);

/* ---------------------------------------------------------------------------------------------------
 * On-device simulation front-end ("next" row f1 of SURVEY.md 8f): the frame generator of the drivers' loop body
 * (mainQuantizedDecoder_LLRDomain.py:151-176): random message -> [CRC] -> polar encode (natural order) ->
 * BPSK + AWGN(sigma) -> llr = 2y/sigma^2 -> channel quantizer (edges + lut, the driver's bisect rule), all on
 * the GPU (Philox counter RNG: frame i of a run always sees the same noise whatever the batch split / GPU).
 * pd_sim_set_channel switches to the front ends of the probability-domain and continuous-domain drivers.
 * Decode with pd_decode_device and count with pd_count_errors afterwards. */
typedef struct pd_sim pd_sim;
typedef struct pd_sim_config {
    int32_t N, K, A;              /* K - A CRC bits are appended when crc_n > 0 (then K == A + crc_n) */
    int32_t device;
    const int32_t *frozen_bits;   /* [N] */
    int32_t crc_n;                /* 0 = no CRC */
    const int32_t *crc_loc;       /* generator exponents as in the drivers' crc_p */
    int32_t crc_loc_len;
    const double *edges;          /* channel quantizer: interval_x, n_edges = M+1 ascending edges; NULL -> emit fp64 LLRs */
    int32_t n_edges;
    const uint8_t *chan_lut;      /* [M] compressed symbol of uniform cell i */
    int32_t q_channel;            /* QChannelCompressed (saturation symbol = q_channel-1) */
} pd_sim_config;
int pd_sim_create(const pd_sim_config *cfg, pd_sim **out);
void pd_sim_destroy(pd_sim *sim);
/* Generates frames [first_frame, first_frame+B) of the run `seed`: dev_msg [B][A] uint8 message bits and
 * dev_out [B][N] in the type of the current channel mode (see pd_sim_set_channel): uint8 symbols for PD_SIM_LLR_QUANT
 * and PD_SIM_Y_QUANT, fp64 for PD_SIM_LLR and PD_SIM_LLR_UNIFORM.  Frame i of a run has the same message and the same
 * channel output y in every mode.  Asynchronous on cuda_stream. */
int pd_sim_generate(pd_sim *sim, double sigma, int64_t B, uint64_t seed, uint64_t first_frame,
                    uint8_t *dev_msg, void *dev_out, void *cuda_stream);

/* Channel front end of a pd_sim: what pd_sim_generate stores for each code bit, from y = 1-2x + sigma*n and
 * llr = 2y/sigma^2.  One mode per reference driver. */
#define PD_SIM_LLR 0          /* fp64 LLRs                                   (what pd_sim_create sets without edges) */
#define PD_SIM_LLR_QUANT 1    /* LLR-domain driver: edges + chan_lut -> uint8 (what pd_sim_create sets with edges)    */
#define PD_SIM_Y_QUANT 2      /* probability-domain driver: y cut at edges[q_channel+1] -> uint8                      */
#define PD_SIM_LLR_UNIFORM 3  /* continuous-domain driver: QUniform(llr, v, r) -> fp64                               */
typedef struct pd_sim_channel {
    int32_t mode;
    const double *edges; int32_t n_edges;   /* LLR_QUANT, Y_QUANT */
    const uint8_t *chan_lut;                /* LLR_QUANT: [n_edges-1] */
    int32_t q_channel;                      /* LLR_QUANT, Y_QUANT */
    double r; int32_t v;                    /* LLR_UNIFORM: step and level count */
} pd_sim_channel;
/* Replaces the channel front end of `sim`; the code, CRC and device stay.  A sweep over Eb/N0 calls this once per point,
 * as the drivers design a new channel quantizer at every point.
 *   PD_SIM_LLR          nothing else is read.
 *   PD_SIM_LLR_QUANT    symbol = 0 if llr <= edges[0], q_channel-1 if llr >= edges[n_edges-1],
 *                       else chan_lut[bisect_left(edges[0..n_edges-2], llr) - 1]  (mainQuantizedDecoder_LLRDomain.py:167-176).
 *                       n_edges >= 2, chan_lut entries < q_channel.
 *   PD_SIM_Y_QUANT      symbol = 0 if y <= edges[0], q_channel-1 if y >= edges[q_channel],
 *                       else bisect_left(edges, y) - 1  (mainQuantizedDecoder_ProbabilityDomain.py:153-177: the MMI channel
 *                       quantizer's edges interval_x[channel_lut]).  n_edges == q_channel + 1.
 *   PD_SIM_LLR_UNIFORM  QUniform (mainQuantizedDecoder_ContinuousDomain.py:29-32): with bound = (v/2 - 0.5) r,
 *                       out = sign(llr) (bound - r/2) if |llr| > bound, else (floor(llr/r) + 0.5) r.  r > 0 finite, v >= 2.
 * q_channel is in [1,256]; edges are ascending and not NaN.  Violations return PD_EINVAL and leave the sim unchanged.
 * The tables are copied into new device buffers that live until pd_sim_destroy: a pd_sim_generate already enqueued on
 * some stream keeps reading the tables it was launched with, so this call needs no synchronisation. */
int pd_sim_set_channel(pd_sim *sim, const pd_sim_channel *ch);

/* Blind-detection entry (kinds PD_BD_DMETRIC / PD_BD_CASCL; fp64 LLR input [B][N]).
 *   PD_BD_DMETRIC: out_metric[b] = DMetricCalculator.calculate(llr_b) (DMetric.cpp:25-176); out_bits / out_pass unused (may be NULL).
 *   PD_BD_CASCL:   CASCL::decode(llr_b, RNTI) (CASCLWithRNTI.cpp:74-252) -> out_bits [B][A], out_metric[b] = the PM it returns
 *                  (PML[0], or PML[i] of the i-th candidate in sorted order that passed -- the reference indexes the
 *                  unsorted array there, reproduced), out_pass[b] = isPass.  rnti: rnti_len 0/1 ints XORed onto the LAST
 *                  rnti_len CRC bits, shared by all frames of the call (rnti_len <= crc_n; may be 0).
 * pd_decode_bd takes host buffers; pd_decode_bd_device device buffers (rnti on the device too), asynchronous on cuda_stream.
 * pd_decode / pd_decode_device also accept these kinds (plain Fast-SC bits / CA-SCL bits without RNTI). */
int pd_decode_bd(pd_decoder *dec, const double *llr, int64_t B, const int32_t *rnti, int32_t rnti_len,
                 uint8_t *out_bits, double *out_metric, uint8_t *out_pass);
int pd_decode_bd_device(pd_decoder *dec, const double *dev_llr, int64_t B, const int32_t *dev_rnti, int32_t rnti_len,
                        uint8_t *dev_bits, double *dev_metric, uint8_t *dev_pass, void *cuda_stream);

/* Batched encoder side of the same object (SURVEY 8f row f2): what the drivers call on the PolarBDEnc package, which is
 * imported by all four drivers (mainFPDecoder.py:12-13,56-57,102-105) but absent from the reference tree.  Bits are one
 * byte each (0/1), as in the drivers' numpy arrays.
 *   PD_ENC_POLAR      in [B][K] -> out [B][N]   PolarEnc(N,K,frozenbits,msgbits).encode: u[msgbits] = in, x = u F^(x)n
 *                                               (natural order, the butterfly of PD/src/FastSCDecoder.cpp:153-164)
 *   PD_ENC_CRC        in [B][A] -> out [B][K]   CRCEnc(crc_n,crc_p).encode: in || CRC::encoding(in) (PD/src/utils.cpp:77-93)
 *   PD_ENC_CRC_POLAR  in [B][A] -> out [B][N]   both in one pass
 * pd_sim_encode takes host buffers (copies inside), pd_sim_encode_device device buffers, asynchronous on cuda_stream. */
#define PD_ENC_POLAR 0
#define PD_ENC_CRC 1
#define PD_ENC_CRC_POLAR 2
int pd_sim_encode(pd_sim *sim, int mode, const uint8_t *in, int64_t B, uint8_t *out);
int pd_sim_encode_device(pd_sim *sim, int mode, const uint8_t *dev_in, int64_t B, uint8_t *dev_out, void *cuda_stream);

/* Lookup-table design (SURVEY 8f row f3): the minimum-distortion quantizer the reference's LLR-domain generator runs on every
 * tree node -- LLRQuantizer.find_OptLS_quantizer(density, quanta, M, K) (QLLRDensityEvolution_MinDistortion.py:107-108;
 * C++ on OpenCV in Quantizers/.../LLRQuantizer.cpp:67-164, numpy restatement MinDistortionQuantizer.py:28-99, which this
 * follows bit for bit) -- for P independent problems at once, one CTA each.  Problem p: M[p] symbols (K < M[p] <= 1024) with
 * probabilities density[p*stride + i] and values quanta[p*stride + i], STRICTLY ASCENDING in i (np.unique output, as the
 * generator passes them).  Out: density / quanta of the K merged symbols [P][K], lut[p*stride + i] = merged symbol of i.
 * Host buffers; runs on `device`. */
int pd_optls_quantize(const double *density, const double *quanta, const int32_t *M, int64_t stride, int32_t P, int32_t K,
                      double *out_density, double *out_quanta, int32_t *out_lut, int32_t device);

/* Probability-domain table design (the other half of SURVEY 8f row f3): the device passes of the maximum-mutual-information
 * quantizer MMIQuantizer.find_opt_quantizer that QDensityEvolution_MMI.py:84,107 runs on every tree node (C++ on OpenCV in
 * Quantizers/quantizers/_cpp/MMIQuantizer/MMIQuantizer.cpp:73-165; numpy restatement QuantizeDensityEvolution/MMIQuantizer.py:
 * 36-84,158-225, which this follows bit for bit).  P problems of M symbols each, sorted by likelihood ratio, conditional
 * probabilities p1[p][i] = P(y_i|x=+1), p2[p][i] = P(y_i|x=-1); K output symbols; W = M-K+1.  Tables are banded: entry
 * [p][a'][w] describes merging the sorted symbols a' .. a'+w into one.
 *   pd_mmi_slice_sums: sum1/sum2[p][a'][w] = np.sum(p1/p2[a' : a'+w+1]) in numpy's pairwise order (MMIQuantizer.py:42-43).
 *   pd_mmi_design:     cost[p][a'][w] = c1*np.sum(p1[..]*l1[p][a'][w]) + c2*np.sum(p2[..]*l2[p][a'][w]) (:55-67; l = log2 of the
 *                      cluster likelihoods, taken by the caller with numpy so that they are numpy's), then the dynamic
 *                      programme and back-trace (:175-215); Az[p][0..K] = cluster boundaries.
 * Host buffers; runs on `device`. */
int pd_mmi_slice_sums(const double *p1, const double *p2, int32_t P, int32_t M, int32_t K, double *sum1, double *sum2, int32_t device);
int pd_mmi_design(const double *p1, const double *p2, const double *l1, const double *l2, double c1, double c2,
                  int32_t P, int32_t M, int32_t K, int32_t *Az, int32_t device);

/* Kernels launched by this library on the calling process so far (bench.py reports it as gpu_launches). */
int64_t pd_launch_count(void);
/* Name of the kernel variant pd_decode* uses for this decoder ("scl_lut_warp", "path_warp", "generic", or "path_cta" for
   every list decoder with L > 32). */
const char *pd_kernel_name(const pd_decoder *dec);
/* Why a LUT-class decoder is NOT on "scl_lut_warp" ("" when it is, or for the float / uniform / Lloyd classes): the shape
   rule that sent it to the slower path_warp / generic kernels.  The same text is printed once on stderr at pd_create
   (POLAR_B200_QUIET=1 silences it). */
const char *pd_kernel_note(const pd_decoder *dec);
/* Static description of the schedule for reports: n_steps, algorithmic lookups per frame, ... */
int pd_schedule_stats(const pd_decoder *dec, int64_t *n_steps, int64_t *elem_ops, int64_t *n_sorts);

/* Pinned host memory for the caller's I/O buffers (pd_decode is PCIe-bound from pageable memory). */
void *pd_host_alloc(size_t bytes);
void pd_host_free(void *p);

const char *pd_last_error(void);
const char *pd_version(void);

#ifdef __cplusplus
}
#endif
#endif /* POLAR_B200_H */
