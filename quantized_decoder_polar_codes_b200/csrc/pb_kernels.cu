// Kernel instantiations of libpolar_b200.so, one translation unit per family so that the objects build in parallel
// (build.py compiles this file once per PB_TU value).  The host side (pb_capi.cu) only sees the *_kernel_fn dispatchers.
//   PB_TU 1  scl_lut_warp L=8 plain + CRC-aided      5  path_warp LUT domain       9  generic (CTA per frame), all domains
//         2  scl_lut_warp L=8 Fast-SSC variants      6  path_warp float
//         3  scl_lut_warp L=1,2                      7  path_warp uniform
//         4  scl_lut_warp L=4                        8  path_warp Lloyd
#if PB_TU >= 1 && PB_TU <= 4
#define PB_TU_SCL
#include "pb_scl_lut.cuh"
namespace pb {
#if PB_TU == 1
const void *scl_fn_l3_plain(bool ca) { return fast_kernel_fn_l<3, false>(ca); }
#elif PB_TU == 2
const void *scl_fn_l3_fast(bool ca) { return fast_kernel_fn_l<3, true>(ca); }
#elif PB_TU == 3
const void *scl_fn_l01(int logL, bool ca, bool fast) { if (logL == 0) return fast ? fast_kernel_fn_l<0, true>(false) : fast_kernel_fn_l<0, false>(false);
    return fast ? fast_kernel_fn_l<1, true>(ca) : fast_kernel_fn_l<1, false>(ca); }
#else
const void *scl_fn_l2(bool ca, bool fast) { return fast ? fast_kernel_fn_l<2, true>(ca) : fast_kernel_fn_l<2, false>(ca); }
#endif
}  // namespace pb
#elif PB_TU >= 5 && PB_TU <= 8
#define PB_TU_PATH
#include "pb_generic.cuh"
#include "pb_path_warp.cuh"
namespace pb {
#if PB_TU == 5
const void *path_fn_lut(int logL) { return path_kernel_fn_d<DOM_LUT>(logL); }
#elif PB_TU == 6
const void *path_fn_float(int logL) { return path_kernel_fn_d<DOM_FLOAT>(logL); }
#elif PB_TU == 7
const void *path_fn_uniform(int logL) { return path_kernel_fn_d<DOM_UNIFORM>(logL); }
#else
const void *path_fn_lloyd(int logL) { return path_kernel_fn_d<DOM_LLOYD>(logL); }
#endif
}  // namespace pb
#elif PB_TU == 9
#include "pb_generic.cuh"
namespace pb {
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
#else
#error "PB_TU must be 1..9"
#endif
