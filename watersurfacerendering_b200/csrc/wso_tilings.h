// wso_tilings.h — the CTA tilings the launch dispatch (wso_kernels.cu) ships, one list for the library and the CPU
// emulator of its kernel bodies (tests/emu/emu.cpp), so that the emulator runs exactly what launch_all() can pick.
// Include after wso_kernels.cuh.
#pragma once

namespace wso {

// CTA tiling.  CP: column pairs per K1 CTA, NF: packed fields per K1 CTA, RI: row items (each = output rows m'
// and N-m') per K2 CTA, RH: row items per K2h CTA (one line each).  CTA threads = lines * N / 16.
template <int CP_, int NF_, int RI_, int RH_>
struct Tiling {
    static constexpr int CP = CP_, NF = NF_, RI = RI_, RH = RH_;
};
// Two tilings per tile size:
//   Bulk - batched launches (many tile-frames per launch): larger CTAs, 32-byte W store segments; tuned with
//          tools/sweep_build.py + tools/sweep_run.sh on B200 (profiles/r1b_sweep.md)
//   Lat  - a launch with few tile-frames (the reference's one ComputeWaves(t) per frame): small CTAs so that a single
//          512^2 or 1024^2 tile still spreads over all 148 SMs
template <int LOGN> struct Cfg;
template <> struct Cfg<4>  { using Bulk = Tiling<8, 4, 8, 8>;   using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<5>  { using Bulk = Tiling<8, 4, 8, 16>;  using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<6>  { using Bulk = Tiling<8, 4, 8, 16>;  using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<7>  { using Bulk = Tiling<4, 4, 8, 16>;  using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<8>  { using Bulk = Tiling<4, 4, 4, 8>;   using Lat = Tiling<2, 2, 1, 2>; };
// (the WSO_TUNE_* macros exist for tuning sweeps: tools/tune_build.sh builds variant libraries)
#ifndef WSO_TUNE_CP9
#define WSO_TUNE_CP9 4
#define WSO_TUNE_NF9 4
#define WSO_TUNE_RI9 1
#define WSO_TUNE_RH9 4
#endif
#ifndef WSO_TUNE_CP10
#define WSO_TUNE_CP10 4
#define WSO_TUNE_NF10 2
#define WSO_TUNE_RI10 2
#define WSO_TUNE_RH10 4
#endif
#ifndef WSO_TUNE_CP11
#define WSO_TUNE_CP11 4
#define WSO_TUNE_NF11 2
#define WSO_TUNE_RI11 1
#define WSO_TUNE_RH11 2
#endif
#ifndef WSO_TUNE_LCP9
#define WSO_TUNE_LCP9 2
#define WSO_TUNE_LNF9 2
#define WSO_TUNE_LRI9 1
#define WSO_TUNE_LRH9 2
#endif
#ifndef WSO_TUNE_LCP10
#define WSO_TUNE_LCP10 2
#define WSO_TUNE_LNF10 2
#define WSO_TUNE_LRI10 1
#define WSO_TUNE_LRH10 2
#endif
template <> struct Cfg<9> {
    using Bulk = Tiling<WSO_TUNE_CP9, WSO_TUNE_NF9, WSO_TUNE_RI9, WSO_TUNE_RH9>;
    using Lat = Tiling<WSO_TUNE_LCP9, WSO_TUNE_LNF9, WSO_TUNE_LRI9, WSO_TUNE_LRH9>;
};
template <> struct Cfg<10> {
    using Bulk = Tiling<WSO_TUNE_CP10, WSO_TUNE_NF10, WSO_TUNE_RI10, WSO_TUNE_RH10>;
    using Lat = Tiling<WSO_TUNE_LCP10, WSO_TUNE_LNF10, WSO_TUNE_LRI10, WSO_TUNE_LRH10>;
};
template <> struct Cfg<11> {
    using Bulk = Tiling<WSO_TUNE_CP11, WSO_TUNE_NF11, WSO_TUNE_RI11, WSO_TUNE_RH11>;
    using Lat = Bulk;
};
template <> struct Cfg<12> { using Bulk = Tiling<4, 1, 2, 4>; using Lat = Bulk; };
template <> struct Cfg<13> { using Bulk = Tiling<2, 1, 1, 2>; using Lat = Bulk; };

// Which kernels of a tiling have a persistent form (Pass1::run_persistent / Pass2::run_persistent): batched launches of
// the fused K1 tilings and of the paired-W K2, 512^2 ... 2048^2.
template <int LOGN, class TL>
struct PersistOk {
    static constexpr bool k1 = Pass1<LOGN, TL::CP, TL::NF, false, true>::kPersistOk && LOGN >= 9 && LOGN <= 11;
    static constexpr bool k2 = WLayout<LOGN>::paired && LOGN >= 9 && LOGN <= 11;
};

}  // namespace wso
