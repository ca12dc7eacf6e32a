// Host-side launchers of the pass kernels for one (line length, precision).
#pragma once
#include "col_groups.cuh"
#include "col_warp.cuh"
#include "passes.cuh"

namespace slm {

template <typename R, int L, bool OK = ColGroupGeom<R, L>::OK> struct GroupLaunch {
    static void prepare() {}
    static int launch(int, const ColGroupArgs&, const TileMap&, const TileMap&, int, cudaStream_t) { return -1; }
};
// Which persistent column kernel serves (R, L): the warp-per-column kernel where it is built (col_warp.cuh),
// else the column-group kernel.  SLM_COL_KERNEL=group selects the latter at run time (A/B measurements).
template <typename R, int L, bool WARP = ColWarpGeom<R, L>::OK> struct ColWarpLaunch {
    static void prepare() {}
    static bool launch(int, const ColGroupArgs&, const TileMap&, const TileMap&, int, cudaStream_t) { return false; }
    static bool enabled() { return false; }
};
template <typename R, int L> struct ColWarpLaunch<R, L, true> {
    using WG = ColWarpGeom<R, L>;
    template <int MODE> static void attr() {
        cudaFuncSetAttribute(col_warp_kernel<R, L, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG::SMEM);
    }
    static void prepare() {
        attr<CGM_GS>(); attr<CGM_GD_FUSED>(); attr<CGM_STATS>(); attr<CGM_COMPLEX>(); attr<CGM_STATS_KEEP>(); attr<CGM_GD_POST>();
        attr<CGM_GD_PIPE>();
    }
    static bool enabled() {
        static const bool on = !(getenv("SLM_COL_KERNEL") && getenv("SLM_COL_KERNEL")[0] == 'g');
        return on;
    }
    template <int MODE> static void run(int mode, const ColGroupArgs& ga, const TileMap& in, const TileMap& out, dim3 grid, dim3 block,
                                        cudaStream_t s) {
        if (mode != MODE) return;
        // (CGM_GD_PIPE: tiles wait for the other tiles of their plane, which other CTAs hold -- all of them must be resident)
        // (SLM_PIPE_COOP=0: plain launch -- the grid is at most one CTA per SM, so on a device the process has to itself it
        //  is resident as a whole anyway; the kernel's time-out turns the exception into an error instead of a hang)
        static const bool coop = !(getenv("SLM_PIPE_COOP") && getenv("SLM_PIPE_COOP")[0] == '0');
        if (MODE == CGM_GD_PIPE && coop) SLM_LAUNCH_COOP((col_warp_kernel<R, L, MODE>), grid, block, WG::SMEM, s, ga, in, out);
        else SLM_LAUNCH_PDL((col_warp_kernel<R, L, MODE>), grid, block, WG::SMEM, s, ga, in, out);
        if constexpr (MODE != CGM_COMPLEX && MODE != CGM_GD_FUSED) {          // (the fused form closes its planes itself)
            if (ga.defer_close)
                SLM_LAUNCH((close_planes_kernel<R, L, MODE>), dim3((unsigned)ga.c.B), dim3(32), 0, s, ga, ga.c.W / WG::TC);
        }
    }
    static bool launch(int mode, const ColGroupArgs& ga, const TileMap& in, const TileMap& out, int ctas, cudaStream_t s) {
        if (!enabled()) return false;
        const long long tiles = (long long)ga.c.B * (ga.c.W / WG::TC);
        const dim3 grid((unsigned)(tiles < ctas ? tiles : ctas)), block(WG::THREADS);
        run<CGM_GS>(mode, ga, in, out, grid, block, s);
        run<CGM_GD_FUSED>(mode, ga, in, out, grid, block, s);
        run<CGM_GD_PIPE>(mode, ga, in, out, grid, block, s);
        run<CGM_STATS>(mode, ga, in, out, grid, block, s);
        run<CGM_STATS_KEEP>(mode, ga, in, out, grid, block, s);
        run<CGM_GD_POST>(mode, ga, in, out, grid, block, s);
        run<CGM_COMPLEX>(mode, ga, in, out, grid, block, s);
        return true;
    }
};

template <typename R, int L> struct GroupLaunch<R, L, true> {
    using GG = ColGroupGeom<R, L>;
    static void prepare() {
        ColWarpLaunch<R, L>::prepare();
        cudaFuncSetAttribute(col_group_kernel<R, L, CGM_GS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GG::SMEM);
        cudaFuncSetAttribute(col_group_kernel<R, L, CGM_STATS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GG::SMEM);
        cudaFuncSetAttribute(col_group_kernel<R, L, CGM_COMPLEX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GG::SMEM);
        cudaFuncSetAttribute(col_group_kernel<R, L, CGM_STATS_KEEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GG::SMEM);
        cudaFuncSetAttribute(col_group_kernel<R, L, CGM_GD_POST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GG::SMEM);
    }
    template <int MODE> static void run(int mode, const ColGroupArgs& ga, const TileMap& in, const TileMap& out, dim3 grid, dim3 block,
                                        cudaStream_t s) {
        if (mode != MODE) return;
        SLM_LAUNCH_PDL((col_group_kernel<R, L, MODE>), grid, block, GG::SMEM, s, ga, in, out);
        if constexpr (MODE != CGM_COMPLEX) {
            if (ga.defer_close)
                SLM_LAUNCH((close_planes_kernel<R, L, MODE>), dim3((unsigned)ga.c.B), dim3(32), 0, s, ga, ga.c.W / GG::TC);
        }
    }
    static int launch(int mode, const ColGroupArgs& ga, const TileMap& in, const TileMap& out, int ctas, cudaStream_t s) {
        static_assert(!ColWarpGeom<R, L>::OK || (ColWarpGeom<R, L>::TC == GG::TC && ColWarpGeom<R, L>::ROWB == GG::ROWB),
                      "both column kernels must share the tile maps and the per-tile partial sums");
        if (ColWarpLaunch<R, L>::launch(mode, ga, in, out, ctas, s)) return 0;
        if (mode == CGM_GD_FUSED || mode == CGM_GD_PIPE) return -1;     // only the warp-per-column kernel has them
        const long long tiles = (long long)ga.c.B * (ga.c.W / GG::TC);
        const dim3 grid((unsigned)(tiles < ctas ? tiles : ctas)), block(GG::THREADS);
        run<CGM_GS>(mode, ga, in, out, grid, block, s);
        run<CGM_STATS>(mode, ga, in, out, grid, block, s);
        run<CGM_STATS_KEEP>(mode, ga, in, out, grid, block, s);
        run<CGM_GD_POST>(mode, ga, in, out, grid, block, s);
        run<CGM_COMPLEX>(mode, ga, in, out, grid, block, s);
        return 0;
    }
};

// Row (line-contiguous) kernels: available for every line length.
template <typename R, int L> struct RowLaunch {
    using RG = RowGeom<R, L>;
    // multi-plane GS and GD (row_multiplane_kernel): built where a line is 16 points per thread or fewer, i.e. not for
    // the row-only long lines
    static constexpr bool MP = FftPlan<L>::E <= 16;
    static int check() { cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? 0 : -(int)e - 1000; }
    static void prepare() {
        if constexpr (MP) {
            cudaFuncSetAttribute(row_multiplane_kernel<R, L, ALG_MP, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
            cudaFuncSetAttribute(row_multiplane_kernel<R, L, ALG_MP, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
            cudaFuncSetAttribute(row_multiplane_kernel<R, L, ALG_MPGD, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
            cudaFuncSetAttribute(row_multiplane_kernel<R, L, ALG_MPGD, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        }
        cudaFuncSetAttribute(row_pass_kernel<R, L, ALG_GS, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        cudaFuncSetAttribute(row_pass_kernel<R, L, ALG_GS, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        cudaFuncSetAttribute(row_pass_kernel<R, L, ALG_GD, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        cudaFuncSetAttribute(row_pass_kernel<R, L, ALG_GD, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        cudaFuncSetAttribute(row_plain_kernel<R, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        cudaFuncSetAttribute(row_fourier_kernel<R, L, RF_GS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        cudaFuncSetAttribute(row_fourier_kernel<R, L, RF_GD_MAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
        cudaFuncSetAttribute(row_fourier_kernel<R, L, RF_GD_POST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RG::SMEM);
    }
    static int row_pass(int alg, const RowArgs& a, cudaStream_t s) {
        const dim3 grid((unsigned)((long long)a.B * a.H / RG::NR)), block(RG::THREADS);
        if (alg == ALG_MP || alg == ALG_MPGD) {
            if constexpr (MP) {
                if (alg == ALG_MPGD) {
                    if (a.final_pass) SLM_LAUNCH_PDL((row_multiplane_kernel<R, L, ALG_MPGD, 1>), grid, block, RG::SMEM, s, a);
                    else SLM_LAUNCH_PDL((row_multiplane_kernel<R, L, ALG_MPGD, 0>), grid, block, RG::SMEM, s, a);
                } else if (a.final_pass) SLM_LAUNCH_PDL((row_multiplane_kernel<R, L, ALG_MP, 1>), grid, block, RG::SMEM, s, a);
                else SLM_LAUNCH_PDL((row_multiplane_kernel<R, L, ALG_MP, 0>), grid, block, RG::SMEM, s, a);
            } else {
                return -1;
            }
        } else if (alg == ALG_GS) {
            if (a.final_pass) SLM_LAUNCH_PDL((row_pass_kernel<R, L, ALG_GS, 1>), grid, block, RG::SMEM, s, a);
            else SLM_LAUNCH_PDL((row_pass_kernel<R, L, ALG_GS, 0>), grid, block, RG::SMEM, s, a);
        } else {
            if (a.final_pass) SLM_LAUNCH_PDL((row_pass_kernel<R, L, ALG_GD, 1>), grid, block, RG::SMEM, s, a);
            else SLM_LAUNCH_PDL((row_pass_kernel<R, L, ALG_GD, 0>), grid, block, RG::SMEM, s, a);
        }
        return check();
    }
    static int row_plain(const PlainRowArgs& a, cudaStream_t s) {
        const dim3 grid((unsigned)((long long)a.B * a.H / RG::NR)), block(RG::THREADS);
        SLM_LAUNCH((row_plain_kernel<R, L>), grid, block, RG::SMEM, s, a);
        return check();
    }
    static int row_fourier(const RowFourierArgs& a, cudaStream_t s) {
        const dim3 grid((unsigned)(a.rows / RG::NR)), block(RG::THREADS);
        if (a.mode == RF_GD_MAX) SLM_LAUNCH((row_fourier_kernel<R, L, RF_GD_MAX>), grid, block, RG::SMEM, s, a);
        else if (a.mode == RF_GD_POST) SLM_LAUNCH((row_fourier_kernel<R, L, RF_GD_POST>), grid, block, RG::SMEM, s, a);
        else SLM_LAUNCH((row_fourier_kernel<R, L, RF_GS>), grid, block, RG::SMEM, s, a);
        return check();
    }
};

// Column kernels: line lengths up to 4096.
template <typename R, int L> struct ColLaunch {
    using CG = ColGeom<R, L>;
    using GG = ColGroupGeom<R, L>;
    static int check() { cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? 0 : -(int)e - 1000; }
    static void prepare() {
        cudaFuncSetAttribute(col_pass_kernel<R, L, ALG_GS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CG::SMEM);
        cudaFuncSetAttribute(col_pass_kernel<R, L, ALG_GD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CG::SMEM);
        cudaFuncSetAttribute(col_pass_kernel<R, L, ALG_GSW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CG::SMEM);
        cudaFuncSetAttribute(col_gsw_stats_kernel<R, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CG::SMEM);
        cudaFuncSetAttribute(col_plain_kernel<R, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CG::SMEM);
        GroupLaunch<R, L>::prepare();
    }
    static int col_pass(int alg, const ColArgs& a, cudaStream_t s) {
        const dim3 grid((unsigned)((long long)a.B * (a.W / CG::TC))), block(CG::THREADS);
        if (alg == ALG_GS) SLM_LAUNCH((col_pass_kernel<R, L, ALG_GS>), grid, block, CG::SMEM, s, a);
        else if (alg == ALG_GSW) SLM_LAUNCH((col_pass_kernel<R, L, ALG_GSW>), grid, block, CG::SMEM, s, a);
        else if (alg == ALG_GSW_STATS) SLM_LAUNCH((col_gsw_stats_kernel<R, L>), grid, block, CG::SMEM, s, a);
        else SLM_LAUNCH((col_pass_kernel<R, L, ALG_GD>), grid, block, CG::SMEM, s, a);
        return check();
    }
    static int col_plain(const PlainColArgs& a, cudaStream_t s) {
        const dim3 grid((unsigned)((long long)a.B * (a.W / CG::TC))), block(CG::THREADS);
        SLM_LAUNCH((col_plain_kernel<R, L>), grid, block, CG::SMEM, s, a);
        return check();
    }
    // warp-specialised persistent column kernel; mode = ColGroupMode.  -1: not available for this line length
    static int col_group(int mode, const ColGroupArgs& ga, const void* map_in, const void* map_out, int ctas, cudaStream_t s) {
        if (!GG::OK) return -1;
        const int r = GroupLaunch<R, L>::launch(mode, ga, *static_cast<const TileMap*>(map_in), *static_cast<const TileMap*>(map_out), ctas, s);
        return r ? r : check();
    }
};

}  // namespace slm
