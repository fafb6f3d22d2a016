// Epilogue shared by the cp.async- and the TMA-staged DMMA tile kernels: each thread owns, per 8x8 fragment,
// row = lane/4 and two adjacent columns 2*(lane%4).
#pragma once
#include "common.cuh"

namespace gpmc {

__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

template <int FM, int FN, int BM_, int BN_>
__device__ __forceinline__ void gemm_epilogue(const GemmArgs &p, int m, int tm, int tn, int wm, int wn, int frow, int fk,
                                              int rows_valid, int cols_valid, double (&acc)[FM][FN][2])
{
    // the C tile's rows lie in one 128-row block: one row stride p.C.ld in either layout of BatchView
    double *Cb = view_elem(p.C, m, p.cr0 + tm * BM_, p.cc0 + tn * BN_);
    const int ldc = p.C.ld;
    const double *sv = (p.epi == EPI_R) ? p.svec + (size_t)m * p.stride_s : nullptr;
#pragma unroll
    for (int i = 0; i < FM; ++i) {
        const int rl = wm * FM * 8 + i * 8 + frow;
        if (rl >= rows_valid) continue;
        const int gr = p.cr0 + tm * BM_ + rl;
        double *crow = Cb + (size_t)rl * ldc;
        const double s_r = sv ? sv[gr] : 0.0;
#pragma unroll
        for (int j = 0; j < FN; ++j) {
            const int cl = wn * FN * 8 + j * 8 + fk * 2;
            if (cl >= cols_valid) continue;
            const bool two = (cl + 1 < cols_valid);
            double v0 = acc[i][j][0], v1 = acc[i][j][1];
            if (p.epi == EPI_SUB) {
                if (two) { const double2 c = *reinterpret_cast<const double2 *>(crow + cl); v0 = c.x - v0; v1 = c.y - v1; }
                else v0 = crow[cl] - v0;
            } else if (p.epi == EPI_ADD) {
                if (two) { const double2 c = *reinterpret_cast<const double2 *>(crow + cl); v0 = c.x + v0; v1 = c.y + v1; }
                else v0 = crow[cl] + v0;
            } else if (p.epi == EPI_NEGSET) {
                v0 = -v0; v1 = -v1;
            } else if (p.epi == EPI_R) {
                // R = S - S P S  (+ 1e-11 on the diagonal, sliceSample.py:205)
                const int gc = p.cc0 + tn * BN_ + cl;
                const double s_c0 = sv[gc], s_c1 = two ? sv[gc + 1] : 0.0;
                v0 = -(s_r * v0 * s_c0);
                v1 = -(s_r * v1 * s_c1);
                if (gr == gc) v0 = (s_r + v0) + 1e-11;
                if (gr == gc + 1) v1 = (s_r + v1) + 1e-11;
            }
            if (two) *reinterpret_cast<double2 *>(crow + cl) = make_double2(v0, v1);
            else crow[cl] = v0;
        }
    }
}

// tile decode shared by both kernels
template <int BM_, int BN_>
__device__ __forceinline__ void gemm_tile_decode(const GemmArgs &p, int t, int &tm, int &tn)
{
    if (p.lower_only) {
        // row tile tm has Q*(tm+1) column tiles on or below the diagonal, Q = BM / BN
        constexpr int Q = BM_ / BN_;
        tm = (int)((sqrt(8.0 * (double)t / Q + 1.0) - 1.0) * 0.5);
        while (Q * (tm + 1) * (tm + 2) / 2 <= t) ++tm;
        while (Q * tm * (tm + 1) / 2 > t) --tm;
        tn = t - Q * tm * (tm + 1) / 2;
    } else {
        const int tiles_n = (p.cols + BN_ - 1) / BN_;
        tm = t / tiles_n;
        tn = t - tm * tiles_n;
    }
}

}  // namespace gpmc
