// b2s_icp_batch_f64: the batched ICP kernel instantiated for float64 input clouds (one translation unit per
// input type so the two sets of template instances compile in parallel).
#include "b2s_icp_kernel.cuh"

using namespace b2s;

extern "C" int b2s_icp_batch_f64(const double *tar_xy, const double *src_xy, int pairs, int n_src,
                                 int n_tar, int max_iter, double tol, double *T_out,
                                 int32_t *iters_out, void *stream)
{
    return launch_icp<double>(tar_xy, src_xy, pairs, n_src, n_tar, max_iter, tol, T_out, iters_out, nullptr, stream);
}

extern "C" int b2s_icp_batch_f64_err(const double *tar_xy, const double *src_xy, int pairs, int n_src, int n_tar,
                                     int max_iter, double tol, double *T_out, int32_t *iters_out, double *err_out,
                                     void *stream)
{
    return launch_icp<double>(tar_xy, src_xy, pairs, n_src, n_tar, max_iter, tol, T_out, iters_out, err_out, stream);
}
