// b2s_icp_batch_f32: the batched ICP kernel instantiated for float32 input clouds (one translation unit per
// input type so the two sets of template instances compile in parallel).
#include "b2s_icp_kernel.cuh"

using namespace b2s;

extern "C" int b2s_icp_batch_f32(const float *tar_xy, const float *src_xy, int pairs, int n_src,
                                 int n_tar, int max_iter, double tol, double *T_out,
                                 int32_t *iters_out, void *stream)
{
    return launch_icp<float>(tar_xy, src_xy, pairs, n_src, n_tar, max_iter, tol, T_out, iters_out, nullptr, stream);
}

extern "C" int b2s_icp_batch_ranges(const float *tar_ranges, const float *src_ranges, const double *beam_cs,
                                    double clamp_inf_to, int pairs, int n, int max_iter, double tol, double *T_out,
                                    int32_t *iters_out, void *stream)
{
    return launch_icp_ranges(tar_ranges, src_ranges, beam_cs, clamp_inf_to, pairs, n, max_iter, tol, T_out, iters_out, stream);
}
