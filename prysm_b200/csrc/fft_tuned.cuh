// Register-resident FFT kernels for the hot shapes (see fft_tuned.cu).  Each try_* returns
// PB_ERR_UNSUPPORTED *without touching the error string* when the shape is not one it covers;
// the caller then falls through to the generic shared-memory pass.
#pragma once
#include "axis_pass.cuh"

namespace pb {

int try_tuned_axis_pass(Handle* h, const AxisPass& p, cudaStream_t st);

int try_tuned_fft2(Handle* h, int dtype, const void* in, int in_kind, const void* amp, int amp_kind, double kturns,
                   int ny, int nx, long long in_ld, int ky, int kx, int dir, double scale, int shift_in,
                   int shift_out, void* out, int out_kind, double weight, int oy, int ox, long long out_ld,
                   cudaStream_t st);

int try_tuned_fft2_batch(Handle* h, int dtype, const void* in, int in_kind, const void* amp, int amp_kind, double kturns,
                         int batch, long long in_bs, long long amp_bs, int ny, int nx, long long in_ld, int ky, int kx,
                         int dir, double scale, int shift_in, int shift_out, void* out, int out_kind, double weight,
                         int oy, int ox, long long out_ld, long long out_bs, cudaStream_t st);

}  // namespace pb
