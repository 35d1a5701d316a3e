// Tensor-core (tcgen05) arithmetic of the step path -- AOG_PRECISION_TENSOR.
#pragma once
#include "common.cuh"

int aog_tensor_create(aog_env* env);
int aog_tensor_table_updated(aog_env* env, int which, const void* host);
int aog_tensor_screens_updated(aog_env* env);
// every env's screen times factor_dev[env] (device [B]) and its phase tiles rewritten, stream-ordered on st
int aog_tensor_rescale_screens(aog_env* env, const double* factor_dev, cudaStream_t st);
int aog_tensor_optics(aog_env* env, bool flat_dm, bool with_reward, const aog_outputs& out, cudaStream_t st);
int aog_tensor_check(aog_env* env);
int aog_tensor_actuators(aog_env* env, const void* actions_dev, int act_dtype, cudaStream_t st);
int aog_tensor_get_field(aog_env* env, int which, int env_in_chunk, double* host_out, size_t count);
// Shack-Hartmann integrator on the tensor cores (sh_tensor.cuh).  AOG_ERR_UNSUPPORTED (nothing launched) when the
// SH tables do not have the structure the kernels need -- the caller then runs the FP64 kernels.
int aog_tensor_sh_step(aog_env* env, int noise_mode, double* action_out_dev, cudaStream_t st);
// noise-free camera image of one env through the tensor-core kernels (tests)
int aog_tensor_sh_image(aog_env* env, int env_index, double* host_out, size_t count);
int aog_tensor_debug_poisson(int device, double lambda, int n, uint64_t seed, double* host_out);
int aog_tensor_debug_normals(int device, int generator, int philox, int n, const uint32_t* words_in, uint32_t* raw_out,
                             float* normals_out);
