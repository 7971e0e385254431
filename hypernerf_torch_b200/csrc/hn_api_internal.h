// Internal helpers shared by the .cu translation units behind include/hypernerf_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/hypernerf_b200.h"

namespace hn {
// thread-local last-error message (hn_last_error)
int set_error(int code, const char* msg);
int set_cuda_error(cudaError_t e, const char* where);  // returns 0 when e == cudaSuccess
int num_sms();                                         // cached SM count of the current device
}  // namespace hn
