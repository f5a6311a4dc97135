// Host plumbing shared by fpc_kernels.cu and fpc_puct.cu: the error path of the C-ABI and the board sizes the kernels
// are compiled for.
#pragma once
#include <cuda_runtime.h>

#include <string>

#include "../../include/fpc.h"
#include "fpc_device.cuh"

namespace fpc {

// Sets the message fpc_last_error returns and gives back `code` (fpc_kernels.cu).
int fail(int code, const std::string &msg);
// FPC_OK, or fail(FPC_ERR_CUDA, "<what>: <CUDA error string>").
int cuda_check(cudaError_t e, const char *what);

#define CK(expr)                         \
  do {                                   \
    int rc_ = cuda_check((expr), #expr); \
    if (rc_ != FPC_OK) return rc_;       \
  } while (0)

// The compiled board sizes: f(Geo<R, IA>()) for one of them (f returns an FPC_* code), FPC_ERR_ARG for any other R.
// Callers name the geometry as decltype(g).
template <class F>
int dispatch(int R, F &&f) {
  switch (R) {
    case 14: return f(Geo<14, 3>());
    case 13: return f(Geo<13, 3>());
    case 10: return f(Geo<10, 2>());
    case 8: return f(Geo<8, 2>());
    default: return fail(FPC_ERR_ARG, "unsupported board size R=" + std::to_string(R));
  }
}

// The invalid-corner width IA of each size above; -1 for any other R (fpc_supported, fpc_invalid_area).
inline int ia_of(int R) { return R == 14 || R == 13 ? 3 : (R == 10 || R == 8 ? 2 : -1); }

}  // namespace fpc
