// compute.cpp -- the C entry points of the tensor-core check (include/b200dp.h, "tensor-core check").
//
// They live apart from ctx.cpp because they are only meaningful with the CUDA half of the library (cuda_backend.cu,
// tc_check.cuh): the CPU half (kfd.cpp, allocator.cpp, labels.cpp, ctx.cpp) builds and links without them.
#include <cstring>

#include "internal.hpp"
#include "tc_math.hpp"

using namespace b2dp;

extern "C" int b2dp_compute_check(b2dp_ctx* c, const b2dp_compute_opts* opts, b2dp_compute_result* out, int cap, int* n) {
    if (!c || !n || cap < 0) return B2DP_E_INVAL;
    CudaBackend* be = ctx_cuda_backend(c);
    if (!be) return ctx_fail(B2DP_E_UNSUPPORTED, "the tensor-core check needs the cuda: backend (there is no CPU fallback)");
    std::vector<b2dp_compute_result> res;
    std::string err;
    int rc = cuda_compute_check(be, opts, res, err);
    if (rc != B2DP_OK) return ctx_fail(rc, err);
    *n = (int)res.size();
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !out) return B2DP_E_INVAL;
    memcpy(out, res.data(), res.size() * sizeof(b2dp_compute_result));
    return B2DP_OK;
}

extern "C" int b2dp_compute_tile(b2dp_ctx* c, int device, int kind, int a_set, int b_set, float* out) {
    if (!c || !out || kind < 0 || kind > 1 || a_set < 0 || a_set >= tc::kSets || b_set < 0 || b_set >= tc::kSets) return B2DP_E_INVAL;
    CudaBackend* be = ctx_cuda_backend(c);
    if (!be) return ctx_fail(B2DP_E_UNSUPPORTED, "cuda: backend only");
    std::string err;
    int rc = cuda_compute_tile(be, device, kind, a_set, b_set, out, err);
    return rc == B2DP_OK ? rc : ctx_fail(rc, err);
}

extern "C" int b2dp_compute_inject_fault(b2dp_ctx* c, int device, int sm, uint32_t mask) {
    if (!c || sm < 0 || sm >= 256) return B2DP_E_INVAL;
    CudaBackend* be = ctx_cuda_backend(c);
    if (!be) return ctx_fail(B2DP_E_UNSUPPORTED, "cuda: backend only");
    std::string err;
    int rc = cuda_compute_inject_fault(be, device, sm, mask, err);
    return rc == B2DP_OK ? rc : ctx_fail(rc, err);
}

extern "C" int b2dp_compute_expected(uint32_t seed, int kind, int a_set, int b_set, uint64_t* row_hash, int cap, int* n) {
    if (!n || kind < 0 || kind > 1 || a_set < 0 || a_set >= tc::kSets || b_set < 0 || b_set >= tc::kSets) return B2DP_E_INVAL;
    *n = tc::kM;
    if (cap < tc::kM) return B2DP_E_NOSPC;
    if (!row_hash) return B2DP_E_INVAL;
    tc::row_hashes(seed, a_set, b_set, row_hash);  // both kinds accumulate the same exact integers
    return B2DP_OK;
}
