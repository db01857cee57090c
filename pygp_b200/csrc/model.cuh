// model.cuh -- the ExactGP device state behind `pgp_model*` (capi.cu owns its life cycle; dist.cu runs
// the distributed factorisation and gradient on the same buffers).
#pragma once

#include "chol.cuh"
#include "gram.cuh"
#include "spec.cuh"

struct pgp_model {
    using DevSpec = pgp::DevSpec;
    pgp_ctx* ctx = nullptr;
    pgp_kernel_spec spec;
    int64_t n = 0;
    int ndim = 0;
    int64_t ld = 0;
    int64_t cap = 0;             // rows F can hold in place (ld = lead_dim(cap)); grows in steps on append
    int64_t xcap = 0;            // rows allocated for X, y, Z, alpha
    double* d_X = nullptr;
    double* d_y = nullptr;
    double* d_Z = nullptr;       // [parts][n][ndim]
    DevSpec* d_spec = nullptr;
    double* d_F = nullptr;       // (n + 1, ld): L below/on the diagonal, a in row n
    double* d_G = nullptr;       // (n, ld): V = L^-T (upper); allocated on first gradient
    double* d_H = nullptr;       // (n, ld): K~^-1 (lower)
    double* d_alpha = nullptr;   // (n)
    double* d_partials = nullptr;
    double* d_res = nullptr;     // [0] lZ, [1..] dlZ
    int* d_info = nullptr;
    double* d_Bc = nullptr;      // predict chunk (bc_rows, ld)
    int64_t bc_rows = 0;
    DevSpec hspec;
    bool factored = false;
    double lZ = 0.0;
    int info = 0;
};
