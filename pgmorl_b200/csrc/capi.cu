// Error plumbing and trivial entry points of the C ABI (include/pgmorl_b200.h).
#include <stdarg.h>

#include "common.cuh"

namespace pgm {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what) {
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return PGM_ERR_CUDA;
}

}  // namespace pgm

extern "C" int pgm_abi_version(void) { return PGM_ABI_VERSION; }
extern "C" const char *pgm_last_error(void) { return pgm::g_err; }
// Validates (hidden, dist, n) of the _x layout functions; `who` names the caller in the error.
static bool layout_args_ok(const char *who, int A, int hidden, int dist) {
    if (!pgm::hidden_supported(hidden)) {
        pgm::set_error("%s: hidden width %d is not one of {32, 64, 128}", who, hidden);
        return false;
    }
    if (!pgm::dist_supported(dist)) {
        pgm::set_error("%s: unknown action head %d (PGM_DIST_GAUSSIAN = 0, PGM_DIST_CATEGORICAL = 1)", who, dist);
        return false;
    }
    if (dist == PGM_DIST_CATEGORICAL && (A < 1 || A > pgm::CAT_MAX)) {
        pgm::set_error("%s: a categorical head has 1..%d categories, got %d", who, pgm::CAT_MAX, A);
        return false;
    }
    return true;
}

extern "C" int pgm_n_par_x(int O, int A, int M, int hidden, int dist) {
    if (!layout_args_ok("pgm_n_par_x", A, hidden, dist)) return -1;
    return pgm::NetLayout(O, A, M, hidden, dist).n_par;
}
extern "C" int pgm_n_par_h(int O, int A, int M, int hidden) {
    if (!pgm::hidden_supported(hidden)) {
        pgm::set_error("pgm_n_par_h: hidden width %d is not one of {32, 64, 128}", hidden);
        return -1;
    }
    return pgm_n_par_x(O, A, M, hidden, PGM_DIST_GAUSSIAN);
}
extern "C" int pgm_n_par(int O, int A, int M) { return pgm_n_par_h(O, A, M, PGM_HIDDEN); }

// Offsets of the 13 parameter tensors (12 for a Categorical head, which has no logstd) inside one flat vector, in
// named_parameters() order (pgmorl_b200/layout.py): the kernels and the Python state_dict slicing must agree on them
// (tests/test_cabi.py, tests/test_oracle_hidden.py, tests/test_oracle_discrete.py).
extern "C" int pgm_param_offsets_x(int O, int A, int M, int hidden, int dist, int *out) {
    if (!out) return PGM_ERR_ARG;
    if (!layout_args_ok("pgm_param_offsets_x", A, hidden, dist)) return PGM_ERR_ARG;
    const pgm::NetLayout L(O, A, M, hidden, dist);
    const int v[13] = {L.oW1a, L.ob1a, L.oW2a, L.ob2a, L.oW1c, L.ob1c, L.oW2c, L.ob2c, L.oWv, L.obv, L.oWmu, L.obmu, L.ols};
    for (int i = 0; i < (L.nls ? 13 : 12); ++i) out[i] = v[i];
    return PGM_OK;
}
extern "C" int pgm_param_offsets_h(int O, int A, int M, int hidden, int *out13) {
    if (!out13) return PGM_ERR_ARG;
    if (!pgm::hidden_supported(hidden)) {
        pgm::set_error("pgm_param_offsets_h: hidden width %d is not one of {32, 64, 128}", hidden);
        return PGM_ERR_ARG;
    }
    return pgm_param_offsets_x(O, A, M, hidden, PGM_DIST_GAUSSIAN, out13);
}
extern "C" int pgm_param_offsets(int O, int A, int M, int *out13) { return pgm_param_offsets_h(O, A, M, PGM_HIDDEN, out13); }
