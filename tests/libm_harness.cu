// Host harness of tests/test_libm_replica*.py: mpp_exp / mpp_pow (mpp_libm.cuh) next to the host libm's exp / pow on
// the same arguments, out[2i] = exp(e[i]), out[2i+1] = pow(x[i], y[i]).  Built with the library's host flags
// (-ffp-contract=off), so the replica is compiled here as it is in libmpp_b200.
#include <math.h>

#include "../maaco_path_planing_b200/csrc/mpp_libm.cuh"

extern "C" void replica_exp_pow(long n, const double *e, const double *x, const double *y, double *out) {
    for (long i = 0; i < n; ++i) {
        out[2 * i] = mpp_exp(e[i]);
        out[2 * i + 1] = mpp_pow(x[i], y[i]);
    }
}

extern "C" void libm_exp_pow(long n, const double *e, const double *x, const double *y, double *out) {
    for (long i = 0; i < n; ++i) {
        out[2 * i] = exp(e[i]);
        out[2 * i + 1] = pow(x[i], y[i]);
    }
}
