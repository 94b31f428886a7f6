// oracle/ref_path_scaled.cpp — TEST INFRASTRUCTURE: libref_path_scaled_<variant>.so, the reference's own source of the path
// with `useScale` on (oracle/scale.mk explains the build): ref_path_shim.cpp as it is, plus the C entry point that sets the
// getScale spec.
#include "_ref/scaled/ref_path_shim.cpp"

extern "C" {
// the spec of getScale: n[2], c[2], a/w/phi[2][4] row-major
void ref_set_scale(void *h, const int *n, const double *c, const double *a, const double *w, const double *phi) {
    auto &S = ((RefCtx *)h)->sv.scale_spec;
    for (int ax = 0; ax < 2; ++ax) {
        S.n[ax] = n[ax];
        S.c[ax] = c[ax];
        for (int k = 0; k < 4; ++k) {
            S.a[ax][k] = a[4 * ax + k];
            S.w[ax][k] = w[4 * ax + k];
            S.phi[ax][k] = phi[4 * ax + k];
        }
    }
}
}
