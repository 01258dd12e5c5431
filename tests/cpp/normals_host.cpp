/* TEST INFRASTRUCTURE ONLY — the host build of the analytic normals (csrc/mcb_bytecode.h: mcb_interp_grad_scalar,
 * mcb_grad_normalise) on the product's own lowering, through oracle/host_interp_fn.cpp (included unchanged).
 *   int mcnh_eval(eq, xyz, n, sx, sy, sz, value, plain, grad, nrm)
 *       for each of the n points (unscaled x, y, z): value = the value part of mcb_interp_grad_scalar at (sx*x, sy*y, sz*z),
 *       plain = mcb_interp_scalar there (what mcb_eval_points returns), grad = the gradient (3 floats), nrm = its normal
 *   void mcnh_normalise(g, out, n)   mcb_grad_normalise of n gradients
 * Built by tests/normals_common.py with -ffp-contract=off, as the product's host code is. */
#include "../../oracle/host_interp_fn.cpp"

extern "C" int mcnh_eval(const char* eq, const float* xyz, long n, float sx, float sy, float sz, float* value, float* plain,
                         float* grad, float* nrm) {
    mcb::Compiled c;
    int rc = mcb::compile(eq, c, nullptr, g_grammar);
    if (rc != MCB_OK) return rc;
    fold(c);
    const uint32_t* code = c.point_code.data();
    const int nc = (int)c.point_code.size();
    for (long i = 0; i < n; i++) {
        const float x = sx * xyz[3 * i], y = sy * xyz[3 * i + 1], z = sz * xyz[3 * i + 2];
        value[i] = mcb_interp_grad_scalar(code, nc, c.kpool.data(), x, y, z, sx, sy, sz, grad + 3 * i);
        plain[i] = mcb_interp_scalar(code, nc, c.kpool.data(), x, y, z, nullptr, nullptr, nullptr);
        mcb_grad_normalise(grad + 3 * i, nrm + 3 * i);
    }
    return MCB_OK;
}

extern "C" void mcnh_normalise(const float* g, float* out, long n) {
    for (long i = 0; i < n; i++) mcb_grad_normalise(g + 3 * i, out + 3 * i);
}
