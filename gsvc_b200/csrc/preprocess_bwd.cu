// Kernel (4'): per-Gaussian backward (SURVEY.md Appendix A.4, second half).
// (dL/dpix, dL/dconic, dL/dopacity, dL/drgb) accumulated by the blend backward  →
// dL/dmeans3D, means2D.grad, dL/dscales, dL/drotations | dL/dcov3D, dL/dcolors | dL/dshs, dL/dopacities.
// Under the orthographic camera the pixel position enters nothing but `pix`, so unlike the
// perspective rasterizer there is no mean → cov2D term.
// Pure stream over P Gaussians: HBM-bound (reads 4 P + ~100 V, writes 68 P bytes).
#include "collective.cuh"

namespace gsvc {

__device__ __forceinline__ float ldVb(const DevSettings& s, int v, int r, int c)
{
    return __ldg(s.vt.V[v] + r * s.vt.vs_r[v] + c * s.vt.vs_c[v]);
}

__constant__ float B_SH_C0 = 0.28209479177387814f;
__constant__ float B_SH_C1 = 0.4886025119029199f;
__constant__ float B_SH_C2[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f,
                                 -1.0925484305920792f, 0.5462742152960396f};
__constant__ float B_SH_C3[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f,
                                 0.3731763325901154f, -0.4570457994644658f, 1.445305721320277f,
                                 -0.5900435899266435f};

// SH backward: basis derivatives of /root/reference/utils/sh_utils.py:57-110 w.r.t. coefficients and direction.
// ACCUMULATES into dsh (the caller zeroes it): a batch of views sums its views' contributions.
__device__ void sh_backward(int deg, int M, const float* sh, float* dsh, const float p[3], const float campos[3],
                            const float dL[3], float dmean[3])
{
    const float dxv = p[0] - campos[0], dyv = p[1] - campos[1], dzv = p[2] - campos[2];
    const float len = sqrtf(dxv * dxv + dyv * dyv + dzv * dzv);
    const float x = dxv / len, y = dyv / len, z = dzv / len;
    float ddx = 0.f, ddy = 0.f, ddz = 0.f;
    for (int c = 0; c < 3; c++) {
        const float g = dL[c];
        float rx = 0.f, ry = 0.f, rz = 0.f;
        dsh[0 * 3 + c] += B_SH_C0 * g;
        if (deg > 0) {
            dsh[1 * 3 + c] += -B_SH_C1 * y * g;
            dsh[2 * 3 + c] += B_SH_C1 * z * g;
            dsh[3 * 3 + c] += -B_SH_C1 * x * g;
            rx = -B_SH_C1 * sh[3 * 3 + c];
            ry = -B_SH_C1 * sh[1 * 3 + c];
            rz = B_SH_C1 * sh[2 * 3 + c];
            if (deg > 1) {
                const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
                dsh[4 * 3 + c] += B_SH_C2[0] * xy * g;
                dsh[5 * 3 + c] += B_SH_C2[1] * yz * g;
                dsh[6 * 3 + c] += B_SH_C2[2] * (2.f * zz - xx - yy) * g;
                dsh[7 * 3 + c] += B_SH_C2[3] * xz * g;
                dsh[8 * 3 + c] += B_SH_C2[4] * (xx - yy) * g;
                rx += B_SH_C2[0] * y * sh[4 * 3 + c] + B_SH_C2[2] * 2.f * -x * sh[6 * 3 + c] +
                      B_SH_C2[3] * z * sh[7 * 3 + c] + B_SH_C2[4] * 2.f * x * sh[8 * 3 + c];
                ry += B_SH_C2[0] * x * sh[4 * 3 + c] + B_SH_C2[1] * z * sh[5 * 3 + c] +
                      B_SH_C2[2] * 2.f * -y * sh[6 * 3 + c] + B_SH_C2[4] * 2.f * -y * sh[8 * 3 + c];
                rz += B_SH_C2[1] * y * sh[5 * 3 + c] + B_SH_C2[2] * 4.f * z * sh[6 * 3 + c] +
                      B_SH_C2[3] * x * sh[7 * 3 + c];
                if (deg > 2) {
                    dsh[9 * 3 + c] += B_SH_C3[0] * y * (3.f * xx - yy) * g;
                    dsh[10 * 3 + c] += B_SH_C3[1] * xy * z * g;
                    dsh[11 * 3 + c] += B_SH_C3[2] * y * (4.f * zz - xx - yy) * g;
                    dsh[12 * 3 + c] += B_SH_C3[3] * z * (2.f * zz - 3.f * xx - 3.f * yy) * g;
                    dsh[13 * 3 + c] += B_SH_C3[4] * x * (4.f * zz - xx - yy) * g;
                    dsh[14 * 3 + c] += B_SH_C3[5] * z * (xx - yy) * g;
                    dsh[15 * 3 + c] += B_SH_C3[6] * x * (xx - 3.f * yy) * g;
                    rx += B_SH_C3[0] * sh[9 * 3 + c] * 6.f * xy + B_SH_C3[1] * sh[10 * 3 + c] * yz +
                          B_SH_C3[2] * sh[11 * 3 + c] * -2.f * xy + B_SH_C3[3] * sh[12 * 3 + c] * -6.f * xz +
                          B_SH_C3[4] * sh[13 * 3 + c] * (-3.f * xx + 4.f * zz - yy) +
                          B_SH_C3[5] * sh[14 * 3 + c] * 2.f * xz + B_SH_C3[6] * sh[15 * 3 + c] * 3.f * (xx - yy);
                    ry += B_SH_C3[0] * sh[9 * 3 + c] * 3.f * (xx - yy) + B_SH_C3[1] * sh[10 * 3 + c] * xz +
                          B_SH_C3[2] * sh[11 * 3 + c] * (-3.f * yy + 4.f * zz - xx) +
                          B_SH_C3[3] * sh[12 * 3 + c] * -6.f * yz + B_SH_C3[4] * sh[13 * 3 + c] * -2.f * xy +
                          B_SH_C3[5] * sh[14 * 3 + c] * -2.f * yz + B_SH_C3[6] * sh[15 * 3 + c] * -6.f * xy;
                    rz += B_SH_C3[1] * sh[10 * 3 + c] * xy + B_SH_C3[2] * sh[11 * 3 + c] * 8.f * yz +
                          B_SH_C3[3] * sh[12 * 3 + c] * 3.f * (2.f * zz - xx - yy) +
                          B_SH_C3[4] * sh[13 * 3 + c] * 8.f * xz + B_SH_C3[5] * sh[14 * 3 + c] * (xx - yy);
                }
            }
        }
        ddx += rx * g; ddy += ry * g; ddz += rz * g;
    }
    const float dot = x * ddx + y * ddy + z * ddz;  // through dir = d / |d|
    dmean[0] += (ddx - x * dot) / len;
    dmean[1] += (ddy - y * dot) / len;
    dmean[2] += (ddz - z * dot) / len;
}

// g: the parameter row.  Shared set (RAGGED false): the views' states at v*P + g, summed over the views.  Ragged: row g
// belongs to `view` alone, and its state is at row g itself.
template <bool RAGGED>
__device__ __forceinline__ void gaussian_backward(const DevSettings& s, const PreInputs& in,
                                                  const int32_t* __restrict__ radii, const GeomView& geo,
                                                  const float4* __restrict__ acc, const BwdOutputs& out, const int g,
                                                  const int view)
{
    float dmean[3] = {0.f, 0.f, 0.f}, dcol[3] = {0.f, 0.f, 0.f}, dop = 0.f;
    float dsc[3] = {0.f, 0.f, 0.f}, drot[4] = {0.f, 0.f, 0.f, 0.f}, dcov[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (in.shs && out.dL_dshs) {
        float* dsh = out.dL_dshs + (size_t)g * s.sh_M * 3;
        for (int k = 0; k < s.sh_M * 3; k++) dsh[k] = 0.f;
    }

    // A batch of views shares the Gaussian parameters: their gradients are summed here, in view order, so the
    // batch writes ONE dense gradient instead of n_views of them plus the adds.  A ragged row has one view: no sum.
    for (int v = RAGGED ? view : 0; v < (RAGGED ? view + 1 : s.n_views); v++) {
    const size_t gv = RAGGED ? (size_t)g : (size_t)v * in.P + g;
    const bool vis = radii[gv] > 0;
    float dm2[2] = {0.f, 0.f};
    if (vis) {
        // blend-backward accumulators: raw moments of w = Gs dL/dGs in the whitened offset (u, v) = L^T d (render.cu)
        //   a0 = (S w u, S w v, S w u^2, S w u v)  a1 = (S w v^2, S w, dL/dr, dL/dg)  a2.x = dL/db
        // with L L^T = K * (stored fp32 conic), K = log2(e)/2, L = (l11 0; l11 rho, l22), rho = rho_hi + rho_lo, as the
        // preprocess kernel stored it (feat0.z, feat3)
        const float4 a0 = acc[3 * gv], a1 = acc[3 * gv + 1], a2 = acc[3 * gv + 2];
        const float4 con = geo.feat3[gv];  // (l11, rho_lo, l22, opacity)
        const double rho = (double)geo.feat0[gv].z + (double)con.y;
        const float w0[3] = {ldVb(s, v, 0, 0), ldVb(s, v, 0, 1), ldVb(s, v, 0, 2)};
        const float w1[3] = {ldVb(s, v, 1, 0), ldVb(s, v, 1, 1), ldVb(s, v, 1, 2)};
        const double W0[3] = {w0[0], w0[1], w0[2]}, W1[3] = {w1[0], w1[1], w1[2]};

        // Sigma and cov2D = (a b; b c) exactly as the forward formed them (fp32, the shared contraction-proof
        // routines of common.cuh): the conic the blend evaluated is fl(inverse) of THESE numbers, so this is the point
        // at which d(conic)/d(cov2D) = -Q (.) Q is taken — in fp64 from here on.  (Recomputing them in fp64 from the
        // inputs gives "the same" (a, b, c) to 1e-7, which for an elongated Gaussian is a different inverse: det
        // cancels by the squared axis ratio.  The oracle and the upstream design differentiate at the forward's values
        // too.)
        float covf[6], Rf[9];
        double R[9], sv[3] = {0., 0., 0.};
        if (in.cov3D_precomp) {
#pragma unroll
            for (int k = 0; k < 6; k++) covf[k] = in.cov3D_precomp[6 * (size_t)g + k];
        } else {
            const float4 q = ld_row4(in.rotations, (size_t)g);
            const float sc3[3] = {in.scales[3 * g], in.scales[3 * g + 1], in.scales[3 * g + 2]};
            cov3d_from_scale_rot(sc3, s.scale_modifier, q, covf);
            quat_to_rot(q, Rf);
#pragma unroll
            for (int k = 0; k < 9; k++) R[k] = Rf[k];
#pragma unroll
            for (int k = 0; k < 3; k++) sv[k] = (double)s.scale_modifier * (double)sc3[k];
        }
        float af, bf, cf;
        cov2d_ortho(covf, w0, w1, s.scale, af, bf, cf);
        const double a = af, b = bf, c = cf;
        const double det_inv = 1. / (a * c - b * b);
        const double qA = c * det_inv, qB = -b * det_inv, qC = a * det_inv;        // Q, exact to fp64
        // d = L^-T (u v)  =>  Q d = X (u v) with X = Q L^-T (equal to L / K up to the conic's fp32 rounding)
        const double l11 = con.x, l21 = l11 * rho, l22 = con.z;
        const double i11 = 1. / l11, i22 = 1. / l22, i12 = -rho * i22;              // L^-T = (i11 i12; 0 i22)
        const double x00 = qA * i11, x01 = qA * i12 + qB * i22;
        const double x10 = qB * i11, x11 = qB * i12 + qC * i22;
        // dL/dpix: the blend evaluates the exponent with the STORED conic = L L^T / K, so d(power)/dd = -(L L^T / K) d
        // and dL/dpix = -(1/K) L (S w u, S w v) — exactly, not through Q
        const double Kd = 0.5 * 1.4426950408889634;
        const float gpx = (float)(-(l11 * (double)a0.x) / Kd);
        const float gpy = (float)(-(l21 * (double)a0.x + l22 * (double)a0.y) / Kd);
        dop += con.w != 0.f ? a1.y / con.w : 0.f;   // a1.y = S w = opacity * S Gs dL/dalpha (zero opacity: never blended)
        const float dcv[3] = {a1.z, a1.w, a2.x};
        dcol[0] += dcv[0]; dcol[1] += dcv[1]; dcol[2] += dcv[2];
        const float p[3] = {in.means3D[3 * g], in.means3D[3 * g + 1], in.means3D[3 * g + 2]};

        if (in.shs && out.dL_dshs) {
            const uint8_t* cl = geo.clamped + 3 * gv;
            const float dL[3] = {cl[0] ? 0.f : dcv[0], cl[1] ? 0.f : dcv[1], cl[2] ? 0.f : dcv[2]};
            const float campos[3] = {s.vt.campos[v][0], s.vt.campos[v][1], s.vt.campos[v][2]};
            sh_backward(s.sh_degree, s.sh_M, in.shs + (size_t)g * s.sh_M * 3, out.dL_dshs + (size_t)g * s.sh_M * 3, p,
                        campos, dL, dmean);
        }
        // pix = (V[:2,:3] p + V[:2,3] - min) * scale - 0.5
#pragma unroll
        for (int k = 0; k < 3; k++) dmean[k] += s.scale * (w0[k] * gpx + w1[k] * gpy);
        dm2[0] = gpx * 0.5f * (float)s.W;  // U3
        dm2[1] = gpy * 0.5f * (float)s.H;

        // dL/dcov2D = -Q (dL/dQ) Q = (1/2) S w (Q d)(Q d)^T = (1/2) X M X^T, M = S w [u v][u v]^T the whitened moments:
        // a congruence — no division by det^2, no terms that cancel for an elongated Gaussian.
        const double muu = a0.z, muv = a0.w, mvv = a1.x;
        const double Jr0[3] = {(double)s.scale * W0[0], (double)s.scale * W0[1], (double)s.scale * W0[2]};   // J = scale * W[0:2,:]
        const double Jr1[3] = {(double)s.scale * W1[0], (double)s.scale * W1[1], (double)s.scale * W1[2]};
        if (in.cov3D_precomp) {
            // the covariance itself is the parameter: dL/dSigma = J^T (1/2 X M X^T) J, symmetric entries summed
            const double t00 = x00 * muu + x01 * muv, t01 = x00 * muv + x01 * mvv;      // rows of X M
            const double t10 = x10 * muu + x11 * muv, t11 = x10 * muv + x11 * mvv;
            const double da = 0.5 * (t00 * x00 + t01 * x01), db = t00 * x10 + t01 * x11, dc = 0.5 * (t10 * x10 + t11 * x11);
            double Gm[9];
#pragma unroll
            for (int k = 0; k < 3; k++)
#pragma unroll
                for (int l = 0; l < 3; l++) Gm[3 * k + l] = da * Jr0[k] * Jr0[l] + db * Jr0[k] * Jr1[l] + dc * Jr1[k] * Jr1[l];
            dcov[0] += (float)Gm[0]; dcov[1] += (float)(Gm[1] + Gm[3]); dcov[2] += (float)(Gm[2] + Gm[6]);
            dcov[3] += (float)Gm[4]; dcov[4] += (float)(Gm[5] + Gm[7]); dcov[5] += (float)Gm[8];
        } else {
            // cov2D = N N^T + 0.3 I with N = J R diag(mod * s) (2x3, column j = the image of axis j), so
            //   dL/dN = 2 (1/2 X M X^T) N = X M Z,  Z = X^T N   and   dL/d(R diag) = J^T X M Z.
            // Column by column: z_j = X^T n_j is the WHITENED image of axis j, formed in fp64 (for the long axis of a
            // needle Q n_j cancels by the squared axis ratio — fine in fp64), and only then meets the fp32 moments.
            // Going through the 3x3 dL/dSigma instead projects its dominant short-axis component away again for
            // the long axis and loses that ratio in accuracy (1e-7 * 256^2 on the test scenes).
            double dM[9];
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const double n0 = (Jr0[0] * R[j] + Jr0[1] * R[3 + j] + Jr0[2] * R[6 + j]) * sv[j];
                const double n1 = (Jr1[0] * R[j] + Jr1[1] * R[3 + j] + Jr1[2] * R[6 + j]) * sv[j];
                const double z0 = x00 * n0 + x10 * n1, z1 = x01 * n0 + x11 * n1;         // X^T n_j
                const double m0 = muu * z0 + muv * z1, m1 = muv * z0 + mvv * z1;         // M z_j
                const double b0 = x00 * m0 + x01 * m1, b1 = x10 * m0 + x11 * m1;         // X M z_j
#pragma unroll
                for (int i = 0; i < 3; i++) dM[3 * i + j] = Jr0[i] * b0 + Jr1[i] * b1;
            }
            double gR[9];
#pragma unroll
            for (int j = 0; j < 3; j++) {
                double t = 0.;
#pragma unroll
                for (int i = 0; i < 3; i++) {
                    t += dM[3 * i + j] * R[3 * i + j];
                    gR[3 * i + j] = dM[3 * i + j] * sv[j];
                }
                dsc[j] += (float)(t * (double)s.scale_modifier);
            }
            const float4 q = ld_row4(in.rotations, (size_t)g);
            const double r = q.x, x = q.y, y = q.z, z = q.w;
            drot[0] += (float)(2. * (-z * gR[1] + y * gR[2] + z * gR[3] - x * gR[5] - y * gR[6] + x * gR[7]));
            drot[1] += (float)(2. * (y * gR[1] + z * gR[2] + y * gR[3] - 2. * x * gR[4] - r * gR[5] + z * gR[6] + r * gR[7] -
                                     2. * x * gR[8]));
            drot[2] += (float)(2. * (-2. * y * gR[0] + x * gR[1] + r * gR[2] + x * gR[3] + z * gR[5] - r * gR[6] + z * gR[7] -
                                     2. * y * gR[8]));
            drot[3] += (float)(2. * (-2. * z * gR[0] - r * gR[1] + x * gR[2] + r * gR[3] - 2. * z * gR[4] + y * gR[5] +
                                     x * gR[6] + y * gR[7]));
        }
    }
    if (out.dL_dmeans2D) {
        out.dL_dmeans2D[3 * gv] = dm2[0]; out.dL_dmeans2D[3 * gv + 1] = dm2[1]; out.dL_dmeans2D[3 * gv + 2] = 0.f;
    }
    }   // views

    if (out.packed) {
        // [P,14] row = (means3D 3, colours 3, opacity 1, scales 3, rotation 4): the layout the frame-sharded
        // all-reduce sums (sharding.GRAD_LAYOUT), written here so that no pack kernel is needed
        float2* row = reinterpret_cast<float2*>(out.packed + 14 * (size_t)g);
        row[0] = make_float2(dmean[0], dmean[1]); row[1] = make_float2(dmean[2], dcol[0]);
        row[2] = make_float2(dcol[1], dcol[2]);   row[3] = make_float2(dop, dsc[0]);
        row[4] = make_float2(dsc[1], dsc[2]);     row[5] = make_float2(drot[0], drot[1]);
        row[6] = make_float2(drot[2], drot[3]);
        return;
    }
    if (out.dL_dmeans3D) { out.dL_dmeans3D[3 * g] = dmean[0]; out.dL_dmeans3D[3 * g + 1] = dmean[1]; out.dL_dmeans3D[3 * g + 2] = dmean[2]; }
    if (out.dL_dcolors) { out.dL_dcolors[3 * g] = dcol[0]; out.dL_dcolors[3 * g + 1] = dcol[1]; out.dL_dcolors[3 * g + 2] = dcol[2]; }
    if (out.dL_dopacities) out.dL_dopacities[g] = dop;
    if (out.dL_dscales) { out.dL_dscales[3 * g] = dsc[0]; out.dL_dscales[3 * g + 1] = dsc[1]; out.dL_dscales[3 * g + 2] = dsc[2]; }
    if (out.dL_drotations) st_row4(out.dL_drotations, (size_t)g, make_float4(drot[0], drot[1], drot[2], drot[3]));
    if (out.dL_dcov3D) {
#pragma unroll
        for (int k = 0; k < 6; k++) out.dL_dcov3D[6 * (size_t)g + k] = dcov[k];
    }
}

// One thread per Gaussian.  With an exchange (ex.n_ex > 0: the packed [P,14] rows are one rank's share of a
// frame-sharded step and live in symmetric memory) the first ex.n_ex CTAs of the launch do not compute: they sum the rows
// over the ranks chunk by chunk while the other CTAs are still producing the later chunks (collective.cuh), so the
// launch ends with the all-reduced buffer in place and most of the transfer hidden under the computation.
// RAGGED: grid (ceil(max_v P_v / 128), n_views), thread i of view v handles row off_v + i for i < P_v; never an exchange.
template <bool RAGGED>
__global__ void __launch_bounds__(256,2) preprocess_backward_kernel(DevSettings s, PreInputs in,
                                                                  const int32_t* __restrict__ radii, GeomView geo,
                                                                  const float4* __restrict__ acc, BwdOutputs out,
                                                                  ExchangeArgs ex)
{
    pdl_prologue();
    if (RAGGED) {
        const int v = blockIdx.y, lo = s.rows.off[v];
        const int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < s.rows.off[v + 1] - lo) gaussian_backward<true>(s, in, radii, geo, acc, out, lo + i, v);
        return;
    }
    if (ex.n_ex > 0 && (int)blockIdx.x < ex.n_ex) {
        exchange_role(ex);
        return;
    }
    const int cta = (int)blockIdx.x - ex.n_ex;
    const int g = cta * blockDim.x + threadIdx.x;
    if (g < in.P) gaussian_backward<false>(s, in, radii, geo, acc, out, g, 0);
    if (ex.n_ex > 0) {
        // device-scope only: a system-scope fence in each of the ~P/128 CTAs cost 100 us per launch.  The chain to the
        // peers is closed by the coordinator CTA: it acquires the chunk's count (device scope), fences at system scope
        // once per chunk and only then raises the chunk's flag in the peers' pads.
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) atomicAdd(ex.state + 2 + cta / ex.chunk_ctas, 1u);
    }
}

cudaError_t launch_preprocess_backward(const DevSettings& s, const PreInputs& in, const int32_t* radii, GeomView g,
                                       const float4* acc, BwdOutputs out, ExchangeArgs ex, cudaStream_t st)
{
    if (in.P <= 0) return cudaSuccess;
    count_launch();
    if (s.ragged) {
        const int Pmax = max_view_rows(s, in.P);
        return launch_pdl(preprocess_backward_kernel<true>, dim3((Pmax + 127) / 128, s.n_views), dim3(128), st, s, in,
                          radii, g, acc, out, ExchangeArgs{});
    }
    const int n_compute = (in.P + 127) / 128;
    return launch_pdl(preprocess_backward_kernel<false>, dim3(n_compute + ex.n_ex), dim3(128), st, s, in, radii, g, acc,
                      out, ex);
}

// Densification statistic at the rasterizer boundary (scene/gaussian_model.py:1298-1314 `training_statis`, called
// once per view, pipeline/train.py:559-565): per Gaussian, over the views of a step,
//   stats[g][0] = sum_v [radii[v][g] > 0] * |dL/dmeans2D[v][g][0:2]|,   stats[g][1] = sum_v [radii[v][g] > 0].
// One stream pass (16 B per (view, Gaussian) in, 8 B per Gaussian out) instead of a masked gather, a norm and a
// masked scatter-add per view.
__global__ void __launch_bounds__(256) densify_stats_kernel(int n_views, int P, const float* __restrict__ dm2d,
                                                            const int32_t* __restrict__ radii,
                                                            float* __restrict__ stats, long long stride, int accumulate)
{
    pdl_prologue();
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= P) return;
    float norm_sum = 0.f, count = 0.f;
    for (int v = 0; v < n_views; v++) {
        const size_t gv = (size_t)v * P + g;
        if (__ldg(radii + gv) > 0) {
            const float x = __ldg(dm2d + 3 * gv), y = __ldg(dm2d + 3 * gv + 1);
            norm_sum += sqrtf(x * x + y * y);
            count += 1.f;
        }
    }
    float* o = stats + (size_t)g * stride;
    if (accumulate) {
        o[0] += norm_sum;
        o[1] += count;
    } else {
        o[0] = norm_sum;
        o[1] = count;
    }
}

cudaError_t launch_densify_stats(int n_views, int P, const float* dm2d, const int32_t* radii, float* stats,
                                 long long stride, bool accumulate, cudaStream_t st)
{
    if (P <= 0) return cudaSuccess;
    count_launch();
    return launch_pdl(densify_stats_kernel, dim3((P + 255) / 256), dim3(256), st, n_views, P, dm2d, radii, stats, stride,
                      accumulate ? 1 : 0);
}

}  // namespace gsvc
