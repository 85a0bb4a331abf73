// dct_kl_logit.cuh -- VATGenerator.kl_div_with_logit as a per-pixel op body: the stand-alone KL launches (dct_kl.cu) and the
// consistency step's JSD launch that carries the VAT KL (dct_jsd_vat.cu) run this same code.
#pragma once
#include "dct_common.cuh"

namespace dct {

// softmax statistics of one pixel (pair): on return x[c] = x[c] - max, e[c] = exp(x[c] - max); gives {1/Z, log Z}
template <int CM, class T>
__device__ __forceinline__ void softmax_stats(T (&x)[CM], T (&e)[CM], int C, T& inv, T& lZ) {
    T mx = x[0];
#pragma unroll
    for (int c = 1; c < CM; ++c)
        if (c < C) mx = vmax(mx, x[c]);
    T Z = vset<T>(0.0f);
#pragma unroll
    for (int c = 0; c < CM; ++c)
        if (c < C) {
            T d = vsub(x[c], mx);
            T ev = vexp(d);
            x[c] = d;
            e[c] = ev;
            Z = vadd(Z, ev);
        }
    inv = vdiv(vset<T>(1.0f), Z);
    lZ = vlog(Z);
}

// VATGenerator.kl_div_with_logit(q_logit, p_logit) -- generalframework/utils/AEGenerator.py:78-91
// (== KL_Divergence_2D_Logit(p_logit, y_logit=q_logit), loss.py:144-162).  in[0] = q_logit, in[1] = p_logit;
// out[0] = grad q_logit, out[1] = grad p_logit.
template <bool GRAD>
struct KlLogit {
    static constexpr int NIN = 2, NOUT = GRAD ? 2 : 0;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = GRAD;
    static constexpr bool HAS_MAP = true, USES_UP = GRAD, CHECKS_SIMPLEX = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[2][CM], int C, T g, float, bool&) {
        T eq[CM], ep[CM];
        T invq, lZq, invp, lZp;
        softmax_stats<CM, T>(x[0], eq, C, invq, lZq);
        softmax_stats<CM, T>(x[1], ep, C, invp, lZp);
        const T dl = vsub(lZp, lZq);
        T out = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                T q = vmul(eq[c], invq);
                T t = vadd(vsub(x[0][c], x[1][c]), dl);  // log q - log p = (dq - dp) + (lZp - lZq)
                eq[c] = q;
                x[0][c] = t;
                out = vfma(q, t, out);
            }
        if constexpr (GRAD) {
#pragma unroll
            for (int c = 0; c < CM; ++c)
                if (c < C) {
                    T q = eq[c];
                    x[0][c] = vmul(vmul(g, q), vsub(x[0][c], out));
                    x[1][c] = vmul(g, vsub(vmul(ep[c], invp), q));
                }
        }
        return out;
    }
};

}  // namespace dct
