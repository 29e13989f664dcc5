// Bit-exact device restatements of the glibc 2.39 libm entry points the reference's STATE path
// reaches (SURVEY Q13). The reference calls std::cos(float) / std::sin(float) on the same argument
// (games/bossfight/common_systems.cpp:80, games/caveflyer/common_systems.cpp:128, 361-364), which
// g++ -O3 fuses into one `sincosf` call (objdump -T of the compiled reference shows `sincosf` as the
// only trigonometric import); on x86-64 with FMA+AVX2 glibc dispatches that to `__sincosf_fma`
// (sysdeps/x86_64/fpu/multiarch/s_sincosf.c), i.e. sysdeps/ieee754/flt-32/s_sincosf.c compiled with
// -mfma -mavx2. The algorithm is the published ARM "optimized routines" sincosf: argument widened to
// double, quadrant reduction, two degree-7/8 polynomials evaluated in double, one rounding to float.
// Where the compiler contracted a*b+c into vfmadd* is visible in the library's disassembly; the
// sequence below reproduces it operation by operation (every fma() here is one vfmadd there), and
// tests/test_libm.py pins it against the host libm over many millions of arguments.
#pragma once
#include "pg2_common.cuh"

namespace pg2 {

struct SinCosTab {
    double sign[4];
    double hpi_inv, hpi;
    double c0, c1, s1, c2, s2, c3, s3, c4;
};

// __sincosf_table (sysdeps/ieee754/flt-32/s_sincosf_data.c), hex-float values as found in libm.so.6
PG2_DEV SinCosTab sincos_table(int which) {
    SinCosTab t;
    t.sign[0] = 1.0; t.sign[1] = -1.0; t.sign[2] = -1.0; t.sign[3] = 1.0;
    t.hpi_inv = 0x1.45f306dc9c883p+23;
    t.hpi = 0x1.921fb54442d18p+0;
    t.s1 = -0x1.555545995a603p-3;
    t.s2 = 0x1.1107605230bc4p-7;
    t.s3 = -0x1.994eb3774cf24p-13;
    if (which == 0) {
        t.c0 = 0x1p0; t.c1 = -0x1.ffffffd0c621cp-2; t.c2 = 0x1.55553e1068f19p-5;
        t.c3 = -0x1.6c087e89a359dp-10; t.c4 = 0x1.99343027bf8c3p-16;
    } else {
        t.c0 = -0x1p0; t.c1 = 0x1.ffffffd0c621cp-2; t.c2 = -0x1.55553e1068f19p-5;
        t.c3 = 0x1.6c087e89a359dp-10; t.c4 = -0x1.99343027bf8c3p-16;
    }
    return t;
}

// sincosf_poly: xs = x * sign, x2 = x * x (reduced argument)
PG2_DEV void sincosf_poly(double xs, double x2, int table, int n, float* sinp, float* cosp) {
    const SinCosTab p = sincos_table(table);
    double x3 = __dmul_rn(x2, xs);
    double x4 = __dmul_rn(x2, x2);
    double s1 = __fma_rn(x2, p.s3, p.s2);
    double c2 = __fma_rn(x2, p.c4, p.c3);
    double x5 = __dmul_rn(x2, x3);
    double x6 = __dmul_rn(x2, x4);
    double c1 = __fma_rn(x2, p.c1, p.c0);
    double s = __fma_rn(x3, p.s1, xs);
    double c = __fma_rn(x4, p.c2, c1);
    float sv = (float)__fma_rn(s1, x5, s);
    float cv = (float)__fma_rn(c2, x6, c);
    if (n & 1) { *cosp = sv; *sinp = cv; }
    else       { *sinp = sv; *cosp = cv; }
}

PG2_TU_LOCAL PG2_DEV_CALL void glibc_sincosf(float y, float* sinp, float* cosp) {
    uint32_t xi = __float_as_uint(y);
    uint32_t top = (xi >> 20) & 0x7ffu;                 // abstop12
    double x = (double)y;
    if (top < 0x3f4u) {                                 // |y| < pi/4
        double x2 = __dmul_rn(x, x);
        if (top < 0x398u) { *sinp = y; *cosp = 1.0f; return; }   // |y| < 2^-12
        sincosf_poly(x, x2, 0, 0, sinp, cosp);
    } else if (top < 0x42fu) {                          // |y| < 120: reduce_fast
        double r = __dmul_rn(x, 0x1.45f306dc9c883p+23);
        int n = (d2i(r) + 0x800000) >> 24;
        double xr = __fma_rn(-(double)n, 0x1.921fb54442d18p+0, x);
        double sgn = ((n & 3) == 1 || (n & 3) == 2) ? -1.0 : 1.0;
        sincosf_poly(__dmul_rn(xr, sgn), __dmul_rn(xr, xr), (n & 2) ? 1 : 0, n, sinp, cosp);
    } else if (top < 0x7f8u) {                          // reduce_large (__inv_pio4)
        const uint32_t inv_pio4[24] = {
            0xa2u, 0xa2f9u, 0xa2f983u, 0xa2f9836eu, 0xf9836e4eu, 0x836e4e44u, 0x6e4e4415u, 0x4e441529u,
            0x441529fcu, 0x1529fc27u, 0x29fc2757u, 0xfc2757d1u, 0x2757d1f5u, 0x57d1f534u, 0xd1f534ddu, 0xf534ddc0u,
            0x34ddc0dbu, 0xddc0db62u, 0xc0db6295u, 0xdb629599u, 0x6295993cu, 0x95993c43u, 0x993c4390u, 0x3c439041u };
        const uint32_t* arr = inv_pio4 + ((xi >> 26) & 15u);
        int shift = (int)((xi >> 23) & 7u);
        uint32_t m = ((xi & 0x7fffffu) | 0x800000u) << shift;
        uint64_t res0 = (uint64_t)(uint32_t)(m * arr[0]);
        uint64_t res1 = (uint64_t)m * arr[4];
        uint64_t res2 = (uint64_t)m * arr[8];
        res0 = (res2 >> 32) | (res0 << 32);
        res0 += res1;
        uint64_t nq = (res0 + (1ull << 61)) >> 62;
        res0 -= nq << 62;
        double xr = __dmul_rn((double)(int64_t)res0, 0x1.921fb54442d18p-62);
        int n = (int)nq;
        int ns = n + (int)(xi >> 31);
        double sgn = ((ns & 3) == 1 || (ns & 3) == 2) ? -1.0 : 1.0;
        sincosf_poly(__dmul_rn(xr, sgn), __dmul_rn(xr, xr), (ns & 2) ? 1 : 0, n, sinp, cosp);
    } else {                                            // inf / nan
        float v = __fsub_rn(y, y);
        *sinp = v; *cosp = v;
    }
}


// ---- atan2f --------------------------------------------------------------------------------------
// std::atan2(float, float) -> glibc 2.39 atan2f = wrapper around __ieee754_atan2f
// (sysdeps/ieee754/flt-32/e_atan2f.c) which calls __atanf (sysdeps/ieee754/flt-32/s_atanf.c): the
// classic fdlibm single-precision code, compiled for baseline x86-64 (scalar SSE, no FMA; atan2f is a
// plain function in libm.so.6, not an ifunc). Used by the jumper compass HUD (jumper.cpp:479).
PG2_DEV float glibc_atanf(float x) {
    const float atanhi[4] = { 4.6364760399e-01f, 7.8539812565e-01f, 9.8279368877e-01f, 1.5707962513e+00f };
    const float atanlo[4] = { 5.0121582440e-09f, 3.7748947079e-08f, 3.4473217170e-08f, 7.5497894159e-08f };
    const float aT[11] = { 3.3333334327e-01f, -2.0000000298e-01f, 1.4285714924e-01f, -1.1111110449e-01f, 9.0908870101e-02f,
                           -7.6918758452e-02f, 6.6610731184e-02f, -5.8335702866e-02f, 4.9768779427e-02f, -3.6531571299e-02f,
                           1.6285819933e-02f };
    int32_t hx = (int32_t)__float_as_uint(x);
    int32_t ix = hx & 0x7fffffff;
    int id;
    if (ix >= 0x4c000000) {                      // |x| >= 2^25
        if (ix > 0x7f800000) return __fadd_rn(x, x);
        return hx > 0 ? __fadd_rn(atanhi[3], atanlo[3]) : __fsub_rn(-atanhi[3], atanlo[3]);
    }
    if (ix < 0x3ee00000) {                       // |x| < 0.4375
        if (ix < 0x31000000) return x;           // |x| < 2^-29
        id = -1;
    } else {
        x = fabsf(x);
        if (ix < 0x3f980000) {
            if (ix < 0x3f300000) { id = 0; x = __fdiv_rn(__fsub_rn(__fmul_rn(2.0f, x), 1.0f), __fadd_rn(2.0f, x)); }
            else { id = 1; x = __fdiv_rn(__fsub_rn(x, 1.0f), __fadd_rn(x, 1.0f)); }
        } else {
            if (ix < 0x401c0000) { id = 2; x = __fdiv_rn(__fsub_rn(x, 1.5f), __fadd_rn(1.0f, __fmul_rn(1.5f, x))); }
            else { id = 3; x = __fdiv_rn(-1.0f, x); }
        }
    }
    float z = __fmul_rn(x, x);
    float w = __fmul_rn(z, z);
    float s1 = __fmul_rn(z, __fadd_rn(aT[0], __fmul_rn(w, __fadd_rn(aT[2], __fmul_rn(w, __fadd_rn(aT[4], __fmul_rn(w, __fadd_rn(aT[6],
               __fmul_rn(w, __fadd_rn(aT[8], __fmul_rn(w, aT[10])))))))))));
    float s2 = __fmul_rn(w, __fadd_rn(aT[1], __fmul_rn(w, __fadd_rn(aT[3], __fmul_rn(w, __fadd_rn(aT[5], __fmul_rn(w, __fadd_rn(aT[7],
               __fmul_rn(w, aT[9])))))))));
    if (id < 0) return __fsub_rn(x, __fmul_rn(x, __fadd_rn(s1, s2)));
    z = __fsub_rn(atanhi[id], __fsub_rn(__fsub_rn(__fmul_rn(x, __fadd_rn(s1, s2)), atanlo[id]), x));
    return hx < 0 ? -z : z;
}

PG2_TU_LOCAL PG2_DEV_CALL float glibc_atan2f(float y, float x) {
    const float tiny = 1.0e-30f, pi_o_4 = 7.8539818525e-01f, pi_o_2 = 1.5707963705e+00f, pi = 3.1415927410e+00f, pi_lo = -8.7422776573e-08f;
    int32_t hx = (int32_t)__float_as_uint(x), hy = (int32_t)__float_as_uint(y);
    int32_t ix = hx & 0x7fffffff, iy = hy & 0x7fffffff;
    if (ix > 0x7f800000 || iy > 0x7f800000) return __fadd_rn(x, y);
    if (hx == 0x3f800000) return glibc_atanf(y);
    int m = ((hy >> 31) & 1) | ((hx >> 30) & 2);
    if (iy == 0) {
        switch (m) {
        case 0: case 1: return y;
        case 2: return __fadd_rn(pi, tiny);
        default: return __fsub_rn(-pi, tiny);
        }
    }
    if (ix == 0) return hy < 0 ? __fsub_rn(-pi_o_2, tiny) : __fadd_rn(pi_o_2, tiny);
    if (ix == 0x7f800000) {
        if (iy == 0x7f800000) {
            switch (m) {
            case 0: return __fadd_rn(pi_o_4, tiny);
            case 1: return __fsub_rn(-pi_o_4, tiny);
            case 2: return __fadd_rn(__fmul_rn(3.0f, pi_o_4), tiny);
            default: return __fsub_rn(__fmul_rn(-3.0f, pi_o_4), tiny);
            }
        } else {
            switch (m) {
            case 0: return 0.0f;
            case 1: return -0.0f;
            case 2: return __fadd_rn(pi, tiny);
            default: return __fsub_rn(-pi, tiny);
            }
        }
    }
    if (iy == 0x7f800000) return hy < 0 ? __fsub_rn(-pi_o_2, tiny) : __fadd_rn(pi_o_2, tiny);
    int k = (iy - ix) >> 23;
    float z;
    if (k > 60) z = __fadd_rn(pi_o_2, __fmul_rn(0.5f, pi_lo));
    else if (hx < 0 && k < -60) z = 0.0f;
    else z = glibc_atanf(fabsf(__fdiv_rn(y, x)));
    switch (m) {
    case 0: return z;
    case 1: return __uint_as_float(__float_as_uint(z) ^ 0x80000000u);
    case 2: return __fsub_rn(pi, __fsub_rn(z, pi_lo));
    default: return __fsub_rn(__fsub_rn(z, pi_lo), pi);
    }
}

}  // namespace pg2
