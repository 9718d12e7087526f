/*
 * pnol_math.h -- transcendental functions with ONE definition for host and device.
 *
 * FD derivatives amplify a 1-ulp difference in f by 1/h (SURVEY.md section 7, hard part 1), so an objective
 * that wants its device functor to agree with its host objEval to the last bit cannot call libm (glibc and
 * CUDA differ in the last ulp). These functions use only + - * / rint, explicit fma() and bit operations, are compiled
 * without implicit FMA contraction on both sides (nvcc -fmad=false, g++ -ffp-contract=off), and therefore return
 * identical bits on CPU and GPU. Accuracy is a few ulp -- they are not correctly rounded and make no such claim.
 */
#ifndef PNOL_MATH_H_
#define PNOL_MATH_H_

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define PNOL_HD __host__ __device__ __forceinline__
#else
#define PNOL_HD inline
#endif
/* unroll hint for the device compiler (gives it independent FP64 chains to interleave); the order of the operations on any
 * one value is unchanged, so results are the same bits with or without it */
#if defined(__CUDA_ARCH__)
#define PNOL_UNROLL(n) _Pragma(PNOL_STR_(unroll n))
#define PNOL_STR_(x) #x
#else
#define PNOL_UNROLL(n)
#endif

namespace pnol {

PNOL_HD double bits_to_double(uint64_t b)
{
#if defined(__CUDA_ARCH__)
	return __longlong_as_double((long long) b);
#else
	double d; memcpy(&d, &b, sizeof d); return d;
#endif
}

/* 2^k for -1022 <= k <= 1023 */
PNOL_HD double pow2i(int k) { return bits_to_double((uint64_t)(k + 1023) << 52); }

/* cos(2 pi x) without branches or table look-ups: exact reduction to r in [0, 1/4] (sign kept aside), the Taylor polynomial of
 * cos(theta) for theta = pi r in [0, pi/4] by Horner's rule with EXPLICIT fused multiply-adds, then the double-angle identity
 * cos(2 theta) = 2 cos^2(theta) - 1. fma() is correctly rounded on both sides (DFMA on the device, libm / the FMA unit on the
 * host), so host and device still agree bit for bit. Absolute error a few 1e-16 (the identity loses relative accuracy near the
 * zeros of the cosine, which an objective of the form x^2 - 10 cos(2 pi x) does not care about). 21 FP64 instructions per call and
 * 4 selects: the population sweep is FP64-issue bound on B200 (DESIGN.md section 5), the first version (sin / cos series chosen per
 * element, unfused Horner steps) cost 45. */
PNOL_HD double cos2pi(double x)
{
	double r = x - rint(x);                 /* exact, |r| <= 0.5 */
	r = fabs(r);
	const bool neg = r > 0.25;
	r = neg ? 0.5 - r : r;                  /* exact; cos(2 pi x) = -cos(2 pi (1/2 - r)) */
	const double t = 3.141592653589793 * r; /* theta in [0, pi/4] */
	const double t2 = t * t;
	double p = 4.7794773323873853e-14;      /*  1/16! */
	p = fma(p, t2, -1.1470745597729725e-11);/* -1/14! */
	p = fma(p, t2, 2.0876756987868100e-09); /*  1/12! */
	p = fma(p, t2, -2.7557319223985888e-07);/* -1/10! */
	p = fma(p, t2, 2.4801587301587302e-05); /*  1/8!  */
	p = fma(p, t2, -1.3888888888888889e-03);/* -1/6!  */
	p = fma(p, t2, 4.1666666666666664e-02); /*  1/4!  */
	p = fma(p, t2, -0.5);                   /* -1/2!  */
	const double c = fma(t2, p, 1.0);       /* cos(theta) */
	const double v = fma(c + c, c, -1.0);   /* cos(2 theta) */
	return neg ? -v : v;
}

/* sin(2 pi x), built as cos2pi is: exact reduction to a = |r| in [0, 1/4] with the sign of r kept aside (sin(2 pi (1/2 - a)) =
 * sin(2 pi a)), theta = pi a in [0, pi/4], the Taylor polynomials of sin(theta) and cos(theta) by Horner's rule with EXPLICIT fused
 * multiply-adds, then the double-angle identity sin(2 theta) = 2 sin(theta) cos(theta). No tables, same bits on host and device. Absolute
 * error a few 1e-16; an integer x (every |x| >= 2^52 included) gives +0. The derivative of the Rastrigin term (RastriginFunctor::partial). */
PNOL_HD double sin2pi(double x)
{
	const double r = x - rint(x);           /* exact, |r| <= 0.5 */
	const bool neg = r < 0;
	double a = fabs(r);
	a = a > 0.25 ? 0.5 - a : a;             /* exact */
	const double t = 3.141592653589793 * a; /* theta in [0, pi/4] */
	const double t2 = t * t;
	double s = 2.8114572543455206e-15;      /*  1/17! */
	s = fma(s, t2, -7.6471637318198164e-13);/* -1/15! */
	s = fma(s, t2, 1.6059043836821613e-10); /*  1/13! */
	s = fma(s, t2, -2.5052108385441720e-08);/* -1/11! */
	s = fma(s, t2, 2.7557319223985893e-06); /*  1/9!  */
	s = fma(s, t2, -1.9841269841269841e-04);/* -1/7!  */
	s = fma(s, t2, 8.3333333333333332e-03); /*  1/5!  */
	s = fma(s, t2, -1.6666666666666666e-01);/* -1/3!  */
	const double sn = fma(t * t2, s, t);    /* sin(theta) */
	double p = 4.7794773323873853e-14;      /* cos(theta): the polynomial of cos2pi */
	p = fma(p, t2, -1.1470745597729725e-11);
	p = fma(p, t2, 2.0876756987868100e-09);
	p = fma(p, t2, -2.7557319223985888e-07);
	p = fma(p, t2, 2.4801587301587302e-05);
	p = fma(p, t2, -1.3888888888888889e-03);
	p = fma(p, t2, 4.1666666666666664e-02);
	p = fma(p, t2, -0.5);
	const double c = fma(t2, p, 1.0);
	const double v = (sn + sn) * c;         /* sin(2 theta) */
	return neg ? -v : v;
}

/* exp(x): k = rint(x log2 e), Cody-Waite reduction, degree-13 Taylor polynomial, scaling by 2^k in two steps */
PNOL_HD double exp_hd(double x)
{
	if (x != x) return x;
	if (x > 709.782712893384) return bits_to_double(0x7FF0000000000000ULL);
	if (x < -745.2) return 0.0;
	double kf = rint(x * 1.4426950408889634);
	double r = x - kf * 6.93147180369123816490e-01;      /* ln2 high part (low 21 bits zero): product exact */
	r = r - kf * 1.90821492927058770002e-10;             /* ln2 low part */
	double p = 1.6059043836821613e-10;                   /* 1/13! */
	p = p * r + 2.0876756987868100e-09;                  /* 1/12! */
	p = p * r + 2.5052108385441720e-08;                  /* 1/11! */
	p = p * r + 2.7557319223985888e-07;                  /* 1/10! */
	p = p * r + 2.7557319223985893e-06;                  /* 1/9!  */
	p = p * r + 2.4801587301587302e-05;                  /* 1/8!  */
	p = p * r + 1.9841269841269841e-04;                  /* 1/7!  */
	p = p * r + 1.3888888888888889e-03;                  /* 1/6!  */
	p = p * r + 8.3333333333333332e-03;                  /* 1/5!  */
	p = p * r + 4.1666666666666664e-02;                  /* 1/4!  */
	p = p * r + 1.6666666666666666e-01;                  /* 1/3!  */
	p = p * r + 0.5;
	p = p * r + 1.0;
	p = p * r + 1.0;
	int k = (int) kf;
	int k1 = k / 2;
	int k2 = k - k1;
	return (p * pow2i(k1)) * pow2i(k2);
}

} // namespace pnol

#endif /* PNOL_MATH_H_ */
