/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root). */
/*
 * simplex_sort.hpp -- the permutation SimplexSearch's simplexSort (host/SimplexSearch.cpp, Source/SimplexSearch.cpp:272-326) applies,
 * in pieces that the G lanes of a group share (simplex_batch_kernel, device/functor_kernels.cuh) and that the host runs with G = 1
 * (simplex_sort_perm, which tests/test_simplex_batch_cpu.py checks against simplexSort itself).
 *
 * simplexSort makes N = n + 1 passes. Pass k scans `if (f[i] < f[c]) c = i` from the candidate c (1 at the first pass, then the
 * entry the previous pass took: it is never reset), copies row c and f[c] to place k and overwrites f[c] with S = 2 M, M the first
 * maximum of f found with `>`. Per pass that is:
 *   - f[c] NaN: take c;
 *   - otherwise, with m the minimum of the non-NaN entries: m < f[c] takes the first index whose value == m (-0 == +0), else c.
 * When 0 < M < inf and no entry is NaN ("the regime") S is above every entry and the N passes amount to a stable ascending order in
 * which index 1 goes first when it ties with the minimum: simplex_rank gives each entry its place independently. Outside the regime a
 * pass can take an entry again: the sorted f then holds sentinels S, and one row appears twice while another is lost.
 */
#ifndef PNOL_DEVICE_SIMPLEX_SORT_HPP_
#define PNOL_DEVICE_SIMPLEX_SORT_HPP_

#include "../functors.hpp"

namespace pnol {

constexpr int kSimplexNone = 0x7fffffff;      // index of an empty maximum / minimum

/* what a lane (entries lane, lane + G, ...) or a group knows of f: the first maximum M at iM and the first minimum m at im of the
 * non-NaN entries (kSimplexNone when there is none), and whether an entry is NaN. Combining is order-free: equal values (==, so -0
 * and +0 alike) go to the smaller index, and an empty side never wins. */
struct SimplexSortStats {
	double M, m;
	int iM, im, nan;
};

PNOL_HD SimplexSortStats simplex_stats_partial(const double * f, int N, int lane, int G)
{
	SimplexSortStats s;
	s.M = 0; s.m = 0; s.iM = kSimplexNone; s.im = kSimplexNone; s.nan = 0;
	for (int i = lane; i < N; i += G) {
		const double v = f[i];
		if (v != v) { s.nan = 1; continue; }
		if (s.iM == kSimplexNone || v > s.M) { s.M = v; s.iM = i; }
		if (s.im == kSimplexNone || v < s.m) { s.m = v; s.im = i; }
	}
	return s;
}

PNOL_HD SimplexSortStats simplex_stats_combine(SimplexSortStats a, const SimplexSortStats & b)
{
	if (b.iM != kSimplexNone && (a.iM == kSimplexNone || b.M > a.M || (b.M == a.M && b.iM < a.iM))) { a.M = b.M; a.iM = b.iM; }
	if (b.im != kSimplexNone && (a.im == kSimplexNone || b.m < a.m || (b.m == a.m && b.im < a.im))) { a.m = b.m; a.im = b.im; }
	a.nan |= b.nan;
	return a;
}

/* simplexSort's M: its running maximum starts from f[0], so a NaN f[0] stays */
PNOL_HD double simplex_first_max(const double * f, const SimplexSortStats & s) { return f[0] != f[0] ? f[0] : s.M; }

PNOL_HD bool simplex_in_regime(const double * f, const SimplexSortStats & s)
{
	const double M = simplex_first_max(f, s);
	return !s.nan && M > 0 && M < HUGE_VAL;
}

/* in the regime: the place of entry i (one_first: f[1] ties with the minimum, so index 1 goes before the other minima) */
PNOL_HD int simplex_rank(const double * f, int N, int i, bool one_first)
{
	const double v = f[i];
	const int ki = (i == 1 && one_first) ? -1 : i;
	int r = 0;
	for (int j = 0; j < N; j++) {
		const int kj = (j == 1 && one_first) ? -1 : j;
		r += (f[j] < v || (f[j] == v && kj < ki)) ? 1 : 0;
	}
	return r;
}

/* outside the regime: the entry a pass with candidate c takes, s the stats of the current f */
PNOL_HD int simplex_pass_take(const double * f, int c, const SimplexSortStats & s)
{
	const double fc = f[c];
	if (fc != fc) return c;
	return (s.im != kSimplexNone && s.m < fc) ? s.im : c;
}

/* simplexSort's permutation on the host, its stats gathered as G lanes would gather them: perm[k] is the entry place k receives,
 * and f is rewritten with the values simplexSort leaves in it (sentinels included). Returns true when the sort was in the regime. */
inline bool simplex_sort_perm(double * f, int N, int G, int * perm)
{
	SimplexSortStats s = simplex_stats_partial(f, N, 0, G);
	for (int l = 1; l < G; l++) s = simplex_stats_combine(s, simplex_stats_partial(f, N, l, G));
	const bool regime = simplex_in_regime(f, s);
	double ft[65];
	if (regime) {
		const bool one_first = f[1] == s.m;
		for (int i = 0; i < N; i++) { const int r = simplex_rank(f, N, i, one_first); perm[r] = i; ft[r] = f[i]; }
	} else {
		const double S = 2 * simplex_first_max(f, s);
		int c = 1;
		for (int k = 0; k < N; k++) {
			SimplexSortStats t = simplex_stats_partial(f, N, 0, G);
			for (int l = 1; l < G; l++) t = simplex_stats_combine(t, simplex_stats_partial(f, N, l, G));
			c = simplex_pass_take(f, c, t);
			perm[k] = c;
			ft[k] = f[c];
			f[c] = S;
		}
	}
	for (int k = 0; k < N; k++) f[k] = ft[k];
	return regime;
}

} // namespace pnol

#endif /* PNOL_DEVICE_SIMPLEX_SORT_HPP_ */
