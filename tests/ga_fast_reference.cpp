// TEST INFRASTRUCTURE -- an O(Npop log Npop) restatement of oracle_ga (oracle/pnol_oracle.cpp, GeneticAlgorithmMPI::findMinBnd at
// P = 1), so that GA generations can be checked bit for bit at populations the O(Npop^2 n) oracle cannot reach.
//
// It draws from the oracle's own stream (oracle_stream_uniform, libpnol_oracle.so) and evaluates with the oracle's own objective code
// (oracle/oracle_objectives.h) or a C function pointer. Everything is the literal algorithm except two parts:
//   * popSort is a stable sort with <. The reference's repeated first-minimum extraction with a 2 FMax sentinel is that sort exactly
//     when every F is finite and FMax > 0; otherwise this restatement refuses (returns -3);
//   * checkIndenticalChildAndReplace looks rows up by content instead of comparing all pairs. Its loop, for i ascending and k > i
//     ascending, replaces row i with n draws whenever row i == row k, and goes on comparing the NEW row i with the rows after k. Step
//     i rewrites only row i and reads only rows k > i, which are still as they were before the loop. So: row i is replaced iff a
//     later original row equals it, the new row is looked up among the original rows after the match, and so on. "Equal" is the
//     reference's per-gene ==: -0 and +0 hash alike, and a row holding a NaN equals no row. The first call, on the all-zero
//     XpopNew, is the same lookup with every row in one group.
// tests/test_ga_fast_reference.py checks every output against oracle_ga bit for bit, and that the check notices a wrong tie order or
// a missed duplicate.
//
// Built by tests/ga_fast_reference.py: g++ -O2 -ffp-contract=off, linked against oracle/libpnol_oracle.so.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <numeric>
#include <utility>
#include <vector>

#include "oracle_objectives.h"
#include "my_ga_objectives.hpp"

using std::vector;

extern "C" double oracle_stream_uniform(uint64_t seed, uint64_t k, double scale);

namespace {

struct Stream {
	const double * values; uint64_t n_values; uint64_t seed; double scale; uint64_t pos; int exhausted;
	double next()
	{
		if (values) {
			if (pos >= n_values) { exhausted = 1; pos++; return 0.0; }
			return values[pos++];
		}
		return oracle_stream_uniform(seed, pos++, scale);
	}
};

// sensitivity switches of the self-test (tests/test_ga_fast_reference.py): a deliberately wrong reference must fail the comparison
int g_flip_ties = 0;          // ties sorted by descending row
int g_miss_duplicate = 0;     // the first replacement of a duplicate row is skipped

// checkPopulationBoundsAndReplace, Source/GeneticAlgorithm.cpp:347-365 (literal)
void check_bounds(double * X, long long Npop, int n, const double * Xlb, const double * Xub, unsigned char * ind, Stream & st)
{
	for (long long i = 0; i < Npop; i++)
		for (int j = 0; j < n; j++)
			if (X[i * n + j] > Xub[j] || X[i * n + j] < Xlb[j]) {
				X[i * n + j] = Xlb[j] + (Xub[j] - Xlb[j]) * st.next();
				if (ind) ind[i] = 1;
			}
}

uint64_t row_hash(const double * r, int n)
{
	uint64_t h = 0x243F6A8885A308D3ULL;
	for (int j = 0; j < n; j++) {
		double v = r[j];
		if (v == 0.0) v = 0.0;                // -0 == +0
		uint64_t b; memcpy(&b, &v, 8);
		h = (h ^ b) * 0x100000001B3ULL;
		h ^= h >> 29;
	}
	return h;
}

bool has_nan(const double * r, int n)
{
	for (int j = 0; j < n; j++) if (r[j] != r[j]) return true;
	return false;
}

bool rows_equal(const double * a, const double * b, int n)
{
	for (int j = 0; j < n; j++) if (!(a[j] == b[j])) return false;
	return true;
}

// checkIndenticalChildAndReplace, Source/GeneticAlgorithm.cpp:313-344, through a table of (hash, row) of the original rows
void check_identical(double * X, long long Npop, int n, const double * Xlb, const double * Xub, unsigned char * ind, Stream & st)
{
	vector<std::pair<uint64_t, long long>> tab;
	tab.reserve((size_t) Npop);
	for (long long r = 0; r < Npop; r++)
		if (!has_nan(X + r * n, n)) tab.push_back(std::make_pair(row_hash(X + r * n, n), r));
	std::sort(tab.begin(), tab.end());
	// smallest original row > k equal to `row`, or -1
	auto next_equal = [&](const double * row, long long k) -> long long {
		if (has_nan(row, n)) return -1;
		const uint64_t h = row_hash(row, n);
		auto it = std::lower_bound(tab.begin(), tab.end(), std::make_pair(h, k + 1));
		for (; it != tab.end() && it->first == h; ++it)
			if (rows_equal(row, X + it->second * n, n)) return it->second;
		return -1;
	};
	int skipped = 0;
	for (long long i = 0; i < Npop; i++) {
		double * row = X + i * n;
		for (long long k = next_equal(row, i); k >= 0; k = next_equal(row, k)) {
			if (g_miss_duplicate && !skipped) { skipped = 1; break; }
			for (int j = 0; j < n; j++) row[j] = Xlb[j] + (Xub[j] - Xlb[j]) * st.next();
			if (ind) ind[i] = 1;
		}
	}
}

// popSort, Source/GeneticAlgorithm.cpp:370-412, as the stable sort it is when every F is finite and FMax > 0 (else: false)
bool pop_sort(double * X, double * F, long long Npop, int n)
{
	double FMax = F[0];
	for (long long i = 0; i < Npop; i++) {
		if (!isfinite(F[i])) return false;
		if (F[i] > FMax) FMax = F[i];
	}
	if (!(FMax > 0)) return false;
	vector<long long> idx((size_t) Npop);
	std::iota(idx.begin(), idx.end(), 0LL);
	if (g_flip_ties)
		std::stable_sort(idx.begin(), idx.end(), [&](long long a, long long b) { return F[a] < F[b] || (!(F[b] < F[a]) && a > b); });
	else
		std::stable_sort(idx.begin(), idx.end(), [&](long long a, long long b) { return F[a] < F[b]; });
	vector<double> Xt((size_t) Npop * n), Ft((size_t) Npop);
	for (long long k = 0; k < Npop; k++) {
		memcpy(&Xt[(size_t) k * n], X + idx[k] * n, (size_t) n * sizeof(double));
		Ft[k] = F[idx[k]];
	}
	memcpy(X, Xt.data(), Xt.size() * sizeof(double));
	memcpy(F, Ft.data(), Ft.size() * sizeof(double));
	return true;
}

} // namespace

extern "C" {

// the test objectives of tests/user_functor/my_ga_objectives.hpp as C functions (objective pointers of ga_fast and oracle_ga_fn)
double ga_fast_quantized(const double * x, int n) { return QuantizedFunctor::eval(pnol::FunctorParams{}, x, n); }
double ga_fast_signed_zero(const double * x, int n) { return SignedZeroFunctor::eval(pnol::FunctorParams{}, x, n); }

void ga_fast_set_faults(int flip_ties, int miss_duplicate) { g_flip_ties = flip_ties; g_miss_duplicate = miss_duplicate; }

// called with the sorted start population (iter 0, parent indices all 0) and after every completed generation with its outputs: the
// sorted population, the parent indices and the stream position
typedef void (*ga_fast_generation_cb)(int iter, const double * Xpop, const double * F, const int * cross_idx, const int * mut_idx,
                                      const int * elite_idx, uint64_t pos);

// oracle_ga_fn's arguments and results (oracle/pnol_oracle.cpp), plus on_generation (may be NULL). Returns the generations
// completed, -1 for invalid fractions, -2 for an exhausted explicit stream, -3 where popSort is not a stable sort (max F <= 0 or a
// non-finite F; the GPU library refuses those populations as well).
int ga_fast(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
            double (*fn)(const double *, int), double * X, const double * Xlb, const double * Xub, int Nparam, int Npop,
            int maxGenerations, double eliteFrac, double crossFrac, double eliteMutationFrac, double mutationSize,
            double eliteMutationSize, double NstaticGenerations, int stopAfter, const double * values, uint64_t n_values,
            uint64_t seed, double scale, double * f0_out, double * fOpt_out, double * Xpop_out, double * F_out, int * cross_idx,
            int * mut_idx, int * elite_idx, uint64_t * stream_pos_out, ga_fast_generation_cb on_generation)
{
	OFunctor fobj = {kind, scalars, ints, cols, m};
	auto objective = [&](const double * x) { return fn ? fn(x, Nparam) : o_scalar(fobj, x, Nparam); };
	Stream st = {values, n_values, seed, scale, 0, 0};
	size_t NN = (size_t) Npop * Nparam;
	vector<double> Xpop(NN, 0.0), XpopNew(NN, 0.0), F(Npop, 0), Fnew(Npop, 0), fitness(Npop, 0);
	vector<unsigned char> ind(Npop, 1);

	int Nelite = (int) ceil(eliteFrac * Npop);
	int NeliteMut = (int) ceil(eliteMutationFrac * Npop);
	int Ncross = (int) ceil(crossFrac * Npop);
	int Nrand = Npop - Nelite - NeliteMut - Ncross;
	if (Nrand <= 0) return -1;
	// parent indices of the generation in progress (the callback sees every generation's; the outputs hold the last one's)
	vector<int> cross((size_t) Ncross * Nparam), mut(Nrand), elite((size_t) NeliteMut * Nparam);

	for (int i = 0; i < Nparam; i++) Xpop[i] = X[i];
	for (int i = 1; i < Npop; i++)
		for (int j = 0; j < Nparam; j++)
			Xpop[(size_t) i * Nparam + j] = Xpop[j] + ((Xub[j] - Xlb[j]) * st.next() + Xlb[j]);
	check_identical(XpopNew.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);      // (sic: XpopNew, as the reference)
	check_bounds(Xpop.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);
	for (int i = 0; i < Npop; i++) if (ind[i]) F[i] = objective(&Xpop[(size_t) i * Nparam]);
	double f0 = F[0];
	if (!pop_sort(Xpop.data(), F.data(), Npop, Nparam)) return -3;
	if (on_generation) on_generation(0, Xpop.data(), F.data(), cross.data(), mut.data(), elite.data(), st.pos);

	double FbestPrev = F[0];
	int Nstatic = 0;
	int iter = 0;
	while (iter < maxGenerations && (stopAfter < 0 || iter < stopAfter)) {
		for (int k = 0; k < Npop; k++) fitness[k] = pow(F[Npop - 1] - F[k], 2);
		double maxFitness = fitness[0];
		for (int k = 0; k < Npop; k++) ind[k] = 1;
		int popIdx = 0;
		for (int k = 0; k < Nelite; k++) {
			for (int i = 0; i < Nparam; i++) XpopNew[(size_t) popIdx * Nparam + i] = Xpop[(size_t) popIdx * Nparam + i];
			Fnew[popIdx] = F[popIdx];
			ind[popIdx] = 0;
			popIdx++;
		}
		for (int k = 0; k < Ncross; k++) {
			for (int i = 0; i < Nparam; i++) {
				int index = 0;
				while (index == 0) {
					int randomIndex = (int) round(st.next() * Npop);
					double selectValue = st.next();
					if (st.exhausted) return -2;
					if (randomIndex < Npop && selectValue <= fitness[randomIndex] / maxFitness) index = randomIndex;
				}
				XpopNew[(size_t) popIdx * Nparam + i] = Xpop[(size_t) index * Nparam + i];
				cross[(size_t) k * Nparam + i] = index;
			}
			popIdx++;
		}
		double spreadRatio = mutationSize * (maxGenerations - iter) / maxGenerations;
		for (int k = 0; k < Nrand; k++) {
			int index = 0;
			while (index == 0) {      // the reference's loop over j re-enters this while only for j = 0
				int randomIndex = (int) round(st.next() * Npop);
				double selectValue = st.next();
				if (st.exhausted) return -2;
				if (randomIndex < Npop && selectValue <= fitness[randomIndex] / maxFitness) index = randomIndex;
			}
			mut[k] = index;
			for (int j = 0; j < Nparam; j++) {
				double mutation = spreadRatio * (Xub[j] - Xlb[j]) * st.next();
				XpopNew[(size_t) popIdx * Nparam + j] = Xpop[(size_t) index * Nparam + j] + mutation;
			}
			popIdx++;
		}
		for (int k = 0; k < NeliteMut; k++) {
			for (int j = 0; j < Nparam; j++) {
				int randomEliteIdx = (int) round(st.next() * Nelite);
				double mutation = eliteMutationSize * (Xub[j] - Xlb[j]) * st.next();
				XpopNew[(size_t) popIdx * Nparam + j] = Xpop[(size_t) randomEliteIdx * Nparam + j] + mutation;
				elite[(size_t) k * Nparam + j] = randomEliteIdx;
			}
			popIdx++;
		}
		check_identical(XpopNew.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);
		check_bounds(XpopNew.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);
		for (int i = 0; i < Npop; i++) if (ind[i]) Fnew[i] = objective(&XpopNew[(size_t) i * Nparam]);
		if (!pop_sort(XpopNew.data(), Fnew.data(), Npop, Nparam)) return -3;
		std::swap(F, Fnew);
		std::swap(Xpop, XpopNew);
		if (on_generation) on_generation(iter + 1, Xpop.data(), F.data(), cross.data(), mut.data(), elite.data(), st.pos);
		double Fbest = F[0];
		if (Fbest == FbestPrev) Nstatic++; else Nstatic = 0;
		if (Nstatic > NstaticGenerations) break;
		FbestPrev = Fbest;
		iter++;
	}
	if (st.exhausted) return -2;
	if (fOpt_out) *fOpt_out = F[0];
	for (int i = 0; i < Nparam; i++) X[i] = Xpop[i];
	if (f0_out) *f0_out = f0;
	if (Xpop_out) memcpy(Xpop_out, Xpop.data(), NN * sizeof(double));
	if (F_out) memcpy(F_out, F.data(), (size_t) Npop * sizeof(double));
	if (cross_idx) memcpy(cross_idx, cross.data(), cross.size() * sizeof(int));
	if (mut_idx) memcpy(mut_idx, mut.data(), mut.size() * sizeof(int));
	if (elite_idx) memcpy(elite_idx, elite.data(), elite.size() * sizeof(int));
	if (stream_pos_out) *stream_pos_out = st.pos;
	return iter;
}

} // extern "C"
