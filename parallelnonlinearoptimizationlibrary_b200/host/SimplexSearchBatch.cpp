/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
// SimplexSearchBatch.cpp -- SimplexSearchBatch::findMin: the whole batch of starts is one pnol_simplex_batch call.
#include "pnol/SimplexSearchBatch.hpp"

#include <cstring>

using std::vector;

// Weak reference, as BFGSBatch.cpp references pnol_bfgs_batch: a C-ABI implementation without pnol_simplex_batch (the CPU stand-in of
// the host-logic tests, programs built with it) still links, and findMin fails there with PNOL_ERR_NO_FUNCTOR.
extern "C" int pnol_simplex_batch( pnol_ctx *, const pnol_functor *, long long, int, double *, const pnol_simplex_params *,
		const pnol_stream_desc *, uint64_t, double *, double *, int *, int *, long long * ) __attribute__(( weak ));

void SimplexSearchBatch::run( long long B, int n, double * X, vector <pnol::SimplexReport> & reports )
{
	if( !pnol_simplex_batch )
		throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "SimplexSearchBatch::findMin: batched simplex search (pnol_simplex_batch) is not provided by the "
				"C-ABI implementation this program is linked against" );
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = objPtr->deviceFunctor();
	if( !f ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "SimplexSearchBatch::findMin: the objective has no device functor (no CPU fallback)" );
	pnol_simplex_params prm;
	prm.alpha = alpha; prm.gamma = gamma; prm.rho = rho; prm.sigma = sigma; prm.max_iter = maxIter;
	prm.init_rand_max = initRandMax; prm.x_min_diff = xMinDiff;
	const pnol_stream_desc stream = rt.defaultStream( 1.0 );
	vector <double> f0( (size_t) B ), fOpt( (size_t) B );
	vector <int> iters( (size_t) B ), stop( (size_t) B );
	vector <long long> evals( (size_t) B );
	rt.check( pnol_simplex_batch( rt.ctx(), f, B, n, X, &prm, &stream, 0, f0.data(), fOpt.data(), iters.data(), stop.data(), evals.data() ) );
	streamPos_ = (unsigned long long) B * (unsigned long long) n * (unsigned long long) n;
	reports.assign( (size_t) B, pnol::SimplexReport() );
	long long total = 0;
	for( long long b = 0; b < B; b++ )
	{
		reports[b].f0 = f0[b];
		reports[b].fOpt = fOpt[b];
		reports[b].iterations = iters[b];
		reports[b].stop = stop[b];
		reports[b].evaluations = evals[b];
		total += evals[b];
	}
	objPtr->noteDeviceEvaluations( total );
}

void SimplexSearchBatch::findMin( vector <vector <double> > & X, vector <pnol::SimplexReport> & reports )
{
	const long long B = (long long) X.size();
	const int n = B > 0 ? (int) X[0].size() : 1;
	vector <double> Xflat( (size_t) B * n );
	for( long long b = 0; b < B; b++ )
	{
		if( (int) X[b].size() != n ) throw pnol::Error( PNOL_ERR_INVALID, "SimplexSearchBatch::findMin: every start needs the same number of parameters" );
		memcpy( Xflat.data() + (size_t) b * n, X[b].data(), (size_t) n * sizeof(double) );
	}
	run( B, n, Xflat.data(), reports );
	for( long long b = 0; b < B; b++ ) memcpy( X[b].data(), Xflat.data() + (size_t) b * n, (size_t) n * sizeof(double) );
}

void SimplexSearchBatch::findMin( vector <double> & X, double & f0, double & fOpt )
{
	vector <pnol::SimplexReport> reports;
	run( 1, (int) X.size(), X.data(), reports );
	f0 = reports[0].f0;
	fOpt = reports[0].fOpt;
}
