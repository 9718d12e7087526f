/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
// BFGSBatch.cpp -- BFGSBatch::findMin: the whole batch of starts is one pnol_bfgs_batch call.
#include "pnol/BFGSBatch.hpp"

#include <cstring>

// Weak reference, as PNOL_Objective.cpp references the analytic derivatives: a C-ABI implementation without pnol_bfgs_batch (the CPU
// stand-in of the host-logic tests, programs built with it) still links, and findMin fails there with PNOL_ERR_NO_FUNCTOR.
extern "C" int pnol_bfgs_batch( pnol_ctx *, const pnol_functor *, long long, int, double *, const pnol_bfgs_params *, int, double *, double *,
		int *, int * ) __attribute__(( weak ));

void BFGSBatch::run( long long B, int n, double * X, vector <pnol::BFGSReport> & reports )
{
	if( !pnol_bfgs_batch )
		throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "BFGSBatch::findMin: batched BFGS (pnol_bfgs_batch) is not provided by the C-ABI "
				"implementation this program is linked against" );
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = objPtr->deviceFunctor();
	if( !f ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "BFGSBatch::findMin: the objective has no device functor (no CPU fallback)" );
	pnol_bfgs_params prm;
	prm.c1 = c1; prm.c2 = c2; prm.dalpha = dalpha; prm.alpha_guess = alphaGuess; prm.max_iter_ls = maxIterLineSearch;
	prm.dx_grad = dXGrad; prm.dx_hess = dXHess; prm.max_iter = maxIter; prm.x_min_diff = xMinDiff; prm.min_grad_2norm = minGrad2Norm;
	prm.init_hess_fd = initHessFD ? 1 : 0;
	const int flags = ( rt.analyticGradient() ? PNOL_BFGS_ANALYTIC_GRADIENT : 0 ) | ( rt.analyticSlope() ? PNOL_BFGS_ANALYTIC_SLOPE : 0 ) |
			( rt.analyticHessian() ? PNOL_BFGS_ANALYTIC_HESSIAN : 0 );
	vector <double> f0( (size_t) B ), fOpt( (size_t) B );
	vector <int> iters( (size_t) B ), stop( (size_t) B );
	rt.check( pnol_bfgs_batch( rt.ctx(), f, B, n, X, &prm, flags, f0.data(), fOpt.data(), iters.data(), stop.data() ) );
	reports.assign( (size_t) B, pnol::BFGSReport() );
	for( long long b = 0; b < B; b++ )
	{
		reports[b].f0 = f0[b];
		reports[b].fOpt = fOpt[b];
		reports[b].iterations = iters[b];
		reports[b].stop = stop[b];
	}
}

void BFGSBatch::findMin( vector <vector <double> > & X, vector <pnol::BFGSReport> & reports )
{
	const long long B = (long long) X.size();
	const int n = B > 0 ? (int) X[0].size() : 1;
	vector <double> Xflat( (size_t) B * n );
	for( long long b = 0; b < B; b++ )
	{
		if( (int) X[b].size() != n ) throw pnol::Error( PNOL_ERR_INVALID, "BFGSBatch::findMin: every start needs the same number of parameters" );
		memcpy( Xflat.data() + (size_t) b * n, X[b].data(), (size_t) n * sizeof(double) );
	}
	run( B, n, Xflat.data(), reports );
	for( long long b = 0; b < B; b++ ) memcpy( X[b].data(), Xflat.data() + (size_t) b * n, (size_t) n * sizeof(double) );
}

void BFGSBatch::findMin( vector <double> & X, double & f0, double & fOpt )
{
	vector <pnol::BFGSReport> reports;
	run( 1, (int) X.size(), X.data(), reports );
	f0 = reports[0].f0;
	fOpt = reports[0].fOpt;
}
