/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
// LevenbergMarquardtBatch.cpp -- LevMarqBatch::findMin: the whole batch is one pnol_lm_batch call.
#include "pnol/LevenbergMarquardtBatch.hpp"

#include <cstring>
#include <string>

// Weak reference, as PNOL_Objective.cpp references the analytic derivatives: a C-ABI implementation without pnol_lm_batch (the CPU
// stand-in of the host-logic tests, programs built with it) still links, and findMin fails there with PNOL_ERR_NO_FUNCTOR.
extern "C" int pnol_lm_batch( pnol_ctx *, const pnol_functor *, const long long *, long long, int, double *, const double *, double, double,
		double, int, int, double *, double *, int *, int *, double * ) __attribute__(( weak ));

namespace {
void runBatch( MultiObjective * obj, const long long * rowOffsets, long long B, int n, double * X, double lambda0, double lambdaFactor,
		double dXGrad, int maxIter, double xMinDiff, vector <double> & chi, vector <double> & lam, vector <int> & iters, vector <int> & stopped,
		double * Fout )
{
	if( !pnol_lm_batch )
		throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "LevMarqBatch::findMin: batched Levenberg-Marquardt (pnol_lm_batch) is not provided by the "
				"C-ABI implementation this program is linked against" );
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = obj->requireFunctor( "LevMarqBatch::findMin" );
	const vector <double> dX( n > 0 ? n : 1, dXGrad );
	chi.assign( (size_t) B, 0.0 ); lam.assign( (size_t) B, 0.0 ); iters.assign( (size_t) B, 0 ); stopped.assign( (size_t) B, 0 );
	rt.check( pnol_lm_batch( rt.ctx(), f, rowOffsets, B, n, X, dX.data(), lambda0, lambdaFactor, xMinDiff, maxIter, rt.jacobianMode(),
			chi.data(), lam.data(), iters.data(), stopped.data(), Fout ) );
}
}

void LevMarqBatch::findMin( const vector <long long> & rowOffsets, vector <vector <double> > & X, vector <pnol::LMReport> & reports )
{
	const long long B = (long long) X.size();
	if( (long long) rowOffsets.size() != B + 1 )
		throw pnol::Error( PNOL_ERR_INVALID, "LevMarqBatch::findMin: rowOffsets must hold one entry more than X has problems" );
	const int n = B > 0 ? (int) X[0].size() : 1;
	vector <double> Xflat( (size_t) B * n );
	for( long long b = 0; b < B; b++ )
	{
		if( (int) X[b].size() != n ) throw pnol::Error( PNOL_ERR_INVALID, "LevMarqBatch::findMin: every problem needs the same number of parameters" );
		memcpy( Xflat.data() + (size_t) b * n, X[b].data(), (size_t) n * sizeof(double) );
	}
	vector <double> chi, lam;
	vector <int> iters, stopped;
	runBatch( mObjPtr, rowOffsets.data(), B, n, Xflat.data(), lambda0, lambdaFactor, dXGrad, maxIter, xMinDiff, chi, lam, iters, stopped, nullptr );
	reports.assign( (size_t) B, pnol::LMReport() );
	for( long long b = 0; b < B; b++ )
	{
		memcpy( X[b].data(), Xflat.data() + (size_t) b * n, (size_t) n * sizeof(double) );
		reports[b].iterations = iters[b];
		reports[b].stopped = stopped[b];
		reports[b].chiSq = chi[b];
		reports[b].lambda = lam[b];
	}
}

void LevMarqBatch::findMin( vector <double> & X, vector <double> & F0, vector <double> & FOpt )
{
	pnol_functor * f = mObjPtr->requireFunctor( "LevMarqBatch::findMin" );
	const long long m = pnol_functor_rows( f );
	if( (long long) F0.size() != m || (long long) FOpt.size() != m )
		throw pnol::Error( PNOL_ERR_INVALID, "LevMarqBatch::findMin: F0 / FOpt must be pre-sized to the number of residuals" );
	pnol::Runtime & rt = pnol::Runtime::instance();
	rt.check( pnol_residual_eval( rt.ctx(), f, X.data(), (int) X.size(), F0.data(), nullptr ) );   // F0 = F(X) as given (:42-49)
	const long long rowOffsets[2] = { 0, m };
	vector <double> chi, lam;
	vector <int> iters, stopped;
	runBatch( mObjPtr, rowOffsets, 1, (int) X.size(), X.data(), lambda0, lambdaFactor, dXGrad, maxIter, xMinDiff, chi, lam, iters, stopped, FOpt.data() );
}
