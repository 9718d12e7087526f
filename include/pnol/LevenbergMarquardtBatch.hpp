/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * LevenbergMarquardtBatch.hpp -- LevMarqBatch: many small independent least-squares fits in one call (pnol_lm_batch).
 * The objective's residual rows hold the problems back to back: problem b owns rows [rowOffsets[b], rowOffsets[b+1]) and row b of X.
 * Every problem gets, bit for bit, what LevMarq::findMin gives on that problem alone with the reference's dense helpers (the shim's
 * sequential sums and LU), not the single-problem path's tensor-core sums. setParams is LevMarq's; the Jacobian mode comes from
 * pnol::Runtime::jacobianMode() (PNOL_JAC_ANALYTIC: the model's own derivative, every other mode the forward difference with dXGrad).
 * n is 1 .. 64. Nothing is printed: `verbose` is kept for the signature only.
 */
#ifndef PNOL_LEVENBERGMARQUARDTBATCH_HPP_
#define PNOL_LEVENBERGMARQUARDTBATCH_HPP_

#include <vector>

#include "LevenbergMarquardtMPI.hpp"

class LevMarqBatch : public MultiAlgorithm {
  private:
	double lambda0;
	double dXGrad;
	double xMinDiff;
	int maxIter;
	double lambdaFactor;
	int verbose;

  public:
	/* rowOffsets: B + 1 non-decreasing row offsets within [0, rows of the objective]; X: B vectors of one length n (in/out); reports:
	 * resized to B, per problem iterations (the reference's counter), stopped, chiSq and lambda (accepted / rejected / xdiff2Norm are
	 * not kept by the batched kernel and stay 0). Throws pnol::Error as LevMarq::findMin does. */
	void findMin( const vector <long long> & rowOffsets, vector <vector <double> > & X, vector <pnol::LMReport> & reports );
	/* all rows as one problem (B = 1): F0 / FOpt pre-sized to the rows, as LevMarq::findMin takes them */
	void findMin( vector <double> & X, vector <double> & F0, vector <double> & FOpt );

	void setParams( double lambda0In, double lambdaFactorIn, double dXGradIn, double maxIterIn, double xMinDiffIn, int verboseIn )
	{  maxIter = maxIterIn; xMinDiff = xMinDiffIn; verbose = verboseIn; dXGrad = dXGradIn; lambda0 = lambda0In; lambdaFactor = lambdaFactorIn; }

	LevMarqBatch()
	{
		dXGrad = 1e-7;
		lambda0 = 0.001;
		maxIter = 10000;
		xMinDiff = 1e-7;
		verbose = 1;
		lambdaFactor = 10;
	}
	~LevMarqBatch(){}
};

#endif
