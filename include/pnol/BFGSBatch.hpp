/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * BFGSBatch.hpp -- BFGSBatch: many independent BFGS minimisations of one objective (multiple starts) in one call (pnol_bfgs_batch).
 * Start b is X[b]; every start gets, bit for bit, what BFGS::findMin gives on that start alone with the reference's dense helpers
 * (sequential sums, the literal two-product inverse-Hessian update, matrixInverse's LU), not the GPU BFGS class's RANK2 / tensor-core
 * products, which agree with it to about 1e-9 only. setParams and the defaults are BFGS's; the derivative modes come from
 * pnol::Runtime::analyticGradient(), analyticSlope() and analyticHessian(). n is 1 .. 64. Nothing is printed: `verbose` is kept for
 * the signature only.
 */
#ifndef PNOL_BFGSBATCH_HPP_
#define PNOL_BFGSBATCH_HPP_

#include <vector>

#include "BFGS_with_linesearch.hpp"

namespace pnol {
struct BFGSReport {          // what findMin returns for one start
	double f0 = 0;           // the objective at the start
	double fOpt = 0;         // at the end
	int iterations = 0;      // BFGS::iterations() of that start
	int stop = 0;            // the first false conjunct of the loop condition: 0 maxIter, 1 xdiff (NaN included), 2 the gradient norm
};
}

class BFGSBatch : public Algorithm {
  private:
	double c1, c2;
	double dalpha;
	double alphaGuess;
	int maxIterLineSearch;
	double dXGrad;
	double dXHess;
	double xMinDiff;
	double minGrad2Norm;
	int maxIter;
	bool initHessFD;
	bool verbose;

  public:
	/* X: B starts of one length n (in/out); reports: resized to B. Throws pnol::Error as BFGS::findMin does. */
	void findMin( vector <vector <double> > & X, vector <pnol::BFGSReport> & reports );
	/* one start (B = 1) */
	void findMin( vector <double> & X, double & f0, double & fOpt );

	void setParams( double c1In, double c2In, double dalphaIn, double alphaGuessIn, int maxIterLineSearchIn, double dXGradIn, double dXHessIn, double maxIterIn,
			double xMinDiffIn, double minGrad2NormIn, bool initHessFDIn, bool verboseIn )
	{
		c1 = c1In; c2 = c2In; dalpha = dalphaIn; alphaGuess = alphaGuessIn; maxIterLineSearch = maxIterLineSearchIn;
		dXGrad = dXGradIn; dXHess = dXHessIn; maxIter = maxIterIn; xMinDiff = xMinDiffIn; minGrad2Norm = minGrad2NormIn;
		initHessFD = initHessFDIn; verbose = verboseIn;
	}

	BFGSBatch()
	{
		c1 = 1e-4; c2 = 0.9; dalpha = 1e-6; alphaGuess = 1; maxIterLineSearch = 1000;
		dXGrad = 1e-6; dXHess = 1e-3; maxIter = 10000; xMinDiff = 1e-5; minGrad2Norm = 1e-5;
		verbose = 0; initHessFD = 0;
	}
	~BFGSBatch(){}

  private:
	void run( long long B, int n, double * X, vector <pnol::BFGSReport> & reports );
};

#endif
