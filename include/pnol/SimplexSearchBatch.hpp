/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * SimplexSearchBatch.hpp -- SimplexSearchBatch: many independent Nelder-Mead minimisations of one objective (multiple starts) in one
 * call (pnol_simplex_batch). Start b is X[b]; every start gets, bit for bit, what SimplexSearch::findMin gives on that start alone when
 * its start simplex draws the same values. The draws come from pnol::Runtime::defaultStream(1.0) from position 0, as SimplexSearch's
 * do: start b takes the n^2 values from position b n^2, so streamPosition() is B n^2 after a call. setSimplexParams and the defaults
 * are SimplexSearch's; n is 1 .. 64. Nothing is printed: `verbose` is kept for the signature only.
 */
#ifndef PNOL_SIMPLEXSEARCHBATCH_HPP_
#define PNOL_SIMPLEXSEARCHBATCH_HPP_

#include <vector>

#include "PNOL_Algorithm.hpp"

namespace pnol {
struct SimplexReport {       // what findMin returns for one start
	double f0 = 0;           // the objective at the start
	double fOpt = 0;         // at the best vertex
	int iterations = 0;      // SimplexSearch::iterations() of that start
	int stop = 0;            // the first false conjunct of the loop condition: 0 maxIter, 1 xdiff (NaN included)
	long long evaluations = 0;   // objective evaluations the reference makes for that start
};
}

class SimplexSearchBatch : public Algorithm {
  private:
	double alpha, rho, gamma, sigma;
	double initRandMax, xMinDiff;
	int maxIter;
	bool verbose;
	unsigned long long streamPos_;

  public:
	/* X: B starts of one length n (in/out); reports: resized to B. Throws pnol::Error as SimplexSearch::findMin does. */
	void findMin( std::vector <std::vector <double> > & X, std::vector <pnol::SimplexReport> & reports );
	/* one start (B = 1) */
	void findMin( std::vector <double> & X, double & f0, double & fOpt );

	void setSimplexParams( double alphaIn, double gammaIn, double rhoIn, double sigmaIn, int maxIterIn,
			double initRandMaxIn, double xMinDiffIn, bool verboseIn )
	{ alpha = alphaIn; gamma = gammaIn; rho = rhoIn; sigma = sigmaIn;
	  maxIter = maxIterIn; initRandMax = initRandMaxIn; xMinDiff = xMinDiffIn; verbose = verboseIn; }

	/* stream values the last call consumed: B n^2 */
	unsigned long long streamPosition() const { return streamPos_; }

	SimplexSearchBatch()
	{
		alpha = 1.0; gamma = 2.0; rho = 0.5; sigma = 0.5;
		maxIter = 10000;
		initRandMax = 1;
		xMinDiff = 1e-7;
		verbose = 0;
		streamPos_ = 0;
	}
	~SimplexSearchBatch(){}

  private:
	void run( long long B, int n, double * X, std::vector <pnol::SimplexReport> & reports );
};

#endif /* PNOL_SIMPLEXSEARCHBATCH_HPP_ */
