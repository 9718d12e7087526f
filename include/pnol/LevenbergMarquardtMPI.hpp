/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * LevenbergMarquardtMPI.hpp -- LevMarqMPI, same interface as /root/reference/Source/LevenbergMarquardtMPI.hpp:27-61
 * (setParams argument order and types included: maxIter arrives as a double, verbose is an int).
 * findMin keeps X/J/F on the device for the whole run; with a communicator the residual rows are sharded
 * (each rank's objective holds its row block) and J^T J / J^T r / chi^2 are all-reduced.
 *
 * DIFFERENCE FROM THE REFERENCE UNDER SHARDING: there every rank's objective holds ALL the data and findMin returns the full
 * residual vectors F0 / FOpt on every rank (Source/LevenbergMarquardtMPI.cpp:42-49, :159-162). Here a rank's MultiObjective
 * holds only its row block, F0 / FOpt are pre-sized to THAT block and receive that block's residuals (X, chi^2 and the
 * iteration history are global and identical on all ranks). pnol::gatherResiduals() rebuilds the reference's full vectors
 * (rank order = row order) where a caller wants them; with one rank the two conventions coincide.
 */
#ifndef PNOL_LEVENBERGMARQUARDTMPI_HPP_
#define PNOL_LEVENBERGMARQUARDTMPI_HPP_

#include <vector>

#include "UtilityFunctions.hpp"
#include "PNOL_Algorithm.hpp"

using namespace std;

namespace pnol {
struct LMReport {            // what the last findMin did (the reference only prints these)
	int iterations = 0;      // loop passes completed (iter at exit)
	int accepted = 0;
	int rejected = 0;
	double chiSq = 0;
	double lambda = 0;
	double xdiff2Norm = 0;
	int stopped = 0;         // LevMarqBatch: 1 when the x_min_diff rule ended the problem's loop
};
void lmFindMin( MultiObjective * obj, double lambda0, double lambdaFactor, double dXGrad, int maxIter, double xMinDiff,
		int verbose, vector <double> & X, vector <double> & F0, vector <double> & FOpt, LMReport & report );
// full = the ranks' blocks of `local` concatenated in rank order, on every rank (block lengths may differ). Collective.
void gatherResiduals( const vector <double> & local, vector <double> & full );
}

class LevMarqMPI : public MultiAlgorithm {
  private:
	double lambda0;
	double dXGrad;
	double xMinDiff;
	int maxIter;
	double lambdaFactor;  // Lambda factor: should be > 1
	int verbose;
	pnol::LMReport report;

  public:
	void findMin( vector <double> & X, vector <double> & f0, vector <double> & fOpt );

	void setParams( double lambda0In, double lambdaFactorIn, double dXGradIn, double maxIterIn, double xMinDiffIn, int verboseIn )
	{  maxIter = maxIterIn; xMinDiff = xMinDiffIn; verbose = verboseIn; dXGrad = dXGradIn; lambda0 = lambda0In; lambdaFactor = lambdaFactorIn; }

	const pnol::LMReport & lastReport() const { return report; }

	LevMarqMPI()
	{
		dXGrad = 1e-7;
		lambda0 = 0.001;
		maxIter = 10000;
		xMinDiff = 1e-7;
		verbose = 1;
		lambdaFactor = 10;
	}
	~LevMarqMPI(){}
};

#endif
