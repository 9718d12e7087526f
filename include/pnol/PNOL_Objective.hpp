/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * PNOL_Objective.hpp -- the objective plugin API, kept source compatible with the reference
 * (/root/reference/Source/PNOL_Objective.hpp:25-62): same class names, same pure virtual objEval signatures (non-const
 * lvalue references), same stencil member functions, `using namespace std;` at header scope and ROOT_ID, because
 * user objectives rely on all of it (Source/ExampleObjectives.hpp).
 *
 * What is new: an objective may expose a DEVICE TWIN (deviceFunctor()). Every stencil below and every algorithm
 * class evaluates through it on the B200; objEval itself stays a host call for the single evaluations the
 * algorithms make. An objective without a device twin cannot use the stencils: they throw pnol::Error -- there is
 * no CPU fallback. <mpi.h> is no longer pulled in (the reference includes it at :20).
 */
#ifndef PNOL_OBJECTIVE_HPP_
#define PNOL_OBJECTIVE_HPP_

using namespace std;

// Parallel commands
#ifndef ROOT_ID
#define ROOT_ID 0 // id of root process
#endif

#include <vector>

#include "Runtime.hpp"

// Evaluates to a single double return
class Objective {
  public:
	virtual ~Objective() {}

	// Pure virtual objective evaluation (Source/PNOL_Objective.hpp:29)
	virtual double objEval( vector <double> & X ) = 0;

	// device twin of objEval: a functor of include/pnol/functors.hpp bound to the runtime's context
	virtual pnol_functor * deviceFunctor() { return nullptr; }
	// the stencils and algorithms report here how many points they evaluated on the device twin, so that stateful objectives can
	// keep the counters the reference's fixtures keep in objEval (`evals++`, Source/ExampleObjectives.hpp:89)
	virtual void noteDeviceEvaluations( long long count ) { (void) count; }

	// forward-difference gradient (Source/PNOL_Objective.cpp:12-34)
	void gradientApproximation( vector <double> & X, vector <double> & dX, vector <double> & dFdX );
	// forward-difference Hessian (Source/PNOL_Objective.cpp:38-85)
	void hessianApproximation( vector <double> & X, vector <double> & dX, vector<vector<double> > & H );
	// "parallel" gradient (Source/PNOL_Objective.cpp:88-159): same kernel; with a communicator the columns are split
	void gradientApproximationMPI( vector <double> & X, vector <double> & dX, vector <double> & dFdX );
	// evaluation with frozen members (Source/PNOL_Objective.cpp:303-333)
	double objEvalRecur( vector <double> & Xrecur, vector <double> & constantX, vector<bool> & constantIndicator );
	// gradient over the free members only (Source/PNOL_Objective.cpp:337-360, 366-459)
	void gradientApproximationRecur( vector <double> & X, vector <double> & dX, vector <double> & dFdX, vector <double> & constantX, vector<bool> & constantIndicator );
	void gradientApproximationMPIRecur( vector <double> & X, vector <double> & dX, vector <double> & dFdX, vector <double> & constantX, vector<bool> & constantIndicator );

  protected:
	pnol_functor * requireFunctor( const char * who );
};

// Evaluates to multiple objective outputs F
class MultiObjective {
  public:
	virtual ~MultiObjective() {}

	// Pure virtual objective evaluation (Source/PNOL_Objective.hpp:57); F is pre-sized by the caller
	virtual void objEval( vector <double> & X, vector <double> & F ) = 0;

	// device twin (a residual functor); its row count is the number of residuals
	virtual pnol_functor * deviceFunctor() { return nullptr; }

	// forward-difference Jacobian, J[i][j] = d F_i / d X_j (Source/PNOL_Objective.cpp:165-197, 202-299)
	void gradientApproximation( vector <double> & X, vector <double> & dX, vector< vector<double> > & J );
	void gradientApproximationMPI( vector <double> & X, vector <double> & dX, vector< vector<double> > & J );

	pnol_functor * requireFunctor( const char * who );
};

namespace pnol {
// phi[k] = f(X + alpha[k] p) and its analytic slope p . grad f(X + alpha[k] p) for the BFGS line searches in the mode
// Runtime::setAnalyticSlope(true): pnol_alpha_pool_analytic on the runtime's context (constInd NULL: no active set). Throws pnol::Error
// with PNOL_ERR_NO_FUNCTOR when the C-ABI implementation the program is linked against does not provide it.
void alphaPoolAnalytic( const char * who, pnol_functor * f, const double * X, const double * p, int n, const double * alpha, int npool,
		const double * constX, const unsigned char * constInd, int nfull, double * phi, double * dphi, int * bad );
}

#endif /* PNOL_OBJECTIVE_HPP_ */
