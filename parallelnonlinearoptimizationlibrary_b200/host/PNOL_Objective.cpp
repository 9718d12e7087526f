/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
// PNOL_Objective.cpp -- the derivative stencils of the plugin API (Source/PNOL_Objective.cpp of the reference),
// each a thin host call into the C-ABI: the N+1 (or n+1 residual-vector) evaluations run as CUDA kernels.
#include "pnol/PNOL_Objective.hpp"

#include <string>

// Weak references: these sources are also linked against C-ABI implementations other than libpnol_b200.so -- the CPU stand-in of the
// host-logic tests (oracle/host_logic_device.cpp) and programs built with it -- that need not provide the analytic derivatives. There
// these symbols are null and the analytic modes fail with PNOL_ERR_NO_FUNCTOR (requireDerivative) instead of the program failing to link.
extern "C" int pnol_gradient( pnol_ctx *, const pnol_functor *, const double *, int, double *, double * ) __attribute__(( weak ));
extern "C" int pnol_gradient_recur( pnol_ctx *, const pnol_functor *, const double *, int, const double *, const unsigned char *, int,
		double *, double * ) __attribute__(( weak ));
extern "C" int pnol_hessian( pnol_ctx *, const pnol_functor *, const double *, int, double * ) __attribute__(( weak ));
extern "C" int pnol_alpha_pool_analytic( pnol_ctx *, const pnol_functor *, const double *, const double *, int, const double *, int,
		const unsigned char *, const double *, const unsigned char *, int, double *, double *, int * ) __attribute__(( weak ));

namespace {
void requireDerivative( bool available, const char * who, const char * what )
{
	if( !available ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, std::string(who) + ": " + what + " "
			"are not provided by the C-ABI implementation this program is linked against" );
}
void requireGradient( bool available, const char * who ) { requireDerivative( available, who, "analytic gradients (Runtime::setAnalyticGradient)" ); }
}

void pnol::alphaPoolAnalytic( const char * who, pnol_functor * f, const double * X, const double * p, int n, const double * alpha, int npool,
		const double * constX, const unsigned char * constInd, int nfull, double * phi, double * dphi, int * bad )
{
	requireDerivative( pnol_alpha_pool_analytic != nullptr, who, "analytic line-search slopes (Runtime::setAnalyticSlope)" );
	Runtime & rt = Runtime::instance();
	rt.check( pnol_alpha_pool_analytic( rt.ctx(), f, X, p, n, alpha, npool, nullptr, constX, constInd, nfull, phi, dphi, bad ) );
}

pnol_functor * Objective::requireFunctor( const char * who )
{
	pnol_functor * f = deviceFunctor();
	if( !f ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, std::string(who) + ": this Objective has no device functor (deviceFunctor() returned "
			"null). The B200 build evaluates stencils on the GPU only; there is no CPU fallback." );
	return f;
}

pnol_functor * MultiObjective::requireFunctor( const char * who )
{
	pnol_functor * f = deviceFunctor();
	if( !f ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, std::string(who) + ": this MultiObjective has no device functor (deviceFunctor() "
			"returned null). The B200 build evaluates stencils on the GPU only; there is no CPU fallback." );
	return f;
}

// Source/PNOL_Objective.cpp:12-34. The serial stencil never touches MPI in the reference, so it runs in local mode here: no
// collective, all coordinates on this GPU, whatever communicator the context carries.
void Objective::gradientApproximation( vector <double> & X, vector <double> & dX, vector <double> & dFdX )
{
	pnol::LocalScope serial;
	gradientApproximationMPI( X, dX, dFdX );
}

// Source/PNOL_Objective.cpp:88-159: the reference deals the N+1 evaluations out to MPI ranks and sums; the values are
// the same as the serial stencil. With a communicator attached the C-ABI splits the coordinates across GPUs (collective call).
// Runtime::setAnalyticGradient(true): the functor's own partial derivatives instead (dX unused, no objective value evaluated).
void Objective::gradientApproximationMPI( vector <double> & X, vector <double> & dX, vector <double> & dFdX )
{
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = requireFunctor( "Objective::gradientApproximation" );
	if( rt.analyticGradient() )
	{
		requireGradient( pnol_gradient != nullptr, "Objective::gradientApproximation" );
		rt.check( pnol_gradient( rt.ctx(), f, X.data(), (int) X.size(), dFdX.data(), nullptr ) );
		return;
	}
	rt.check( pnol_fd_gradient( rt.ctx(), f, X.data(), dX.data(), (int) X.size(), dFdX.data(), nullptr ) );
	noteDeviceEvaluations( (long long) X.size() + 1 );                        // N + 1 points (:19-32)
}

// Source/PNOL_Objective.cpp:38-85. Runtime::setAnalyticHessian(true): the functor's own second derivatives instead (dX unused, no
// objective value evaluated).
void Objective::hessianApproximation( vector <double> & X, vector <double> & dX, vector<vector<double> > & H )
{
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = requireFunctor( "Objective::hessianApproximation" );
	int N = (int) X.size();
	vector<double> flat( (size_t) N*N );
	if( rt.analyticHessian() )
	{
		requireDerivative( pnol_hessian != nullptr, "Objective::hessianApproximation", "analytic Hessians (Runtime::setAnalyticHessian)" );
		rt.check( pnol_hessian( rt.ctx(), f, X.data(), N, flat.data() ) );
	}
	else
	{
		rt.check( pnol_fd_hessian( rt.ctx(), f, X.data(), dX.data(), N, flat.data() ) );
		noteDeviceEvaluations( 3LL*N*(N + 1)/2 + 1 );                        // what the reference evaluates (:47-71); the kernels reuse f_i
	}
	for( int i = 0; i < N; i++ )
		for( int j = 0; j < N; j++ )
			H[i][j] = flat[(size_t) i*N + j];
}

// Source/PNOL_Objective.cpp:303-333: scatter the free members into the full point, one host evaluation
double Objective::objEvalRecur( vector <double> & Xrecur, vector <double> & constantX, vector<bool> & constantIndicator )
{
	int Nparam = (int) constantX.size();
	vector <double> X( Nparam, 0 );
	int iRecur = 0;
	for( int i = 0; i < Nparam; i++ )
	{
		if( constantIndicator[i] ) X[i] = constantX[i];
		else { X[i] = Xrecur[iRecur]; iRecur++; }
	}
	return objEval( X );
}

// Source/PNOL_Objective.cpp:337-360 (serial: local mode, see gradientApproximation)
void Objective::gradientApproximationRecur( vector <double> & X, vector <double> & dX, vector <double> & dFdX,
		vector <double> & constantX, vector<bool> & constantIndicator )
{
	pnol::LocalScope serial;
	gradientApproximationMPIRecur( X, dX, dFdX, constantX, constantIndicator );
}

// Source/PNOL_Objective.cpp:366-459 (coordinates split across the communicator's GPUs: collective call)
void Objective::gradientApproximationMPIRecur( vector <double> & X, vector <double> & dX, vector <double> & dFdX,
		vector <double> & constantX, vector<bool> & constantIndicator )
{
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = requireFunctor( "Objective::gradientApproximationRecur" );
	vector<unsigned char> ind( constantIndicator.size() );
	for( size_t i = 0; i < ind.size(); i++ ) ind[i] = constantIndicator[i] ? 1 : 0;
	if( rt.analyticGradient() )
	{
		requireGradient( pnol_gradient_recur != nullptr, "Objective::gradientApproximationRecur" );
		rt.check( pnol_gradient_recur( rt.ctx(), f, X.data(), (int) X.size(), constantX.data(), ind.data(), (int) constantX.size(),
				dFdX.data(), nullptr ) );
		return;
	}
	rt.check( pnol_fd_gradient_recur( rt.ctx(), f, X.data(), dX.data(), (int) X.size(), constantX.data(), ind.data(),
			(int) constantX.size(), dFdX.data(), nullptr ) );
	noteDeviceEvaluations( (long long) X.size() + 1 );                        // (:345-358)
}

// Source/PNOL_Objective.cpp:165-197. The drop-in signature returns J as Ndata host rows; the device produces it
// row-major in one kernel and it is copied out row by row. LevMarq[MPI]::findMin keeps J on the device instead.
void MultiObjective::gradientApproximation( vector <double> & X, vector <double> & dX, vector< vector<double> > & J )
{
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = requireFunctor( "MultiObjective::gradientApproximation" );
	long long m = pnol_functor_rows( f );
	int n = (int) X.size();
	if( (long long) J.size() != m ) throw pnol::Error( PNOL_ERR_INVALID, "MultiObjective::gradientApproximation: J has the wrong number of rows" );
	vector<double> flat( (size_t) m*n );
	rt.check( pnol_fd_jacobian( rt.ctx(), f, X.data(), dX.data(), n, flat.data(), nullptr, rt.jacobianMode() ) );
	for( long long i = 0; i < m; i++ )
		for( int j = 0; j < n; j++ )
			J[i][j] = flat[(size_t) i*n + j];
}

// Source/PNOL_Objective.cpp:202-299
void MultiObjective::gradientApproximationMPI( vector <double> & X, vector <double> & dX, vector< vector<double> > & J )
{
	gradientApproximation( X, dX, J );
}
