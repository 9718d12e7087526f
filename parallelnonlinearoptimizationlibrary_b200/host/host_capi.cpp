/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
// host_capi.cpp -- C entry points that drive the host C++ plugin classes (include/pnol/*.hpp) so that Python tests and
// bench.py can exercise exactly what a C++ user of the reference API would call (LevMarqMPI::findMin, BFGS*::findMin*,
// GeneticAlgorithmMPI::findMinBnd, Objective::gradientApproximation ...). Not part of the drop-in C-ABI
// (include/pnol_b200.h); it sits above it, next to the classes.
#include <cstring>
#include <memory>
#include <sstream>
#include <string>

#include "pnol/ExampleObjectives.hpp"
#include "pnol/LevenbergMarquardt.hpp"
#include "pnol/LevenbergMarquardtMPI.hpp"
#include "pnol/LevenbergMarquardtBatch.hpp"
#include "pnol/BFGS_with_linesearch.hpp"
#include "pnol/BFGSBatch.hpp"
#include "pnol/BFGS_with_linesearch_MPI.hpp"
#include "pnol/BFGS_bnd_linesearch_MPI_SW.hpp"
#include "pnol/BFGS_bnd_linesearch.hpp"
#include "pnol/BFGS_with_bnd_linesearch_MPI.hpp"
#include "pnol/GeneticAlgorithm.hpp"
#include "pnol/GeneticAlgorithmMPI.hpp"
#include "pnol/Box_boundary_functions.hpp"
#include "pnol/SimplexSearch.hpp"
#include "pnol/SimplexSearchBatch.hpp"

namespace {

std::string gErr;
long long gLastEvals = 0;          // objective evaluations of the last pnolhost_bfgs / pnolhost_simplex[_batch] run

struct CoutSilencer {
	std::streambuf * old;
	bool on;
	explicit CoutSilencer( bool silence ) : old( nullptr ), on( silence ) { if( on ) old = std::cout.rdbuf( nullptr ); }
	~CoutSilencer() { if( on ) std::cout.rdbuf( old ); }
};

template <class Fn> int guarded( Fn && fn )
{
	try { fn(); return PNOL_OK; }
	catch( const pnol::Error & e ) { gErr = e.what(); return e.status(); }
	catch( const std::exception & e ) { gErr = e.what(); return PNOL_ERR_INVALID; }
}

std::unique_ptr<Objective> makeScalar( const std::string & spec )
{
	if( spec == "rosenbrock" ) return std::unique_ptr<Objective>( new RosenbrockObject() );
	if( spec == "booth" ) return std::unique_ptr<Objective>( new BoothFunction() );
	if( spec == "goldstein" ) return std::unique_ptr<Objective>( new GoldsteinFunction() );
	if( spec == "rastrigin" ) return std::unique_ptr<Objective>( new RastriginObject() );
	if( spec == "expsingle" ) return std::unique_ptr<Objective>( new ExpCurveObjectiveSingle() );
	if( spec.compare( 0, 6, "power:" ) == 0 ) { PowerObject * o = new PowerObject(); o->setPower( atoi( spec.c_str() + 6 ) ); return std::unique_ptr<Objective>( o ); }
	throw pnol::Error( PNOL_ERR_INVALID, "unknown scalar objective " + spec );
}

// forwards to an objective and counts what it evaluates: host objEval calls and the points the device reports
struct CountingObjective : public Objective {
	Objective & o;
	long long evals = 0;
	explicit CountingObjective( Objective & obj ) : o( obj ) {}
	double objEval( vector <double> & X ) { evals++; return o.objEval( X ); }
	pnol_functor * deviceFunctor() { return o.deviceFunctor(); }
	void noteDeviceEvaluations( long long count ) { evals += count; }
};

// a built-in residual model over caller data (host arrays are copied): the objective LevMarqBatch fits
template <class R> struct BatchModel : public pnol::FunctorMultiObjective<R> {
	BatchModel( const double * scalars, const double * const * columns, int ncols, long long m )
	{
		for( int k = 0; k < PNOL_MAX_SCALARS; k++ ) this->P.scalars[k] = scalars ? scalars[k] : 0.0;
		this->cols.resize( ncols );
		for( int c = 0; c < ncols; c++ ) this->cols[c].assign( columns[c], columns[c] + m );
		this->bindColumns();
	}
};

std::unique_ptr<MultiObjective> makeResidual( int kind, const double * scalars, const double * const * columns, int ncols, long long m )
{
	if( kind == PNOL_F_EXPCURVE && ncols == 2 ) return std::unique_ptr<MultiObjective>( new BatchModel<pnol::ExpCurveFunctor>( scalars, columns, ncols, m ) );
	if( kind == PNOL_F_CUBIC && ncols == 3 ) return std::unique_ptr<MultiObjective>( new BatchModel<pnol::CubicFunctor>( scalars, columns, ncols, m ) );
	if( kind == PNOL_F_LORENTZ_SUM && ncols == 2 ) return std::unique_ptr<MultiObjective>( new BatchModel<pnol::LorentzSumFunctor>( scalars, columns, ncols, m ) );
	throw pnol::Error( PNOL_ERR_INVALID, "unknown residual model / column count" );
}

}

extern "C" {

const char * pnolhost_last_error() { return gErr.c_str(); }

int pnolhost_attach( pnol_ctx * ctx ) { return guarded( [&] { pnol::Runtime::instance().attach( ctx ); } ); }
int pnolhost_detach() { return guarded( [&] { pnol::Runtime::instance().reset(); } ); }
int pnolhost_set_pool_width( int w ) { pnol::Runtime::instance().setPoolWidth( w ); return PNOL_OK; }
int pnolhost_set_hinv_mode( int m ) { pnol::Runtime::instance().setHessianUpdateMode( m ); return PNOL_OK; }
int pnolhost_set_jacobian_cache( int on ) { pnol::Runtime::instance().setJacobianCache( on != 0 ); return PNOL_OK; }
int pnolhost_set_store_jacobian( int on ) { pnol::Runtime::instance().setStoreJacobian( on != 0 ); return PNOL_OK; }
int pnolhost_set_jac_mode( int m ) { pnol::Runtime::instance().setJacobianMode( m ); return PNOL_OK; }
int pnolhost_set_analytic_gradient( int on ) { pnol::Runtime::instance().setAnalyticGradient( on != 0 ); return PNOL_OK; }
int pnolhost_set_analytic_hessian( int on ) { pnol::Runtime::instance().setAnalyticHessian( on != 0 ); return PNOL_OK; }
int pnolhost_set_analytic_slope( int on ) { pnol::Runtime::instance().setAnalyticSlope( on != 0 ); return PNOL_OK; }
int pnolhost_set_stream( const double * values, unsigned long long n_values, unsigned long long seed, double scale )
{
	pnol_stream_desc s;
	s.values = values; s.n_values = n_values; s.seed = seed; s.scale = scale;
	pnol::Runtime::instance().setRandomStream( s );
	return PNOL_OK;
}
int pnolhost_clear_stream() { pnol::Runtime::instance().clearRandomStream(); return PNOL_OK; }

// LevMarqMPI::findMin (serial != 0: LevMarq) on the Lorentz-sum model with caller data. report[6] = iterations,
// accepted, rejected, chiSq, lambda, xdiff2Norm
int pnolhost_lm_lorentz( const double * t, const double * y, long long m, double w, double * X, int n, double lambda0, double factor,
		double dxgrad, double maxiter, double xmindiff, int serial, double * F0, double * F, double * report )
{
	return guarded( [&] {
		CoutSilencer quiet( true );
		vector<double> tv( t, t + m ), yv( y, y + m );
		LorentzSumObjective obj( tv, yv, w );
		vector<double> Xv( X, X + n ), F0v( m ), Fv( m );
		pnol::LMReport rep;
		if( serial ) { LevMarq lm; lm.setObjPtr( obj ); lm.setParams( lambda0, factor, dxgrad, maxiter, xmindiff, -1 ); lm.findMin( Xv, F0v, Fv ); rep = lm.lastReport(); }
		else { LevMarqMPI lm; lm.setObjPtr( obj ); lm.setParams( lambda0, factor, dxgrad, maxiter, xmindiff, -1 ); lm.findMin( Xv, F0v, Fv ); rep = lm.lastReport(); }
		memcpy( X, Xv.data(), n*sizeof(double) );
		if( F0 ) memcpy( F0, F0v.data(), m*sizeof(double) );
		if( F ) memcpy( F, Fv.data(), m*sizeof(double) );
		if( report ) { report[0] = rep.iterations; report[1] = rep.accepted; report[2] = rep.rejected; report[3] = rep.chiSq; report[4] = rep.lambda; report[5] = rep.xdiff2Norm; }
	} );
}

// The same through a problem handle, the way a C++ user holds it: the objective (with its host data) is built once, every run
// is `lm.setObjPtr(obj); lm.setParams(...); lm.findMin(X, F0, F)` on caller-lifetime vectors -- no copies added by this C face.
// fresh_device_twin != 0 drops the objective's device functor first, so that the upload of the data columns happens inside
// this findMin (what a first call on a new objective pays).
struct LMProblem {
	LorentzSumObjective obj;
	vector<double> F0, F;
	LMProblem( const vector<double> & t, const vector<double> & y, double w ) : obj( t, y, w ), F0( t.size() ), F( t.size() ) {}
};

void * pnolhost_lm_problem_create( const double * t, const double * y, long long m, double w )
{
	void * out = nullptr;
	guarded( [&] { vector<double> tv( t, t + m ), yv( y, y + m ); out = new LMProblem( tv, yv, w ); } );
	return out;
}

void pnolhost_lm_problem_destroy( void * prob ) { guarded( [&] { delete static_cast<LMProblem *>( prob ); } ); }

int pnolhost_lm_problem_run( void * prob, double * X, int n, double lambda0, double factor, double dxgrad, double maxiter, double xmindiff,
		int serial, int fresh_device_twin, double * report, const double ** F0, const double ** F )
{
	return guarded( [&] {
		CoutSilencer quiet( true );
		LMProblem * p = static_cast<LMProblem *>( prob );
		if( !p ) throw pnol::Error( PNOL_ERR_INVALID, "null LM problem" );
		if( fresh_device_twin ) p->obj.releaseDeviceFunctor();
		vector<double> Xv( X, X + n );
		pnol::LMReport rep;
		if( serial ) { LevMarq lm; lm.setObjPtr( p->obj ); lm.setParams( lambda0, factor, dxgrad, maxiter, xmindiff, -1 ); lm.findMin( Xv, p->F0, p->F ); rep = lm.lastReport(); }
		else { LevMarqMPI lm; lm.setObjPtr( p->obj ); lm.setParams( lambda0, factor, dxgrad, maxiter, xmindiff, -1 ); lm.findMin( Xv, p->F0, p->F ); rep = lm.lastReport(); }
		memcpy( X, Xv.data(), n*sizeof(double) );
		if( F0 ) *F0 = p->F0.data();
		if( F ) *F = p->F.data();
		if( report ) { report[0] = rep.iterations; report[1] = rep.accepted; report[2] = rep.rejected; report[3] = rep.chiSq; report[4] = rep.lambda; report[5] = rep.xdiff2Norm; }
	} );
}

// LM on the reference's own fixtures: name = "expcurve" | "cubic" (m = 100)
int pnolhost_lm_example( const char * name, double * X, int n, double lambda0, double factor, double dxgrad, double maxiter, double xmindiff,
		double * F0, double * F, double * report )
{
	return guarded( [&] {
		CoutSilencer quiet( true );
		std::unique_ptr<MultiObjective> obj;
		if( std::string( name ) == "expcurve" ) obj.reset( new ExpCurveObjective() );
		else if( std::string( name ) == "cubic" ) obj.reset( new CubicObjective() );
		else throw pnol::Error( PNOL_ERR_INVALID, std::string( "unknown residual objective " ) + name );
		long long m = pnol_functor_rows( obj->requireFunctor( "pnolhost_lm_example" ) );
		vector<double> Xv( X, X + n ), F0v( m ), Fv( m );
		LevMarqMPI lm; lm.setObjPtr( *obj ); lm.setParams( lambda0, factor, dxgrad, maxiter, xmindiff, -1 );
		lm.findMin( Xv, F0v, Fv );
		memcpy( X, Xv.data(), n*sizeof(double) );
		if( F0 ) memcpy( F0, F0v.data(), m*sizeof(double) );
		if( F ) memcpy( F, Fv.data(), m*sizeof(double) );
		const pnol::LMReport & rep = lm.lastReport();
		if( report ) { report[0] = rep.iterations; report[1] = rep.accepted; report[2] = rep.rejected; report[3] = rep.chiSq; report[4] = rep.lambda; report[5] = rep.xdiff2Norm; }
	} );
}

// LevMarqBatch::findMin(rowOffsets, X, reports) on a built-in residual model (kind, scalars[8], ncols columns of m rows). X is B x n
// row-major (in/out); iters / stopped / chi / lam receive the per-problem reports
int pnolhost_lm_batch( int kind, const double * scalars, const double * const * columns, int ncols, long long m, const long long * rowOff,
		long long B, double * X, int n, double lambda0, double factor, double dxgrad, double maxiter, double xmindiff, int * iters, int * stopped,
		double * chi, double * lam )
{
	return guarded( [&] {
		std::unique_ptr<MultiObjective> obj = makeResidual( kind, scalars, columns, ncols, m );
		vector<long long> ro( rowOff, rowOff + B + 1 );
		vector<vector<double> > Xv( (size_t) B );
		for( long long b = 0; b < B; b++ ) Xv[b].assign( X + b*n, X + (b + 1)*n );
		vector<pnol::LMReport> rep;
		LevMarqBatch lm; lm.setObjPtr( *obj ); lm.setParams( lambda0, factor, dxgrad, maxiter, xmindiff, -1 );
		lm.findMin( ro, Xv, rep );
		for( long long b = 0; b < B; b++ )
		{
			memcpy( X + b*n, Xv[b].data(), n*sizeof(double) );
			iters[b] = rep[b].iterations; stopped[b] = rep[b].stopped; chi[b] = rep[b].chiSq; lam[b] = rep[b].lambda;
		}
	} );
}

// the base class's findMin(X, F0, FOpt) of LevMarqBatch: all m rows as one problem
int pnolhost_lm_batch_single( int kind, const double * scalars, const double * const * columns, int ncols, long long m, double * X, int n,
		double lambda0, double factor, double dxgrad, double maxiter, double xmindiff, double * F0, double * F )
{
	return guarded( [&] {
		std::unique_ptr<MultiObjective> obj = makeResidual( kind, scalars, columns, ncols, m );
		vector<double> Xv( X, X + n ), F0v( m ), Fv( m );
		LevMarqBatch lm; lm.setObjPtr( *obj ); lm.setParams( lambda0, factor, dxgrad, maxiter, xmindiff, -1 );
		lm.findMin( Xv, F0v, Fv );
		memcpy( X, Xv.data(), n*sizeof(double) );
		if( F0 ) memcpy( F0, F0v.data(), m*sizeof(double) );
		if( F ) memcpy( F, Fv.data(), m*sizeof(double) );
	} );
}

// stencils through the plugin classes. which: 0 gradientApproximation, 1 gradientApproximationMPI
int pnolhost_gradient( const char * objective, const double * X, const double * dX, int n, int which, double * g )
{
	return guarded( [&] {
		std::unique_ptr<Objective> obj = makeScalar( objective );
		vector<double> Xv( X, X + n ), dXv( dX, dX + n ), gv( n );
		if( which == 0 ) obj->gradientApproximation( Xv, dXv, gv ); else obj->gradientApproximationMPI( Xv, dXv, gv );
		memcpy( g, gv.data(), n*sizeof(double) );
	} );
}

int pnolhost_gradient_recur( const char * objective, const double * Xr, const double * dXr, int nr, const double * constX,
		const unsigned char * constInd, int nfull, double * g, double * f )
{
	return guarded( [&] {
		std::unique_ptr<Objective> obj = makeScalar( objective );
		vector<double> Xv( Xr, Xr + nr ), dXv( dXr, dXr + nr ), gv( nr ), cx( constX, constX + nfull );
		vector<bool> ci( nfull );
		for( int i = 0; i < nfull; i++ ) ci[i] = constInd[i] != 0;
		obj->gradientApproximationMPIRecur( Xv, dXv, gv, cx, ci );
		memcpy( g, gv.data(), nr*sizeof(double) );
		if( f ) *f = obj->objEvalRecur( Xv, cx, ci );
	} );
}

int pnolhost_hessian( const char * objective, const double * X, const double * dX, int n, double * B )
{
	return guarded( [&] {
		std::unique_ptr<Objective> obj = makeScalar( objective );
		vector<double> Xv( X, X + n ), dXv( dX, dX + n );
		vector<vector<double> > H( n, vector<double>( n ) );
		obj->hessianApproximation( Xv, dXv, H );
		for( int i = 0; i < n; i++ ) for( int j = 0; j < n; j++ ) B[(size_t) i*n + j] = H[i][j];
	} );
}

// BFGS_Bnd_MPI_SW::evaluateAlphaPoolAndDerivatives on one pool (constInd NULL: no frozen members, nfull = n); *evals = the objective
// evaluations it reports
int pnolhost_alpha_pool_sw( const char * objective, const double * X, const double * p, int n, const double * alpha, int npool,
		const double * constX, const unsigned char * constInd, int nfull, double * phi, double * dphi, long long * evals )
{
	return guarded( [&] {
		CoutSilencer quiet( true );
		std::unique_ptr<Objective> obj = makeScalar( objective );
		CountingObjective counted( *obj );
		BFGS_Bnd_MPI_SW alg; alg.setObjPtr( counted );
		vector<double> Xv( X, X + n ), pv( p, p + n ), av( alpha, alpha + npool ), phiv( npool ), dphiv( npool );
		vector<double> cx( constInd ? constX : X, ( constInd ? constX : X ) + nfull );
		vector<bool> ci( nfull, false );
		if( constInd ) for( int i = 0; i < nfull; i++ ) ci[i] = constInd[i] != 0;
		alg.evaluateAlphaPoolAndDerivatives( av, Xv, pv, cx, ci, phiv, dphiv );
		memcpy( phi, phiv.data(), npool*sizeof(double) );
		memcpy( dphi, dphiv.data(), npool*sizeof(double) );
		if( evals ) *evals = counted.evals;
	} );
}

double pnolhost_obj_eval( const char * objective, const double * X, int n )
{
	double v = NAN;
	guarded( [&] { std::unique_ptr<Objective> obj = makeScalar( objective ); vector<double> Xv( X, X + n ); v = obj->objEval( Xv ); } );
	return v;
}

// Jacobian through MultiObjective::gradientApproximation on "expcurve" | "cubic"; J is 100 x n row-major
int pnolhost_jacobian_example( const char * name, const double * X, const double * dX, int n, double * J, double * F )
{
	return guarded( [&] {
		std::unique_ptr<MultiObjective> obj;
		if( std::string( name ) == "expcurve" ) obj.reset( new ExpCurveObjective() );
		else if( std::string( name ) == "cubic" ) obj.reset( new CubicObjective() );
		else throw pnol::Error( PNOL_ERR_INVALID, std::string( "unknown residual objective " ) + name );
		int m = 100;
		vector<double> Xv( X, X + n ), dXv( dX, dX + n ), Fv( m );
		vector<vector<double> > Jv( m, vector<double>( n ) );
		obj->gradientApproximationMPI( Xv, dXv, Jv );
		obj->objEval( Xv, Fv );
		for( int i = 0; i < m; i++ ) for( int j = 0; j < n; j++ ) J[(size_t) i*n + j] = Jv[i][j];
		if( F ) memcpy( F, Fv.data(), m*sizeof(double) );
	} );
}

// BFGS family. variant: "bfgs" | "bfgs_mpi" | "bfgs_bnd" | "bfgs_bnd_sw" | "bfgsbnd_mpi". params (doubles):
//   bfgs        : c1 c2 dalpha alphaGuess maxIterLS dXGrad dXHess maxIter xMinDiff minGrad2Norm initHessFD
//   bfgs_mpi    : c1 c2 maxAlphaMult alphaGuess maxIterLS dXGrad dXHess maxIter xMinDiff minGrad2Norm initHessFD
//   bfgsbnd_mpi : c1 c2 alphaMin maxAlphaMult alphaGuess maxIterLS dXGrad dXHess maxIter xMinDiff minGrad2Norm FStepTolerance initHessFD
//   bfgs_bnd / bfgs_bnd_sw : c1 c2 dalpha alphaGuess alphaTol alphaMult maxIterLS bndTol dXGrad dXHess maxIter xMinDiff minGrad2Norm initHessFD
int pnolhost_bfgs( const char * variant, const char * objective, double * X, int n, const double * p, const double * xlb, const double * xub,
		int poolWidth, int verbose, double * f0, double * fOpt, int * iters )
{
	return guarded( [&] {
		CoutSilencer quiet( verbose == 0 );
		std::unique_ptr<Objective> made = makeScalar( objective );
		CountingObjective counted( *made );
		Objective * obj = &counted;
		vector<double> Xv( X, X + n );
		std::string v( variant );
		double a = 0, b = 0;
		int it = 0;
		if( v == "bfgs" )
		{
			BFGS alg; alg.setObjPtr( *obj );
			alg.setParams( p[0], p[1], p[2], p[3], (int) p[4], p[5], p[6], p[7], p[8], p[9], p[10] != 0, verbose != 0 );
			alg.findMin( Xv, a, b ); it = alg.iterations();
		}
		else if( v == "bfgs_mpi" )
		{
			BFGS_MPI alg; alg.setObjPtr( *obj );
			alg.setParams( p[0], p[1], p[2], p[3], (int) p[4], p[5], p[6], p[7], p[8], p[9], p[10] != 0, verbose != 0 );
			if( poolWidth > 0 ) alg.setPoolWidth( poolWidth );
			alg.findMin( Xv, a, b ); it = alg.iterations();
		}
		else if( v == "bfgs_bnd_sw" )
		{
			BFGS_Bnd_MPI_SW alg; alg.setObjPtr( *obj );
			alg.setParams( p[0], p[1], p[2], p[3], p[4], p[5], (int) p[6], p[7], p[8], p[9], p[10], p[11], p[12], p[13] != 0, verbose );
			if( poolWidth > 0 ) alg.setPoolWidth( poolWidth );
			vector<double> lb( xlb, xlb + n ), ub( xub, xub + n );
			alg.findMinBnd( Xv, lb, ub, a, b ); it = alg.iterations();
		}
		else if( v == "bfgs_bnd" )
		{
			BFGS_Bnd alg; alg.setObjPtr( *obj );
			alg.setParams( p[0], p[1], p[2], p[3], p[4], p[5], (int) p[6], p[7], p[8], p[9], p[10], p[11], p[12], p[13] != 0, verbose );
			vector<double> lb( xlb, xlb + n ), ub( xub, xub + n );
			alg.findMinBnd( Xv, lb, ub, a, b ); it = alg.iterations();
		}
		else if( v == "bfgsbnd_mpi" )
		{
			BFGSBnd_MPI alg; alg.setObjPtr( *obj );
			alg.setParams( p[0], p[1], p[2], p[3], p[4], (int) p[5], p[6], p[7], p[8], p[9], p[10], p[11], p[12] != 0, verbose != 0 );
			if( poolWidth > 0 ) alg.setPoolWidth( poolWidth );
			vector<double> lb( xlb, xlb + n ), ub( xub, xub + n );
			alg.findMinBnd( Xv, lb, ub, a, b ); it = alg.iterations();
		}
		else throw pnol::Error( PNOL_ERR_INVALID, "unknown BFGS variant " + v );
		memcpy( X, Xv.data(), n*sizeof(double) );
		if( f0 ) *f0 = a;
		if( fOpt ) *fOpt = b;
		if( iters ) *iters = it;
		gLastEvals = counted.evals;
	} );
}

// BFGSBatch::findMin(X, reports) on one of the example objectives: X is B x n row-major (in/out), p[11] as for pnolhost_bfgs("bfgs");
// single != 0: the base class's findMin(X, f0, fOpt) on the one start of X (B = 1; iters / stop are then not written)
int pnolhost_bfgs_batch( const char * objective, double * X, long long B, int n, const double * p, int single, double * f0, double * fOpt,
		int * iters, int * stop )
{
	return guarded( [&] {
		std::unique_ptr<Objective> obj = makeScalar( objective );
		BFGSBatch alg; alg.setObjPtr( *obj );
		alg.setParams( p[0], p[1], p[2], p[3], (int) p[4], p[5], p[6], p[7], p[8], p[9], p[10] != 0, false );
		if( single )
		{
			vector<double> Xv( X, X + n );
			alg.findMin( Xv, f0[0], fOpt[0] );
			memcpy( X, Xv.data(), n*sizeof(double) );
			return;
		}
		vector<vector<double> > Xv( (size_t) B );
		for( long long b = 0; b < B; b++ ) Xv[b].assign( X + b*n, X + (b + 1)*n );
		vector<pnol::BFGSReport> rep;
		alg.findMin( Xv, rep );
		for( long long b = 0; b < B; b++ )
		{
			memcpy( X + b*n, Xv[b].data(), n*sizeof(double) );
			f0[b] = rep[b].f0; fOpt[b] = rep[b].fOpt; iters[b] = rep[b].iterations; stop[b] = rep[b].stop;
		}
	} );
}

// objective evaluations (host objEval calls and points evaluated on the device twin) of the last pnolhost_bfgs, pnolhost_simplex or
// pnolhost_simplex_batch run
long long pnolhost_last_evaluations() { return gLastEvals; }

// SimplexSearch::findMin on one of the example objectives. p[7] = alpha gamma rho sigma maxIter initRandMax xMinDiff; the start simplex
// draws from the stream set with pnolhost_set_stream(). report[2] = iterations, stream position
int pnolhost_simplex( const char * objective, double * X, int n, const double * p, int verbose, double * f0, double * fOpt, double * report )
{
	return guarded( [&] {
		CoutSilencer quiet( verbose == 0 );
		std::unique_ptr<Objective> obj = makeScalar( objective );
		CountingObjective counted( *obj );
		gLastEvals = 0;
		vector<double> Xv( X, X + n );
		SimplexSearch alg; alg.setObjPtr( counted );
		alg.setSimplexParams( p[0], p[1], p[2], p[3], (int) p[4], p[5], p[6], verbose != 0 );
		double a = 0, b = 0;
		alg.findMin( Xv, a, b );
		gLastEvals = counted.evals;
		memcpy( X, Xv.data(), n*sizeof(double) );
		if( f0 ) *f0 = a;
		if( fOpt ) *fOpt = b;
		if( report ) { report[0] = alg.iterations(); report[1] = (double) alg.streamPosition(); }
	} );
}

// SimplexSearchBatch::findMin(X, reports) on one of the example objectives: X is B x n row-major (in/out), p[7] as for pnolhost_simplex;
// the start simplices draw from the stream set with pnolhost_set_stream(). single != 0: the base class's findMin(X, f0, fOpt) on the
// one start of X (B = 1; iters / stop / evals are then not written). report[1] (may be NULL): the stream position afterwards.
int pnolhost_simplex_batch( const char * objective, double * X, long long B, int n, const double * p, int single, double * f0, double * fOpt,
		int * iters, int * stop, long long * evals, double * report )
{
	return guarded( [&] {
		std::unique_ptr<Objective> obj = makeScalar( objective );
		CountingObjective counted( *obj );
		gLastEvals = 0;
		SimplexSearchBatch alg; alg.setObjPtr( counted );
		alg.setSimplexParams( p[0], p[1], p[2], p[3], (int) p[4], p[5], p[6], false );
		if( single )
		{
			vector<double> Xv( X, X + n );
			alg.findMin( Xv, f0[0], fOpt[0] );
			memcpy( X, Xv.data(), n*sizeof(double) );
		}
		else
		{
			vector<vector<double> > Xv( (size_t) B );
			for( long long b = 0; b < B; b++ ) Xv[b].assign( X + b*n, X + (b + 1)*n );
			vector<pnol::SimplexReport> rep;
			alg.findMin( Xv, rep );
			for( long long b = 0; b < B; b++ )
			{
				memcpy( X + b*n, Xv[b].data(), n*sizeof(double) );
				f0[b] = rep[b].f0; fOpt[b] = rep[b].fOpt; iters[b] = rep[b].iterations; stop[b] = rep[b].stop; evals[b] = rep[b].evaluations;
			}
		}
		gLastEvals = counted.evals;
		if( report ) { report[0] = 0; report[1] = (double) alg.streamPosition(); }
	} );
}

// GeneticAlgorithmMPI::findMinBnd (serial != 0: GeneticAlgorithm). report[7] = generations, stopped, stream position,
// Nelite, NeliteMut, Ncross, Nrand. The random stream is the one set with pnolhost_set_stream().
int pnolhost_ga( const char * objective, double * X, int n, const double * xlb, const double * xub, int npop, int maxgen, double eliteFrac,
		double crossFrac, double eliteMutFrac, double mutSize, double eliteMutSize, double nstatic, int serial, double * f0, double * fOpt,
		double * report )
{
	return guarded( [&] {
		CoutSilencer quiet( true );
		std::unique_ptr<Objective> obj = makeScalar( objective );
		vector<double> Xv( X, X + n ), lb( xlb, xlb + n ), ub( xub, xub + n );
		double a = 0, b = 0;
		pnol::GAReport rep;
		if( serial )
		{
			GeneticAlgorithm ga; ga.setObjPtr( *obj );
			ga.setGAParams( npop, maxgen, eliteFrac, crossFrac, eliteMutFrac, mutSize, eliteMutSize, 0.5, nstatic, false, false );
			ga.findMinBnd( Xv, lb, ub, a, b ); rep = ga.lastReport();
		}
		else
		{
			GeneticAlgorithmMPI ga; ga.setObjPtr( *obj );
			ga.setGAParams( npop, maxgen, eliteFrac, crossFrac, eliteMutFrac, mutSize, eliteMutSize, 0.5, nstatic, false );
			ga.findMinBnd( Xv, lb, ub, a, b ); rep = ga.lastReport();
		}
		memcpy( X, Xv.data(), n*sizeof(double) );
		if( f0 ) *f0 = a;
		if( fOpt ) *fOpt = b;
		if( report ) { report[0] = rep.generations; report[1] = rep.stoppedStatic; report[2] = (double) rep.streamPos; report[3] = rep.Nelite;
			report[4] = rep.NeliteMut; report[5] = rep.Ncross; report[6] = rep.Nrand; }
	} );
}

int pnolhost_check_box_bounds( double * X, const double * xlb, const double * xub, int n )
{
	return guarded( [&] {
		CoutSilencer quiet( true );
		vector<double> Xv( X, X + n ), lb( xlb, xlb + n ), ub( xub, xub + n );
		checkBoxBounds( Xv, lb, ub );
		memcpy( X, Xv.data(), n*sizeof(double) );
	} );
}

double pnolhost_compute_alpha_bnd( const double * X, const double * xlb, const double * xub, const double * p, int n )
{
	vector<double> Xv( X, X + n ), lb( xlb, xlb + n ), ub( xub, xub + n ), pv( p, p + n );
	return computeAlphaBnd( Xv, lb, ub, pv );
}

} // extern "C"
