/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
// BFGS_with_linesearch.cpp -- BFGS::findMin, the strong-Wolfe cubic-interpolation line search, and the shared
// inverse-Hessian machinery. Control flow follows Source/BFGS_with_linesearch.cpp of the reference; the gradient
// stencil, p = -D g, every phi(alpha) evaluation and updateHessianInv run on the device through the C-ABI.
#include "pnol/BFGS_with_linesearch.hpp"

#include <cmath>
#include <iostream>

namespace pnol {

InverseHessian::InverseHessian( int n ) : n_(n), D_( (size_t) n*n ) {}

void InverseHessian::setIdentity()
{
	vector<double> d( n_, 1.0 );
	setDiagonal( d );
}

void InverseHessian::setDiagonal( const vector<double> & d )
{
	Runtime & rt = Runtime::instance();
	rt.check( pnol_memset( rt.ctx(), D_.data(), 0, (size_t) n_*n_*sizeof(double) ) );
	// strided upload of the diagonal: one small copy per row would be n copies; stage a dense host row block instead
	const int rowsPerBlock = n_ > 2048 ? 64 : (n_ > 0 ? n_ : 1);
	vector<double> block( (size_t) rowsPerBlock*n_, 0.0 );
	for( int r0 = 0; r0 < n_; r0 += rowsPerBlock )
	{
		int rows = std::min( rowsPerBlock, n_ - r0 );
		std::fill( block.begin(), block.end(), 0.0 );
		for( int r = 0; r < rows; r++ ) block[(size_t) r*n_ + r0 + r] = d[r0 + r];
		rt.check( pnol_memcpy( rt.ctx(), D_.data() + (size_t) r0*n_, block.data(), (size_t) rows*n_*sizeof(double) ) );
	}
}

void InverseHessian::setFromHost( const vector<vector<double> > & D )
{
	vector<double> flat( (size_t) n_*n_ );
	for( int i = 0; i < n_; i++ ) for( int j = 0; j < n_; j++ ) flat[(size_t) i*n_ + j] = D[i][j];
	D_.upload( flat.data(), flat.size() );
}

void InverseHessian::toHost( vector<vector<double> > & D ) const
{
	vector<double> flat( (size_t) n_*n_ );
	D_.download( flat.data(), flat.size() );
	D.resize( n_ );
	for( int i = 0; i < n_; i++ ) D[i].resize( n_ );
	for( int i = 0; i < n_; i++ ) for( int j = 0; j < n_; j++ ) D[i][j] = flat[(size_t) i*n_ + j];
}

// p = -D dFdX  (Source/BFGS_with_linesearch.cpp:78-79)
void InverseHessian::direction( const vector<double> & dFdX, vector<double> & p )
{
	Runtime & rt = Runtime::instance();
	rt.check( pnol_matvec_neg( rt.ctx(), D_.data(), dFdX.data(), n_, p.data() ) );
}

// updateHessianInv (Source/BFGS_with_linesearch.cpp:389-432)
void InverseHessian::update( const vector<double> & g, const vector<double> & s )
{
	Runtime & rt = Runtime::instance();
	rt.check( pnol_bfgs_update_hinv( rt.ctx(), D_.data(), g.data(), s.data(), n_, rt.hessianUpdateMode() ) );
}

// D = inverse of the forward-difference Hessian (Source/BFGS_with_linesearch.cpp:35-41, BFGS_bnd_linesearch_MPI_SW.cpp:51-59):
// B from the FD stencil, then the reference's `matrixInverse` -- LU with partial pivoting, on the device (pnol_lu_inverse), ONE
// factorisation and n pairs of substitutions. An indefinite Hessian (the normal case away from a minimum) is inverted like any
// other and the run carries on with an indefinite D, exactly as the reference does.
void InverseHessian::setFromInverseOfFDHessian( Objective * obj, vector<double> & X, double dXHess )
{
	Runtime & rt = Runtime::instance();
	vector<double> dXH( n_, dXHess );
	vector<vector<double> > B( n_, vector<double>( n_ ) );
	obj->hessianApproximation( X, dXH, B );
	vector<double> flat( (size_t) n_*n_ );
	for( int i = 0; i < n_; i++ ) for( int j = 0; j < n_; j++ ) flat[(size_t) i*n_ + j] = B[i][j];
	DeviceArray Bd( flat.size() );
	Bd.upload( flat.data(), flat.size() );
	int info = 0;
	rt.check( pnol_lu_inverse( rt.ctx(), Bd.data(), n_, D_.data(), &info ) );
}

} // namespace pnol

// host-matrix form of the update, kept for source compatibility (Source/BFGS_with_linesearch.hpp:109)
void updateHessianInv( vector<vector<double> > & D, vector<double> & g, vector<double> & s )
{
	pnol::InverseHessian H( (int) g.size() );
	H.setFromHost( D );
	H.update( g, s );
	H.toHost( D );
}

// Source/BFGS_with_linesearch.cpp:359-385
double cubicInterpMin( double alpha_lo, double alpha_hi, double phi_lo, double phi_hi, double dphi_lo_dalpha, double dphi_hi_dalpha,
		vector <double> &, vector <double> & )
{
	double d1 = dphi_lo_dalpha + dphi_hi_dalpha - 3*( phi_lo - phi_hi )/( alpha_lo - alpha_hi );
	double d2 = sign( alpha_hi - alpha_lo )*sqrt( pow(d1,2) - dphi_lo_dalpha*dphi_hi_dalpha );
	double alphaNew = alpha_hi - ( alpha_hi - alpha_lo )*( dphi_hi_dalpha + d2 - d1 )/( dphi_hi_dalpha - dphi_lo_dalpha + 2*d2 );
	// if outside the region, use bisection instead
	if( alpha_lo < alpha_hi )
	{
		if( alphaNew < alpha_lo ) alphaNew = (alpha_hi + alpha_lo)/2;
	}
	else
	{
		if( alphaNew < alpha_hi ) alphaNew = (alpha_hi + alpha_lo)/2;
	}
	return alphaNew;
}

// phi(alpha) = f(X + alpha p) and (f(X + (alpha + dalpha) p) - phi)/dalpha: lineSearchObj + lineSearchFDDerivative
// (Source/BFGS_with_linesearch.cpp:144-172) as one two-point pool launch. The serial reference has no NaN sentinel,
// so raw values are wanted: a sentinel-free pool is obtained by undoing the 1e10 replacement only when bad > 0.
void BFGS::evalPhiAndSlope( double alpha, vector <double> & X, vector <double> & p, double & phi, double & dphi )
{
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = objPtr->deviceFunctor();
	if( !f ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "BFGS: the objective has no device functor (no CPU fallback)" );
	int bad = 0;
	if( rt.analyticSlope() )
	{
		// Runtime::setAnalyticSlope(true): the slope p . grad f(X + alpha p), one evaluation; a bad phi is recomputed on the host, the
		// device slope kept
		pnol::alphaPoolAnalytic( "BFGS", f, X.data(), p.data(), (int) X.size(), &alpha, 1, nullptr, nullptr, (int) X.size(), &phi, &dphi, &bad );
		if( bad == 0 ) objPtr->noteDeviceEvaluations( 1 );
		else phi = lineSearchObj( alpha, X, p );
		return;
	}
	rt.check( pnol_alpha_pool( rt.ctx(), f, X.data(), p.data(), (int) X.size(), &alpha, 1, dalpha, nullptr, nullptr, nullptr,
			(int) X.size(), &phi, &dphi, &bad ) );
	if( bad == 0 ) objPtr->noteDeviceEvaluations( 2 );                        // phi and the point of its forward-difference slope
	if( bad > 0 )
	{
		// the serial reference lets NaN/inf flow into its comparisons; reproduce that by re-evaluating on the host
		phi = lineSearchObj( alpha, X, p );
		dphi = lineSearchFDDerivative( alpha, phi, X, p );
	}
}

double BFGS::lineSearchObj( double alpha, vector <double> & X, vector <double> & p )
{
	vector <double> Xalphap( X.size(), 0 );
	for( size_t i = 0; i < X.size(); i++ ) Xalphap[i] = X[i] + alpha*p[i];
	return objPtr->objEval( Xalphap );
}

double BFGS::lineSearchFDDerivative( double alpha, double phialpha, vector <double> & X, vector <double> & p )
{
	vector <double> Xalphap_dalpha( X.size(), 0 );
	for( size_t i = 0; i < X.size(); i++ ) Xalphap_dalpha[i] = X[i] + (alpha+dalpha)*p[i];
	double Falpha_dalpha = objPtr->objEval( Xalphap_dalpha );
	return ( Falpha_dalpha - phialpha )/dalpha;
}

// Source/BFGS_with_linesearch.cpp:12-139
void BFGS::findMin( vector <double> & X, double & f0, double & fOpt )
{
	pnol::LocalScope serial;             // the serial class never touches the communicator (Source/BFGS_with_linesearch.cpp)
	int Nparam = (int) X.size();
	vector<double> Xprev( Nparam, 0 );
	vector<double> dX( Nparam, dXGrad );
	vector<double> dFdX( Nparam, 0 );
	vector<double> dFdX_prev( Nparam, 0 );
	vector<double> p( Nparam, 0 ), s( Nparam, 0 ), g( Nparam, 0 );

	pnol::InverseHessian D( Nparam );
	if( initHessFD ) D.setFromInverseOfFDHessian( objPtr, X, dXHess );      // (:35-41)
	else D.setIdentity();                                                    // (:45-57)

	// Initial gradient approximation (:62-65)
	objPtr->gradientApproximation( X, dX, dFdX );
	for( int i = 0; i < Nparam; i++ ) dFdX_prev[i] = dFdX[i];
	double F = objPtr->objEval( X );
	f0 = F;

	int iter = 0;
	double xdiff = xMinDiff*2;
	double grad2Norm = 2*minGrad2Norm;
	while( iter < maxIter && xdiff > xMinDiff && grad2Norm > minGrad2Norm )      // (:72)
	{
		for( int i = 0; i < Nparam; i++ ) dFdX_prev[i] = dFdX[i];
		D.direction( dFdX, p );                                              // (:78-79)

		double alpha, Fopt;
		cubicInterpolationLineSearch( X, F, dFdX, p, alpha, Fopt );          // (:84)

		for( int i = 0; i < Nparam; i++ )                                    // (:88-93)
		{
			Xprev[i] = X[i];
			X[i] = X[i] + alpha*p[i];
		}
		F = Fopt;

		objPtr->gradientApproximation( X, dX, dFdX );                        // (:97)
		for( int i = 0; i < Nparam; i++ )                                    // (:100-105)
		{
			s[i] = alpha*p[i];
			g[i] = dFdX[i] - dFdX_prev[i];
		}
		D.update( g, s );

		xdiff = 0;
		for( int i = 0; i < Nparam; i++ ) xdiff += fabs( X[i] - Xprev[i] );  // (:111-113)
		grad2Norm = vector2Norm( dFdX );
		if( verbose == true )
		{
			cout << "At iter = " << iter << " the mean abs xdiff is " << xdiff << " and the grad2norm = " << grad2Norm << endl;
			cout << " with a minimum function evaluation of " << F << endl;
		}
		iter = iter + 1;
	}
	iterationsDone = iter;
	fOpt = F;
	if( verbose == true )
	{
		cout << endl << "Completed bfgs. f0 = " << f0 << ", fOpt = " << fOpt << " with variable:" << endl;
		cout << "X = "; print1DVector( X );
	}
}

// Source/BFGS_with_linesearch.cpp:177-291
void BFGS::cubicInterpolationLineSearch( vector <double> & X, double FX,
		vector <double> & dFdX, vector <double> & p, double & alphaOpt, double & Fopt )
{
	double alpha_lo, alpha_hi, phi_lo, phi_hi, dphi_lo_dalpha, dphi_hi_dalpha;
	double dphiOptdalpha;

	alphaOpt = 0;
	Fopt = FX;

	double phi0 = FX;
	double dphi0dalpha = dotProd( dFdX, p );

	double alphaim1 = 0;
	double phiim1 = phi0;
	double dphiim1dalpha = dphi0dalpha;

	double alphai = alphaGuess;
	int iter = 0;
	while( iter < maxIterLineSearch )
	{
		double phii, dphiidalpha;
		evalPhiAndSlope( alphai, X, p, phii, dphiidalpha );

		// 1. sufficient decrease (:209)
		if( ( phii > phi0 + c1*alphai*dphi0dalpha ) || ( phii >= phiim1 && iter > 1 ) )
		{
			alpha_lo = alphaim1; phi_lo = phiim1; dphi_lo_dalpha = dphiim1dalpha;
			alpha_hi = alphai; phi_hi = phii; dphi_hi_dalpha = dphiidalpha;
			lineSearchZoom( alpha_lo, alpha_hi, phi_lo, phi_hi, dphi_lo_dalpha, dphi_hi_dalpha,
					phi0, dphi0dalpha, X, p, alphaOpt, Fopt, dphiOptdalpha );
			break;
		}
		// 2. curvature (:233)
		if( fabs(dphiidalpha) <= fabs( c2*dphi0dalpha ) )
		{
			alphaOpt = alphai;
			Fopt = phii;
			break;
		}
		// 3. positive slope: zoom on the reversed bracket (:248)
		if( dphiidalpha >= 0 )
		{
			alpha_lo = alphai; phi_lo = phii; dphi_lo_dalpha = dphiidalpha;
			alpha_hi = alphaim1; phi_hi = phiim1; dphi_hi_dalpha = dphiim1dalpha;
			lineSearchZoom( alpha_lo, alpha_hi, phi_lo, phi_hi, dphi_lo_dalpha, dphi_hi_dalpha,
					phi0, dphi0dalpha, X, p, alphaOpt, Fopt, dphiOptdalpha );
			break;
		}
		// extend (:272-277)
		alphaim1 = alphai;
		phiim1 = phii;
		dphiim1dalpha = dphiidalpha;
		alphai = 2*alphai;
		iter++;
	}
}

// Source/BFGS_with_linesearch.cpp:296-356
void BFGS::lineSearchZoom( double alpha_lo, double alpha_hi, double phi_lo, double phi_hi, double dphi_lo_dalpha, double dphi_hi_dalpha,
		double phi0, double dphi0dalpha, vector <double> & X, vector <double> & p, double & alphaOpt, double & phiOpt, double & dphiOptdalpha )
{
	int iter = 0;
	while( iter < maxIterLineSearch )
	{
		double alphaj = cubicInterpMin( alpha_lo, alpha_hi, phi_lo, phi_hi, dphi_lo_dalpha, dphi_hi_dalpha, X, p );
		double phij, dphijdalpha;
		evalPhiAndSlope( alphaj, X, p, phij, dphijdalpha );

		if( phij > phi0 + c1*alphaj*dphi0dalpha || phij >= phi_lo )
		{
			alpha_hi = alphaj; phi_hi = phij; dphi_hi_dalpha = dphijdalpha;
		}
		else
		{
			if( fabs(dphijdalpha) <= fabs( c2*dphi0dalpha ) )
			{
				alphaOpt = alphaj; phiOpt = phij; dphiOptdalpha = dphijdalpha;
				break;
			}
			if( dphijdalpha*( alpha_hi - alpha_lo ) >= 0 )
			{
				alpha_hi = alpha_lo; phi_hi = phi_lo; dphi_hi_dalpha = dphi_lo_dalpha;
			}
			alpha_lo = alphaj; phi_lo = phij; dphi_lo_dalpha = dphijdalpha;
		}
		iter++;
	}
}
