/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
// BFGS_bnd_linesearch_MPI_SW.cpp -- BFGS_Bnd_MPI_SW: bounded BFGS, pooled strong-Wolfe line search, active-set
// recursion. The host control flow follows Source/BFGS_bnd_linesearch_MPI_SW.cpp of the reference decision for
// decision (iterates must match it); gradient stencils, p = -D g, the alpha pools and updateHessianInv are device work.
#include "pnol/BFGS_bnd_linesearch_MPI_SW.hpp"

#include <cmath>
#include <iostream>

BFGS_Bnd_MPI_SW::BFGS_Bnd_MPI_SW()
{
	c1 = 1e-4; c2 = 0.9; dalpha = 1e-6; alphaGuess = 1; alphaTol = 1e-20; alphaMult = 2; maxIterLineSearch = 50;
	bndTol = 1e-5; dXGrad = 1e-6; dXHess = 1e-3; maxIter = 10000; xMinDiff = 1e-5; minGrad2Norm = 1e-5; initHessFD = 0;
	verbose = 0;
	// the reference asks MPI for the rank count here (Source/BFGS_bnd_linesearch_MPI_SW.hpp:134-135)
	Nprocs = pnol::Runtime::instance().poolWidth();
	procID = 0;
	optimFlag = true;
	recurFlag = 0;
	totalIter = 0;
	serialSearch = false;
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:12-113
void BFGS_Bnd_MPI_SW::findMinBnd( vector <double> & X, vector <double> & Xlb, vector <double> & Xub, double & f0, double & fOpt )
{
	totalIter = 0;
	int Nparam = (int) X.size();

	checkBoxBounds( X, Xlb, Xub );                                           // (:27)

	vector<double> constantX( Nparam, 0 );
	vector<bool> constantIndicator( Nparam, false );
	vector<double> dX( Nparam, dXGrad );
	vector<double> dFdX( Nparam, 0 );
	if( dXGradVec.size() > 0 )
		for( int i = 0; i < Nparam; i++ ) dX[i] = dXGradVec[i];              // (:38-44)

	pnol::InverseHessian D( Nparam );
	if( initHessFD ) D.setFromInverseOfFDHessian( objPtr, X, dXHess );        // (:51-59)
	else if( initialScalingVec.size() > 0 ) D.setDiagonal( initialScalingVec );   // (:63-78)
	else D.setIdentity();

	objPtr->gradientApproximationMPIRecur( X, dX, dFdX, constantX, constantIndicator );   // (:83)
	double F = objPtr->objEvalRecur( X, constantX, constantIndicator );       // (:86)
	f0 = F;

	optimFlag = true;
	recurFlag = 0;
	mainBFGSLoop( F, X, dFdX, D, Xlb, Xub, dX, constantX, constantIndicator );   // (:92)

	fOpt = F;
	if( verbose > 0 )
	{
		cout << endl << "  Completed bounded BFGS. f0 = " << f0 << ", fOpt = " << fOpt << endl;
		cout << "  Xopt = "; print1DVector( X );
	}
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:116-207
void BFGS_Bnd_MPI_SW::mainBFGSLoop( double & F, vector <double> & X, vector<double> & dFdX, pnol::InverseHessian & D,
		vector <double> & Xlb, vector <double> & Xub, vector<double> & dX, vector<double> & constantX,
		vector<bool> & constantIndicator )
{
	int Nparam = (int) X.size();
	vector<double> dFdX_prev( Nparam, 0 );
	vector<double> p( Nparam, 0 ), s( Nparam, 0 ), g( Nparam, 0 ), Xprev( Nparam, 0 );
	for( int i = 0; i < Nparam; i++ ) dFdX_prev[i] = dFdX[i];

	int iter = 0;
	double xdiff = xMinDiff*2;
	double grad2Norm = 2*minGrad2Norm;
	while( optimFlag && iter < maxIter && xdiff > xMinDiff && grad2Norm > minGrad2Norm && totalIter < maxIter )   // (:135)
	{
		if( verbose > 0 ) cout << endl << "Iter = " << iter << " of bounded BFGS search starting with previous F = " << F << "." << endl;

		// 1. search direction (:143-144)
		D.direction( dFdX, p );

		// 2. step length (:148-149)
		double alpha, Fopt;
		if( serialSearch ) serialLineSearchBnd( X, Xlb, Xub, F, dFdX, p, constantX, constantIndicator, alpha, Fopt );
		else cubicInterpolationLineSearchBnd( X, Xlb, Xub, F, dFdX, p, constantX, constantIndicator, alpha, Fopt );

		// 3. update variables and inverse Hessian (:153-174)
		for( int i = 0; i < Nparam; i++ )
		{
			Xprev[i] = X[i];
			X[i] = X[i] + alpha*p[i];
		}
		F = Fopt;
		for( int i = 0; i < Nparam; i++ ) dFdX_prev[i] = dFdX[i];
		objPtr->gradientApproximationMPIRecur( X, dX, dFdX, constantX, constantIndicator );
		for( int i = 0; i < Nparam; i++ )
		{
			s[i] = alpha*p[i];
			g[i] = dFdX[i] - dFdX_prev[i];
		}
		D.update( g, s );

		// 4. boundary (:178)
		boundaryAssessment( F, X, p, dFdX, D, Xlb, Xub, dX, constantX, constantIndicator );

		xdiff = 0;
		for( int i = 0; i < Nparam; i++ ) xdiff += fabs( X[i] - Xprev[i] );   // (:181-184)
		grad2Norm = vector2Norm( dFdX );
		if( verbose > 0 )
			cout << "  Step completed with F = " << F << " and mean abs xdiff is " << xdiff << " and the grad2norm = " << grad2Norm << endl;
		iter = iter + 1;
		totalIter = totalIter + 1;
	}
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:209-397
void BFGS_Bnd_MPI_SW::cubicInterpolationLineSearchBnd( vector <double> & X, vector <double> & Xlb, vector <double> & Xub,
		double FX, vector <double> & dFdX, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
		double & alphaOpt, double & Fopt )
{
	bool bndIndicator = false;
	double alphaMax;
	double phiOpt, dphiOptdalpha;

	alphaOpt = 0;
	phiOpt = FX;
	Fopt = FX;

	double alpha0 = 0;
	double phi0 = FX;
	double dphi0dalpha = dotProd( dFdX, p );

	// Initial alpha pool (:229-256)
	int Npool = Nprocs+1;
	vector <int> evalIndicator( Npool, 1 );
	vector <double> alphaPool( Npool, 0 );
	vector <double> phiPool( Npool, 0 );
	vector <double> dphidalphaPool( Npool, 0 );
	evalIndicator[0] = 0;
	alphaPool[0] = alpha0;
	phiPool[0] = phi0;
	dphidalphaPool[0] = dphi0dalpha;

	alphaMax = computeAlphaBnd( X, Xlb, Xub, p );
	double alphai = alphaGuess;
	if( alphai > alphaMax ) alphai = alphaMax;
	double delta_alpha = alphai/Nprocs;
	for( int i = 1; i < Npool; i++ ) alphaPool[i] = delta_alpha*i;

	int iter_ls = 0;
	bool extendFlag = true;
	bool zoomFlag = false;
	while( iter_ls < maxIterLineSearch && extendFlag )
	{
		evaluateAlphaPoolAndDerivativesIndicator( alphaPool, evalIndicator, X, p, constantX, constantIndicator, phiPool, dphidalphaPool );

		// 1. interval large enough (magnitude) (:276-283)
		for( int i = 1; i < Npool; i++ )
			if( ( phiPool[i] > phi0 + c1*alphaPool[i]*dphi0dalpha ) || ( phiPool[i] >= phiPool[0] && iter_ls > 1 ) )
			{ extendFlag = false; zoomFlag = true; }

		// 2. close enough to the optimum (:288-295)
		for( int i = 1; i < Npool; i++ )
			if( fabs(dphidalphaPool[i]) <= fabs( c2*dphi0dalpha ) )
			{ extendFlag = false; zoomFlag = false; }

		// 3. interval large enough (slope) (:299-307)
		for( int i = 1; i < Npool; i++ )
			if( dphidalphaPool[i] >= 0 )
			{ extendFlag = false; zoomFlag = true; }

		// 4. boundary already met (:310-316)
		if( extendFlag && alphaPool[Npool-1] == alphaMax )
		{ extendFlag = false; zoomFlag = false; bndIndicator = true; }

		// 5. extend (:320-335)
		if( extendFlag )
		{
			double alphaNext = (Nprocs+1)*alphaPool[Npool-1];
			if( alphaNext > alphaMax ) alphaNext = alphaMax;
			double first = alphaPool[Npool-1];
			linspace( first, alphaNext, Npool, alphaPool );
			for( int i = 0; i < Npool; i++ ) evalIndicator[i] = 1;
			evalIndicator[0] = 0;
			phiPool[0] = phiPool[Npool-1];
			dphidalphaPool[0] = dphidalphaPool[Npool-1];
		}
		iter_ls++;
	}

	if( zoomFlag )                                                           // (:345-370)
	{
		double alpha_a, alpha_b, phi_a, phi_b, dphi_a_dalpha, dphi_b_dalpha;
		computeZoomRegion( alphaPool, phiPool, dphidalphaPool, alpha_a, alpha_b, phi_a, phi_b, dphi_a_dalpha, dphi_b_dalpha );
		if( alpha_b - alpha_a > alphaTol )
		{
			lineSearchZoomBnd( alpha_a, alpha_b, phi_a, phi_b, dphi_a_dalpha, dphi_b_dalpha, phi0, dphi0dalpha,
					X, p, constantX, constantIndicator, iter_ls, alphaOpt, phiOpt, dphiOptdalpha );
		}
		else
		{
			double phiMin; int indexMin;
			vectorMin( phiPool, (int) phiPool.size(), phiMin, indexMin );
			alphaOpt = alphaPool[indexMin];
			phiOpt = phiMin;
			dphiOptdalpha = dphidalphaPool[indexMin];
		}
		Fopt = phiOpt;
	}
	else                                                                     // (:371-381)
	{
		double phiMin; int indexMin;
		vectorMin( phiPool, (int) phiPool.size(), phiMin, indexMin );
		alphaOpt = alphaPool[indexMin];
		phiOpt = phiMin;
		dphiOptdalpha = dphidalphaPool[indexMin];
		Fopt = phiOpt;
	}

	if( verbose > 0 )
		cout << ( bndIndicator ? "  ! Line search terminated at boundary with alpha = " : "  Line search completed with alpha = " ) << alphaOpt
		     << " and F = " << Fopt << " after " << iter_ls << " iterations. Note: alphaMax = " << alphaMax << endl;
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:399-431. The reference indexes indexMin-1 / indexMin+1 unguarded; the
// neighbours are clamped into the pool here (they are in range whenever the reference's reads were defined).
void computeZoomRegion( vector <double> & alphaPool, vector <double> & phiPool, vector <double> & dphidalphaPool,
		double & alpha_a, double & alpha_b, double & phi_a, double & phi_b, double & dphi_a_dalpha, double & dphi_b_dalpha )
{
	double phiMin; int indexMin;
	vectorMin( phiPool, (int) phiPool.size(), phiMin, indexMin );
	int last = (int) phiPool.size() - 1;
	int lo, hi;
	if( dphidalphaPool[indexMin] > 0 ) { lo = indexMin-1; hi = indexMin; }
	else { lo = indexMin; hi = indexMin+1; }
	if( lo < 0 ) lo = 0;
	if( hi > last ) hi = last;
	alpha_a = alphaPool[lo]; alpha_b = alphaPool[hi];
	phi_a = phiPool[lo]; phi_b = phiPool[hi];
	dphi_a_dalpha = dphidalphaPool[lo]; dphi_b_dalpha = dphidalphaPool[hi];
}

// Source/BFGS_bnd_linesearch.cpp:733-750
double cubicInterpMinSimple( double alpha_a, double alpha_b, double phi_a, double phi_b, double dphi_a_dalpha, double dphi_b_dalpha )
{
	double d1 = dphi_a_dalpha + dphi_b_dalpha - 3*( phi_a - phi_b )/( alpha_a - alpha_b );
	double d2 = sign( alpha_b - alpha_a )*sqrt( pow(d1,2) - dphi_a_dalpha*dphi_b_dalpha );
	double alphaNew = alpha_b - ( alpha_b - alpha_a )*( dphi_b_dalpha + d2 - d1 )/( dphi_b_dalpha - dphi_a_dalpha + 2*d2 );
	if( alphaNew < alpha_a || alphaNew > alpha_b || alphaNew != alphaNew )
		alphaNew = ( alpha_a + alpha_b )/2;
	return alphaNew;
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:434-482
void computeZoomPool( double alpha_a, double alpha_b, double phi_a, double phi_b, double dphi_a_dalpha, double dphi_b_dalpha,
		vector <double> & alphaPool, vector <double> & phiPool, vector <double> & dphidalphaPool, vector <int> & evalIndicator )
{
	int Npool = (int) alphaPool.size();
	double alpha_c = cubicInterpMinSimple( alpha_a, alpha_b, phi_a, phi_b, dphi_a_dalpha, dphi_b_dalpha );

	if( alpha_c == ( alpha_a + alpha_b )/2 )
	{
		linspace( alpha_a, alpha_b, Npool, alphaPool );
	}
	else
	{
		int Nlinear = Npool-1;
		vector<double> alphaLinear( Nlinear, 0 );
		linspace( alpha_a, alpha_b, Nlinear, alphaLinear );
		alphaPool[0] = alphaLinear[0];
		int iLinear = 1;
		for( int i = 1; i < (int) alphaPool.size(); i++ )
		{
			// iLinear stays in range exactly as in the reference: alpha_c lies in [alpha_a, alpha_b] so it is placed
			// (and consumed) before the linear points run out
			if( iLinear < Nlinear && alpha_c >= alphaLinear[iLinear-1] && alpha_c <= alphaLinear[iLinear] )
			{
				alphaPool[i] = alpha_c;
				alpha_c = -1;
			}
			else
			{
				alphaPool[i] = alphaLinear[iLinear < Nlinear ? iLinear : Nlinear-1];
				iLinear++;
			}
		}
	}

	for( int i = 0; i < Npool; i++ ) evalIndicator[i] = 1;
	phiPool[0] = phi_a;
	dphidalphaPool[0] = dphi_a_dalpha;
	evalIndicator[0] = 0;
	phiPool[Npool-1] = phi_b;
	dphidalphaPool[Npool-1] = dphi_b_dalpha;
	evalIndicator[Npool-1] = 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// The serial class BFGS_Bnd (Source/BFGS_bnd_linesearch.cpp) shares mainBFGSLoop and boundaryAssessment with this class word
// for word (its copies differ only in prints and in calling the non-MPI gradient, which returns the same numbers); what
// differs is the line search: one trial step at a time, bracketing by doubling, then a cubic-interpolation zoom.
// ---------------------------------------------------------------------------------------------------------------------
// Source/BFGS_bnd_linesearch.cpp:207-380
void BFGS_Bnd_MPI_SW::serialLineSearchBnd( vector <double> & X, vector <double> & Xlb, vector <double> & Xub,
		double FX, vector <double> & dFdX, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
		double & alphaOpt, double & Fopt )
{
	bool success = false;
	double dphiOptdalpha;
	double phii = FX;

	alphaOpt = 0;
	Fopt = FX;

	// initial values, with the initial slope from the gradient (:222-224)
	double phi0 = FX;
	double dphi0dalpha = dotProd( dFdX, p );
	double alphaim1 = 0;
	double phiim1 = phi0;
	double dphiim1dalpha = dphi0dalpha;

	double alphaMax = computeAlphaBnd( X, Xlb, Xub, p );                      // (:232)
	double alphai = alphaGuess;
	if( alphai > alphaMax ) alphai = alphaMax;

	int iter_ls = 0;
	while( iter_ls < maxIterLineSearch )
	{
		double dphiidalpha;
		serialPhiAndSlope( alphai, X, p, constantX, constantIndicator, phii, dphiidalpha );

		// 1. sufficient decrease violated, or no longer decreasing: the minimum is bracketed (:266-273)
		if( ( phii > phi0 + c1*alphai*dphi0dalpha ) || ( phii >= phiim1 && iter_ls > 1 ) )
		{
			serialZoomBnd( alphaim1, alphai, phiim1, phii, dphiim1dalpha, dphiidalpha, phi0, dphi0dalpha, X, p, constantX, constantIndicator,
					iter_ls, alphaOpt, Fopt, dphiOptdalpha );
			success = true;
			break;
		}
		// 2. curvature condition holds (:277-283)
		if( fabs( dphiidalpha ) <= fabs( c2*dphi0dalpha ) )
		{
			alphaOpt = alphai; Fopt = phii; success = true;
			break;
		}
		// 3. slope turned positive: bracketed (:287-294)
		if( dphiidalpha >= 0 )
		{
			serialZoomBnd( alphaim1, alphai, phiim1, phii, dphiim1dalpha, dphiidalpha, phi0, dphi0dalpha, X, p, constantX, constantIndicator,
					iter_ls, alphaOpt, Fopt, dphiOptdalpha );
			success = true;
			break;
		}
		// 4. the box was reached (:297-304)
		if( alphai == alphaMax )
		{
			alphaOpt = alphai; Fopt = phii; success = true;
			break;
		}
		alphaim1 = alphai; phiim1 = phii; dphiim1dalpha = dphiidalpha;
		// 5. extend the interval (:314-318)
		alphai = 2*alphai;
		if( alphai > alphaMax ) alphai = alphaMax;
		iter_ls++;
	}

	// ran out of iterations: best of what was seen (:325-343)
	if( !success )
	{
		if( phiim1 < phii ) { alphaOpt = alphaim1; Fopt = phiim1; }
		else if( phi0 < phii ) { alphaOpt = 0; Fopt = phi0; }
		else { alphaOpt = alphai; Fopt = phii; }
	}
	if( verbose > 0 )
		cout << "  Line search completed with alpha = " << alphaOpt << " and F = " << Fopt << " after " << iter_ls << " iterations. Note: alphaMax = " << alphaMax << endl;
}

// one trial step of the serial line search: lineSearchObj + lineSearchFDDerivative (host evaluations, as the reference), or with
// Runtime::setAnalyticSlope(true) phi and its analytic slope from one device call, a bad phi recomputed on the host (the serial reference
// lets NaN/inf flow into its comparisons), the device slope kept
void BFGS_Bnd_MPI_SW::serialPhiAndSlope( double alpha, vector <double> & X, vector <double> & p, vector<double> & constantX,
		vector<bool> & constantIndicator, double & phi, double & dphi )
{
	if( !pnol::Runtime::instance().analyticSlope() )
	{
		phi = lineSearchObj( alpha, X, p, constantX, constantIndicator );
		dphi = lineSearchFDDerivative( alpha, phi, X, p, constantX, constantIndicator );
		return;
	}
	pnol_functor * f = objPtr->deviceFunctor();
	if( !f ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "BFGS_Bnd: the objective has no device functor (no CPU fallback)" );
	vector<unsigned char> ind( constantIndicator.size() );
	for( size_t i = 0; i < ind.size(); i++ ) ind[i] = constantIndicator[i] ? 1 : 0;
	int bad = 0;
	pnol::alphaPoolAnalytic( "BFGS_Bnd", f, X.data(), p.data(), (int) X.size(), &alpha, 1, constantX.data(), ind.data(), (int) constantX.size(),
			&phi, &dphi, &bad );
	if( bad == 0 ) objPtr->noteDeviceEvaluations( 1 );
	else phi = lineSearchObj( alpha, X, p, constantX, constantIndicator );
}

// Source/BFGS_bnd_linesearch.cpp:385-460
void BFGS_Bnd_MPI_SW::serialZoomBnd( double alpha_a, double alpha_b, double phi_a, double phi_b, double dphi_a_dalpha, double dphi_b_dalpha,
		double phi0, double dphi0dalpha, vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
		int & iter_ls, double & alphaOpt, double & phiOpt, double & dphiOptdalpha )
{
	bool success = false;
	while( iter_ls < maxIterLineSearch && ( alpha_b - alpha_a > alphaTol ) )
	{
		// 0. new trial step by cubic interpolation (:396-398)
		double alpha_c = cubicInterpMinSimple( alpha_a, alpha_b, phi_a, phi_b, dphi_a_dalpha, dphi_b_dalpha );
		double phi_c, dphi_c_dalpha;
		serialPhiAndSlope( alpha_c, X, p, constantX, constantIndicator, phi_c, dphi_c_dalpha );

		// 1. shrink the interval from the side with the larger value (:415-431)
		double phi_min = phi_a;
		if( phi_b < phi_a ) phi_min = phi_b;
		if( phi_c > phi0 + c1*alpha_c*dphi0dalpha || phi_c >= phi_min )
		{
			if( phi_a < phi_b ) { alpha_b = alpha_c; phi_b = phi_c; dphi_b_dalpha = dphi_c_dalpha; }
			else { alpha_a = alpha_c; phi_a = phi_c; dphi_a_dalpha = dphi_c_dalpha; }
		}
		else
		{
			// 2. close enough (:435-442)
			if( fabs( dphi_c_dalpha ) <= fabs( c2*dphi0dalpha ) )
			{
				alphaOpt = alpha_c; phiOpt = phi_c; dphiOptdalpha = dphi_c_dalpha;
				success = true;
				break;
			}
			// 3. keep the minimum inside (:445-456)
			if( dphi_c_dalpha < 0 ) { alpha_a = alpha_c; phi_a = phi_c; dphi_a_dalpha = dphi_c_dalpha; }
			else { alpha_b = alpha_c; phi_b = phi_c; dphi_b_dalpha = dphi_c_dalpha; }
		}
		iter_ls++;
	}
	if( !success )                                                           // (:463-477)
	{
		if( phi_a < phi_b ) { alphaOpt = alpha_a; phiOpt = phi_a; dphiOptdalpha = dphi_a_dalpha; }
		else { alphaOpt = alpha_b; phiOpt = phi_b; dphiOptdalpha = dphi_b_dalpha; }
	}
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:484-548
void BFGS_Bnd_MPI_SW::lineSearchZoomBnd( double alpha_a, double alpha_b, double phi_a, double phi_b, double dphi_a_dalpha, double dphi_b_dalpha,
		double phi0, double dphi0dalpha, vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
		int & iter_ls, double & alphaOpt, double & phiOpt, double & dphiOptdalpha )
{
	int Npool = Nprocs+2;
	vector <int> evalIndicator( Npool, 1 );
	vector <double> alphaPool( Npool, 0 );
	vector <double> phiPool( Npool, 0 );
	vector <double> dphidalphaPool( Npool, 0 );

	bool zoomFlag = true;
	bool success = false;
	while( iter_ls < maxIterLineSearch && ( alpha_b - alpha_a > alphaTol ) && zoomFlag )
	{
		computeZoomPool( alpha_a, alpha_b, phi_a, phi_b, dphi_a_dalpha, dphi_b_dalpha, alphaPool, phiPool, dphidalphaPool, evalIndicator );
		evaluateAlphaPoolAndDerivativesIndicator( alphaPool, evalIndicator, X, p, constantX, constantIndicator, phiPool, dphidalphaPool );

		for( int i = 1; i < Npool-1; i++ )
			if( ( phiPool[i] <= phi0 + c1*alphaPool[i]*dphi0dalpha ) && ( fabs(dphidalphaPool[i]) <= fabs( c2*dphi0dalpha ) ) )
			{ zoomFlag = false; success = true; }

		if( !success )
			computeZoomRegion( alphaPool, phiPool, dphidalphaPool, alpha_a, alpha_b, phi_a, phi_b, dphi_a_dalpha, dphi_b_dalpha );
		iter_ls++;
	}

	double phiMin; int indexMin;
	vectorMin( phiPool, (int) phiPool.size(), phiMin, indexMin );
	alphaOpt = alphaPool[indexMin];
	phiOpt = phiMin;
	dphiOptdalpha = dphidalphaPool[indexMin];
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:552-594: compact the pool to the entries that need evaluation, evaluate, scatter back
void BFGS_Bnd_MPI_SW::evaluateAlphaPoolAndDerivativesIndicator( vector <double> & alphaPool, vector<int> evalIndicator,
		vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
		vector <double> & phiPool, vector <double> & dphidalphaPool )
{
	vector <double> alphaPoolTemp, phiPoolTemp, dphidalphaPoolTemp;
	for( size_t i = 0; i < evalIndicator.size(); i++ )
		if( evalIndicator[i] == 1 )
		{
			alphaPoolTemp.push_back( alphaPool[i] );
			phiPoolTemp.push_back( phiPool[i] );
			dphidalphaPoolTemp.push_back( dphidalphaPool[i] );
		}
	evaluateAlphaPoolAndDerivatives( alphaPoolTemp, X, p, constantX, constantIndicator, phiPoolTemp, dphidalphaPoolTemp );
	int idxTemp = 0;
	for( size_t i = 0; i < evalIndicator.size(); i++ )
		if( evalIndicator[i] == 1 )
		{
			alphaPool[i] = alphaPoolTemp[idxTemp];
			phiPool[i] = phiPoolTemp[idxTemp];
			dphidalphaPool[i] = dphidalphaPoolTemp[idxTemp];
			idxTemp++;
		}
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:599-699: the whole pool (phi and its forward-difference slope, 2 evaluations
// per entry) is ONE kernel launch; NaN/inf values come back as the 1e10 sentinel, which ends the optimisation.
// (The reference only tests phi for NaN, :657-668; the kernel also guards the slope and counts both.)
void BFGS_Bnd_MPI_SW::evaluateAlphaPoolAndDerivatives( vector <double> & alphaPool, vector <double> & X, vector <double> & p,
		vector<double> & constantX, vector<bool> & constantIndicator, vector <double> & phiPool, vector <double> & dphidalphaPool )
{
	int N = (int) alphaPool.size();
	if( N == 0 ) return;
	pnol::Runtime & rt = pnol::Runtime::instance();
	pnol_functor * f = objPtr->deviceFunctor();
	if( !f ) throw pnol::Error( PNOL_ERR_NO_FUNCTOR, "BFGS_Bnd_MPI_SW: the objective has no device functor (no CPU fallback)" );
	vector<unsigned char> ind( constantIndicator.size() );
	for( size_t i = 0; i < ind.size(); i++ ) ind[i] = constantIndicator[i] ? 1 : 0;
	int bad = 0;
	if( rt.analyticSlope() )
	{
		// Runtime::setAnalyticSlope(true): phi and its analytic slope, one evaluation per entry
		pnol::alphaPoolAnalytic( "BFGS_Bnd_MPI_SW", f, X.data(), p.data(), (int) X.size(), alphaPool.data(), N, constantX.data(), ind.data(),
				(int) constantX.size(), phiPool.data(), dphidalphaPool.data(), &bad );
		objPtr->noteDeviceEvaluations( N );
	}
	else
	{
		rt.check( pnol_alpha_pool( rt.ctx(), f, X.data(), p.data(), (int) X.size(), alphaPool.data(), N, dalpha, nullptr,
				constantX.data(), ind.data(), (int) constantX.size(), phiPool.data(), dphidalphaPool.data(), &bad ) );
		objPtr->noteDeviceEvaluations( 2LL*N );                              // lineSearchObj + lineSearchFDDerivative per entry (:629-640)
	}
	for( int i = 0; i < N; i++ )
		if( phiPool[i] == 1e10 )
		{
			cout << "Line search crashed ... ending search..." << endl;
			optimFlag = false;                                               // (:684-693)
		}
}

double BFGS_Bnd_MPI_SW::lineSearchObj( double alpha, vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator )
{
	vector <double> Xalphap( X.size(), 0 );
	for( size_t i = 0; i < X.size(); i++ ) Xalphap[i] = X[i] + alpha*p[i];
	return objPtr->objEvalRecur( Xalphap, constantX, constantIndicator );
}

double BFGS_Bnd_MPI_SW::lineSearchFDDerivative( double alpha, double phialpha, vector <double> & X, vector <double> & p,
		vector<double> & constantX, vector<bool> & constantIndicator )
{
	vector <double> Xalphap_dalpha( X.size(), 0 );
	for( size_t i = 0; i < X.size(); i++ ) Xalphap_dalpha[i] = X[i] + (alpha+dalpha)*p[i];
	double Falpha_dalpha = objPtr->objEvalRecur( Xalphap_dalpha, constantX, constantIndicator );
	return ( Falpha_dalpha - phialpha )/dalpha;
}

// Source/BFGS_bnd_linesearch_MPI_SW.cpp:741-967
void BFGS_Bnd_MPI_SW::boundaryAssessment( double & F, vector <double> & X, vector <double> & p, vector<double> & dFdX, pnol::InverseHessian & D,
		vector <double> & Xlb, vector <double> & Xub, vector<double> & dX, vector<double> & constantX, vector<bool> & constantIndicator )
{
	vector<int> idxCurrRecur;
	int Ndim_current = (int) X.size();
	vector <double> constantX_current( Ndim_current, 0 );
	vector <bool> constantIndicator_current( Ndim_current, false );
	int Ndim = (int) constantX.size();
	bool bndFlag = false;

	// 1. freeze variables sitting on a bound whose search / steepest-descent direction points outward (:755-786)
	int iCurrent = 0;
	for( int i = 0; i < Ndim; i++ )
	{
		if( !constantIndicator[i] )
		{
			if( ( fabs(X[iCurrent] - Xlb[iCurrent]) < bndTol ) && ( (p[iCurrent] < 0) || (dFdX[iCurrent] > 0) ) )
			{
				bndFlag = true;
				constantIndicator[i] = true;
				constantX[i] = X[iCurrent];
				constantIndicator_current[iCurrent] = true;
				constantX_current[iCurrent] = X[iCurrent];
				idxCurrRecur.push_back( i );
			}
			else if( ( fabs(X[iCurrent] - Xub[iCurrent]) < bndTol ) && ( (p[iCurrent] > 0) || (dFdX[iCurrent] < 0) ) )
			{
				bndFlag = true;
				constantIndicator[i] = true;
				constantX[i] = X[iCurrent];
				constantIndicator_current[iCurrent] = true;
				constantX_current[iCurrent] = X[iCurrent];
				idxCurrRecur.push_back( i );
			}
			iCurrent++;
		}
	}

	int Nconst = 0;
	for( size_t i = 0; i < constantIndicator.size(); i++ ) Nconst = Nconst + constantIndicator[i];

	int NdimRecur = Ndim - Nconst;
	if( bndFlag && NdimRecur > 0 )
	{
		double FRecur = F;
		vector <double> XRecur( NdimRecur, 0 ), dFdXRecur( NdimRecur, 0 ), XlbRecur( NdimRecur, 0 ), XubRecur( NdimRecur, 0 ), dXRecur( NdimRecur, 0 );

		int irecur = 0;
		for( iCurrent = 0; iCurrent < Ndim_current; iCurrent++ )             // (:826-839)
			if( !constantIndicator_current[iCurrent] )
			{
				FRecur = F;
				XRecur[irecur] = X[iCurrent];
				dFdXRecur[irecur] = dFdX[iCurrent];
				XlbRecur[irecur] = Xlb[iCurrent];
				XubRecur[irecur] = Xub[iCurrent];
				dXRecur[irecur] = dX[iCurrent];
				irecur++;
			}

		// start the reduced problem from (scaled) steepest descent (:841-854)
		pnol::InverseHessian DRecur( NdimRecur );
		if( initialScalingVec.size() > 0 )
		{
			vector<double> diag( NdimRecur, 1.0 );
			int j = 0;
			for( int i = 0; i < Ndim; i++ )
				if( !constantIndicator[i] ) { if( j < NdimRecur ) diag[j] = initialScalingVec[i]; j++; }
			DRecur.setDiagonal( diag );
		}
		else DRecur.setIdentity();

		// 2. recursive solve on the free variables (:857-858)
		recurFlag = true;
		mainBFGSLoop( FRecur, XRecur, dFdXRecur, DRecur, XlbRecur, XubRecur, dXRecur, constantX, constantIndicator );

		// 3. scatter back (:862-876)
		irecur = 0;
		for( iCurrent = 0; iCurrent < Ndim_current; iCurrent++ )
			if( !constantIndicator_current[iCurrent] )
			{
				F = FRecur;
				X[iCurrent] = XRecur[irecur];
				dFdX[iCurrent] = dFdXRecur[irecur];
				Xlb[iCurrent] = XlbRecur[irecur];
				Xub[iCurrent] = XubRecur[irecur];
				dX[iCurrent] = dXRecur[irecur];
				irecur++;
			}

		for( size_t k = 0; k < idxCurrRecur.size(); k++ ) constantIndicator[idxCurrRecur[k]] = false;   // (:879-882)

		// reset D to the (scaled) identity (:885-895); the scaling loop walks the NON-constant variables with its own
		// counter, as the reference does
		if( initialScalingVec.size() > 0 )
		{
			vector<double> diag( Ndim_current, 1.0 );
			int j = 0;
			for( int i = 0; i < Ndim; i++ )
				if( !constantIndicator[i] ) { if( j < Ndim_current ) diag[j] = initialScalingVec[i]; j++; }
			D.setDiagonal( diag );
		}
		else D.setIdentity();

		// 4. gradient of the original variables (:899)
		objPtr->gradientApproximationMPIRecur( X, dX, dFdX, constantX, constantIndicator );

		// 5. can the solution continue into the interior? (:903-919)
		bool continueFlag = false;
		for( iCurrent = 0; iCurrent < Ndim_current; iCurrent++ )
			if( constantIndicator_current[iCurrent] )
			{
				if( ( fabs(X[iCurrent] - Xlb[iCurrent]) < bndTol ) && ( dFdX[iCurrent] < 0 ) ) continueFlag = true;
				else if( ( fabs(X[iCurrent] - Xub[iCurrent]) < bndTol ) && ( dFdX[iCurrent] > 0 ) ) continueFlag = true;
			}

		Nconst = 0;
		for( size_t i = 0; i < constantIndicator.size(); i++ ) Nconst = Nconst + constantIndicator[i];
		if( Nconst == 0 ) recurFlag = false;

		optimFlag = continueFlag;                                            // (:930-950)
	}
	else if( NdimRecur == 0 )
	{
		optimFlag = false;                                                   // (:954-963)
	}
}
