/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * BFGS_bnd_linesearch_MPI_SW.hpp -- BFGS_Bnd_MPI_SW: box-bounded BFGS with a pooled strong-Wolfe line search and
 * active-set recursion. Interface of /root/reference/Source/BFGS_bnd_linesearch_MPI_SW.hpp:29-164 (setParams order
 * included: bndTol sits between maxIterLineSearch and dXGrad). The reference sizes its step-length pools by the MPI
 * rank count (Source/BFGS_bnd_linesearch_MPI_SW.cpp:229, 252, 322, 490); here that number is poolWidth.
 */
#ifndef PNOL_BFGS_BND_LINESEARCH_MPI_SW_HPP_
#define PNOL_BFGS_BND_LINESEARCH_MPI_SW_HPP_

#include <vector>

#include "UtilityFunctions.hpp"
#include "PNOL_Algorithm.hpp"
#include "BFGS_with_linesearch.hpp"
#include "Box_boundary_functions.hpp"

using namespace std;

class BFGS_Bnd_MPI_SW : public AlgorithmBnd {
  private:
	double c1, c2;
	double dalpha;
	double alphaGuess;
	double alphaTol;
	double alphaMult;
	int maxIterLineSearch;
	double bndTol;
	double dXGrad;
	double dXHess;
	double xMinDiff;
	double minGrad2Norm;
	vector<double> dXGradVec;
	vector<double> initialScalingVec;
	int maxIter;
	int totalIter;
	bool initHessFD;
	int verbose;
	int Nprocs;             // pool width ("number of processes" of the reference)
	int procID;
	bool optimFlag;
	int recurFlag;
	bool serialSearch;      // true: one step length at a time, the line search of the serial class BFGS_Bnd

	// the line search of Source/BFGS_bnd_linesearch.cpp (:207-380 and :385-460), used by class BFGS_Bnd
	void serialLineSearchBnd( vector <double> & X, vector <double> & Xlb, vector <double> & Xub,
			double FX, vector <double> & dFdX, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
			double & alphaOpt, double & Fopt );
	void serialZoomBnd( double alpha_a, double alpha_b, double phi_a, double phi_b, double dphi_a_dalpha, double dphi_b_dalpha,
			double phi0, double dphi0dalpha, vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
			int & iter_ls, double & alphaOpt, double & phiOpt, double & dphiOptdalpha );
	// phi(alpha) and its slope for the serial line search: forward difference, or analytic (Runtime::setAnalyticSlope)
	void serialPhiAndSlope( double alpha, vector <double> & X, vector <double> & p, vector<double> & constantX,
			vector<bool> & constantIndicator, double & phi, double & dphi );

  public:
	void findMinBnd( vector <double> & X, vector <double> & Xlb, vector <double> & Xub, double & f0, double & fOpt );
	void mainBFGSLoop( double & F, vector <double> & X, vector<double> & dFdX, pnol::InverseHessian & D,
			vector <double> & Xlb, vector <double> & Xub, vector<double> & dX, vector<double> & constantX,
			vector<bool> & constantIndicator );
	void evaluateAlphaPoolAndDerivativesIndicator( vector <double> & alphaPool, vector<int> evalIndicator,
			vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
			vector <double> & phiPool, vector <double> & dphidalphaPool );
	void evaluateAlphaPoolAndDerivatives( vector <double> & alphaPool, vector <double> & X, vector <double> & p,
			vector<double> & constantX, vector<bool> & constantIndicator, vector <double> & phiPool, vector <double> & dphidalphaPool );
	double lineSearchObj( double alpha, vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator );
	double lineSearchFDDerivative( double alpha, double phialpha, vector <double> & X, vector <double> & p,
			vector<double> & constantX, vector<bool> & constantIndicator );
	void lineSearchZoomBnd( double alpha_a, double alpha_b, double phi_a, double phi_b, double dphi_a_dalpha, double dphi_b_dalpha,
			double phi0, double dphi0dalpha, vector <double> & X, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
			int & iter_ls, double & alphaOpt, double & phiOpt, double & dphiOptdalpha );
	void cubicInterpolationLineSearchBnd( vector <double> & X, vector <double> & Xlb, vector <double> & Xub,
			double FX, vector <double> & dFdX, vector <double> & p, vector<double> & constantX, vector<bool> & constantIndicator,
			double & alphaOpt, double & Fopt );
	void boundaryAssessment( double & F, vector <double> & X, vector <double> & p, vector<double> & dFdX, pnol::InverseHessian & D,
			vector <double> & Xlb, vector <double> & Xub, vector<double> & dX, vector<double> & constantX, vector<bool> & constantIndicator );

	void setParams( double c1In, double c2In, double dalphaIn, double alphaGuessIn, double alphaTolIn, double alphaMultIn,
			int maxIterLineSearchIn, double bndTolIn, double dXGradIn, double dXHessIn, double maxIterIn,
			double xMinDiffIn, double minGrad2NormIn, bool initHessFDIn, int verboseIn )
	{
		c1 = c1In; c2 = c2In; dalpha = dalphaIn; alphaGuess = alphaGuessIn; alphaTol = alphaTolIn; alphaMult = alphaMultIn;
		maxIterLineSearch = maxIterLineSearchIn; bndTol = bndTolIn; dXGrad = dXGradIn; dXHess = dXHessIn; maxIter = maxIterIn;
		xMinDiff = xMinDiffIn; minGrad2Norm = minGrad2NormIn; initHessFD = initHessFDIn; verbose = verboseIn;
	}
	void setPoolWidth( int w ){ Nprocs = w < 1 ? 1 : w; }
	void setSerialLineSearch( bool on ){ serialSearch = on; }
	int iterations() const { return totalIter; }

	BFGS_Bnd_MPI_SW();

	void setGradVec( vector <double> & dXGradVecIn ){ dXGradVec = dXGradVecIn; }
	void setinitialScalingVec( vector <double> & initialScalingVecIn ){ initialScalingVec = initialScalingVecIn; }

	~BFGS_Bnd_MPI_SW(){}
};

void computeZoomRegion( vector <double> & alphaPool, vector <double> & phiPool, vector <double> & dphidalphaPool,
		double & alpha_a, double & alpha_b, double & phi_a, double & phi_b, double & dphi_a_dalpha, double & dphi_b_dalpha );
void computeZoomPool( double alpha_a, double alpha_b, double phi_a, double phi_b, double dphi_a_dalpha, double dphi_b_dalpha,
		vector <double> & alphaPool, vector <double> & phiPool, vector <double> & dphidalphaPool, vector <int> & evalIndicator );
double cubicInterpMinSimple( double alpha_lo, double alpha_hi, double phi_lo, double phi_hi, double dphi_lo_dalpha, double dphi_hi_dalpha );

#endif
