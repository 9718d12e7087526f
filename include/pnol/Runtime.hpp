/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * Runtime.hpp -- process-wide device runtime behind the PNOL plugin classes.
 *
 * The reference's algorithm classes find their "parallel machine" implicitly through MPI_COMM_WORLD
 * (e.g. /root/reference/Source/LevenbergMarquardtMPI.cpp:15-17). Here the implicit machine is one pnol_ctx
 * (one B200, optionally one rank of an NCCL communicator) owned by pnol::Runtime. Launchers that already hold a
 * context (bench.py, tests, a torchrun rank) attach it; otherwise one is created on first use on device
 * $PNOL_DEVICE (else $LOCAL_RANK, else 0).
 */
#ifndef PNOL_RUNTIME_HPP_
#define PNOL_RUNTIME_HPP_

#include <stdexcept>
#include <string>
#include <vector>

#include "../pnol_b200.h"

namespace pnol {

class Error : public std::runtime_error {
  public:
	Error(int status, const std::string & what) : std::runtime_error(what), status_(status) {}
	int status() const { return status_; }
  private:
	int status_;
};

class Runtime {
  public:
	static Runtime & instance();
	pnol_ctx * ctx();                         // creates the context on first use; throws pnol::Error without a GPU
	void attach(pnol_ctx * ctx);              // use a caller-owned context (not destroyed by the runtime)
	void reset();                             // drop (and destroy if owned) the current context
	// width of the alpha pools of the pooled line searches: the reference ties it to the MPI rank count
	// (Source/BFGS_bnd_linesearch_MPI_SW.cpp:229, BFGS_with_linesearch_MPI.cpp:235); here it is a parameter
	// ($PNOL_POOL_WIDTH, default 8) independent of the GPU count.
	int poolWidth() const { return poolWidth_; }
	void setPoolWidth(int w) { poolWidth_ = w < 1 ? 1 : w; }
	// random stream used by the genetic algorithms (replaces srand(time(0)) + timeRand(),
	// Source/GeneticAlgorithmMPI.cpp:57,66)
	void setRandomStream(const pnol_stream_desc & s) { stream_ = s; haveStream_ = true; }
	void clearRandomStream() { haveStream_ = false; }   // back to the default (clock-seeded, rank-0-broadcast) stream
	bool haveRandomStream() const { return haveStream_; }
	const pnol_stream_desc & randomStream() const { return stream_; }
	// The stream an algorithm uses when the caller set none: srand((unsigned) time(0)) of the reference
	// (Source/GeneticAlgorithmMPI.cpp:57, Source/SimplexSearch.cpp:57) as a clock-seeded counter stream. The reference takes
	// every random decision from ROOT (zero-and-Allreduce of the population, Source/GeneticAlgorithmMPI.cpp:300-330), so ranks
	// seeded from their own clocks are harmless there; here every rank replays the same stream, so the seed is drawn on rank 0
	// and broadcast over the context's communicator (a collective call: all ranks enter the algorithm together, as in the reference).
	pnol_stream_desc defaultStream(double scale);
	// BFGS inverse-Hessian update form (PNOL_HINV_RANK2 default, PNOL_HINV_LITERAL = the reference's two products)
	int hessianUpdateMode() const { return hinvMode_; }
	void setHessianUpdateMode(int m) { hinvMode_ = m; }
	// Jacobian mode of LevMarq[MPI]::findMin and MultiObjective::gradientApproximation: PNOL_JAC_AUTO (default) / PNOL_JAC_BLACKBOX /
	// PNOL_JAC_STRUCTURED forward differences, or PNOL_JAC_ANALYTIC: the model's own derivative (R::jacobian, include/pnol/functors.hpp;
	// a model without one makes the call fail with PNOL_ERR_NO_FUNCTOR)
	int jacobianMode() const { return jacMode_; }
	void setJacobianMode(int m) { jacMode_ = m; }
	// LM: keep J^T J across a rejected step (X restored, so J is unchanged). The reference recomputes the identical J
	// (Source/LevenbergMarquardtMPI.cpp:60 after :120-129); false reproduces that work, the results are the same.
	bool jacobianCache() const { return jacCache_; }
	void setJacobianCache(bool on) { jacCache_ = on; }
	// LM: keep the whole Jacobian in HBM (default), or sum the normal equations over row blocks and never store J
	// (SURVEY.md 8(f) item 2: work space 512 MB instead of m*n*8 bytes; same iterates up to the summation order of J^T J)
	bool storeJacobian() const { return storeJ_; }
	void setStoreJacobian(bool on) { storeJ_ = on; }
	// Gradients of Objective::gradientApproximation[MPI][Recur] (hence of BFGS, BFGS_MPI, BFGS_Bnd, BFGS_Bnd_MPI_SW, BFGSBnd_MPI): the
	// forward difference (false, default) or the objective's own derivative (true: pnol_gradient[_recur] from F::partial,
	// include/pnol/functors.hpp; dX is ignored, an objective without one makes the call fail with PNOL_ERR_NO_FUNCTOR). In the analytic
	// mode a gradient evaluates no objective value, so the evaluation counts the classes report (getEvals(), "function evaluations")
	// count objective evaluations only.
	bool analyticGradient() const { return gradAnalytic_; }
	void setAnalyticGradient(bool on) { gradAnalytic_ = on; }
	// Hessians of Objective::hessianApproximation (hence initHessFD of the five BFGS classes): the forward difference (false, default)
	// or the objective's own second derivative (true: pnol_hessian from F::partial2, include/pnol/functors.hpp; dX is ignored, an
	// objective without one makes the call fail with PNOL_ERR_NO_FUNCTOR). A switch of its own: a functor may define partial() without
	// partial2(). In the analytic mode a Hessian evaluates no objective value and adds nothing to the evaluation counts.
	bool analyticHessian() const { return hessAnalytic_; }
	void setAnalyticHessian(bool on) { hessAnalytic_ = on; }
	// Line-search slopes phi'(alpha) = d/dalpha f(X + alpha p) of BFGS, BFGS_Bnd and BFGS_Bnd_MPI_SW: the forward difference with their
	// dalpha (false, default) or p . grad f(X + alpha p) from the objective's own derivative (true: pnol_alpha_pool_analytic from
	// F::partial, include/pnol/functors.hpp; dalpha is ignored, an objective without one makes the call fail with PNOL_ERR_NO_FUNCTOR).
	// Meant to be used together with setAnalyticGradient(true): the strong-Wolfe tests compare every phi'(alpha) with the slope at 0,
	// p . dFdX, which then has the same bits as the analytic slope at alpha = 0. A switch of its own, so that the analytic gradient alone
	// keeps its iterates. In the analytic mode a pool entry counts one objective evaluation instead of two. BFGS_MPI and BFGSBnd_MPI
	// use values only and are not affected.
	bool analyticSlope() const { return slopeAnalytic_; }
	void setAnalyticSlope(bool on) { slopeAnalytic_ = on; }
	void check(int status) const;             // throws pnol::Error with pnol_last_error() text
  private:
	Runtime();
	~Runtime();
	pnol_ctx * ctx_;
	bool owned_;
	int poolWidth_;
	pnol_stream_desc stream_;
	bool haveStream_;
	int hinvMode_;
	int jacMode_;
	bool jacCache_;
	bool storeJ_ = true;
	bool gradAnalytic_ = false;
	bool hessAnalytic_ = false;
	bool slopeAnalytic_ = false;
};

// RAII local (non-collective) mode for the serial classes: the reference's BFGS, BFGS_Bnd, LevMarq, GeneticAlgorithm and the
// non-MPI stencil members never call MPI (a program may run them on one rank only), so nothing under this scope may issue a
// collective even when the context carries a communicator (pnol_comm_set_local).
class LocalScope {
  public:
	LocalScope() : ctx_(Runtime::instance().ctx()), prev_(pnol_comm_set_local(ctx_, 1)) {}
	~LocalScope() { pnol_comm_set_local(ctx_, prev_); }
	LocalScope(const LocalScope &) = delete;
	LocalScope & operator=(const LocalScope &) = delete;
  private:
	pnol_ctx * ctx_;
	int prev_;
};

// RAII device functor (the device twin an Objective / MultiObjective hands to the algorithms)
class DeviceFunctor {
  public:
	DeviceFunctor() : f_(nullptr) {}
	~DeviceFunctor() { release(); }
	DeviceFunctor(const DeviceFunctor &) = delete;
	DeviceFunctor & operator=(const DeviceFunctor &) = delete;
	// (re)creates the functor when none exists yet
	pnol_functor * get(int kind, const std::vector<double> & scalars = std::vector<double>(),
	                   const std::vector<long long> & ints = std::vector<long long>(),
	                   const std::vector<const double *> & columns = std::vector<const double *>(), long long m = 0);
	void release();
  private:
	pnol_functor * f_;
};

// RAII device array of doubles
class DeviceArray {
  public:
	DeviceArray() : p_(nullptr), n_(0) {}
	explicit DeviceArray(size_t n) : p_(nullptr), n_(0) { resize(n); }
	~DeviceArray() { free(); }
	DeviceArray(const DeviceArray &) = delete;
	DeviceArray & operator=(const DeviceArray &) = delete;
	void resize(size_t n);
	void free();
	double * data() const { return p_; }
	size_t size() const { return n_; }
	void upload(const double * host, size_t n);
	void download(double * host, size_t n) const;
	void swap(DeviceArray & o) { double * p = p_; p_ = o.p_; o.p_ = p; size_t n = n_; n_ = o.n_; o.n_ = n; }
  private:
	double * p_;
	size_t n_;
};

} // namespace pnol

#endif
