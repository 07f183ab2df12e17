#pragma once
// ml::EM: Gaussian-mixture expectation-maximisation with the reference's public surface
// (ML/EM.hpp:18-166) on the B200 backend.  fit() copies the data to HBM (sharded over the GPUs of
// the process-wide context), runs the fused E+M kernel once per iteration through the C-ABI of
// include/mlb200.h, and keeps the initialisers, the pseudo-random stream and the convergence test
// on the host exactly as the reference does (ML/EM.cpp:91-174).
//
// Differences from the reference header, all additive:
//   - number_iterations(): iterations run by the last fit (requested by the north star; the
//     reference does not store it);
//   - assign_responsibilities(points): the batched form of assign_responsibilities(x, u), on the device;
//   - log_likelihoods(points), log_likelihood(points), log_likelihoods() and final_log_likelihood(): log p(x) under the
//     returned parameters, per point and as a mean, for new points or the fitted ones, on the device;
//   - the built-in KPP and ClosestCentroid initialisers run their O(N K D) distance passes on the device (the draws
//     stay on the host with the model's PRNG, so the initial state is the reference's);
//   - responsibilities() and labels() are out of line: the N x K matrix (25.6 GB at N=1e8, K=32) and the N labels
//     (400 MB) stay on the device until first asked for, then are materialised once; the values are the reference's;
//   - shapes: any K; D <= 128 (the device refresh of a component factorises its D x D covariance inside one SM);
//     larger D makes fit() throw std::invalid_argument.
#include <memory>
#include <random>
#include <vector>
#include <Eigen/Core>
#include "Clustering.hpp"
#include "dll.hpp"

namespace ml
{
	namespace detail { class EmDevice; }

	class EM: public Clustering::Model
	{
	public:
		/** @throw std::invalid_argument If `number_components` is zero. */
		DLL_DECLSPEC EM(unsigned int number_components);
		DLL_DECLSPEC ~EM() override;
		EM(const EM&) = delete;
		EM& operator=(const EM&) = delete;

		DLL_DECLSPEC void set_seed(unsigned int seed);

		/** @throw std::domain_error If negative. */
		DLL_DECLSPEC void set_absolute_tolerance(double absolute_tolerance);

		/** @throw std::domain_error If negative. */
		DLL_DECLSPEC void set_relative_tolerance(double relative_tolerance);

		/** @throw std::invalid_argument If less than 2. */
		DLL_DECLSPEC void set_maximum_steps(unsigned int maximum_steps);

		/** @throw std::invalid_argument If null. */
		DLL_DECLSPEC void set_means_initialiser(std::shared_ptr<const Clustering::CentroidsInitialiser> means_initialiser);

		/** @throw std::invalid_argument If null. */
		DLL_DECLSPEC void set_responsibilities_initialiser(std::shared_ptr<const Clustering::ResponsibilitiesInitialiser> responsibilities_initialiser);

		void set_verbose(bool verbose)
		{
			verbose_ = verbose;
		}

		/** Start from an M-step on initial responsibilities instead of from initial means. */
		void set_maximise_first(bool maximise_first)
		{
			maximise_first_ = maximise_first;
		}

		/** @throw std::invalid_argument If data has no rows or fewer columns than components. */
		DLL_DECLSPEC bool fit(DataView data) override;

		auto number_components() const { return number_components_; }

		unsigned int number_clusters() const override { return number_components(); }

		/** D x K. */
		const auto& means() const { return means_; }

		const Eigen::MatrixXd& centroids() const override { return means(); }

		const auto& covariances() const { return covariances_; }

		/** @throw std::invalid_argument If k is out of range. */
		DLL_DECLSPEC const Eigen::MatrixXd& covariance(unsigned int k) const;

		const auto& mixing_probabilities() const { return mixing_probabilities_; }

		/** N x K, from the last E-step of the fit. */
		DLL_DECLSPEC const Eigen::MatrixXd& responsibilities() const;

		/** Mean log-likelihood per point at the parameters of the last E-step of the fit (before its M-step). */
		double log_likelihood() const { return log_likelihood_; }

		/** log p(x) = log sum_k w_k N(x | mu_k, Sigma_k) of every column of `points` (D x m) under the current parameters,
		on the device.
		@throw std::invalid_argument If `points` has the wrong number of rows.
		@throw std::logic_error If there is no fitted device state (no fit yet, the N == K exact fit, or after release_device()). */
		DLL_DECLSPEC Eigen::VectorXd log_likelihoods(DataView points) const;

		/** The mean of log_likelihoods(points).
		@throw std::invalid_argument If `points` has the wrong number of rows.
		@throw std::logic_error If there is no fitted device state. */
		DLL_DECLSPEC double log_likelihood(DataView points) const;

		/** log p(x) of every fitted point (this process's own points under ml::Distributed) under the current parameters.
		@throw std::logic_error If there is no fitted device state. */
		DLL_DECLSPEC Eigen::VectorXd log_likelihoods() const;

		/** The mean log-likelihood of the fitted points at the parameters the fit returned (log_likelihood() belongs to the
		parameters before the last M-step).  Under ml::Distributed: over all ranks' points, and collective.
		@throw std::logic_error If there is no fitted device state. */
		DLL_DECLSPEC double final_log_likelihood() const;

		std::shared_ptr<const Clustering::CentroidsInitialiser> means_initialiser() const { return means_initialiser_; }

		/** Responsibilities of the fitted components for a point x (u must have K entries).
		@throw std::invalid_argument On size mismatch. */
		DLL_DECLSPEC void assign_responsibilities(PointView x, VectorOut u) const;

		/** The same for every column of `points` (D x m) at once, on the device: m x K.
		@throw std::invalid_argument If `points` has the wrong number of rows.
		@throw std::logic_error If there is no fitted device state (no fit yet, or the N == K exact fit). */
		DLL_DECLSPEC Eigen::MatrixXd assign_responsibilities(DataView points) const;

		/** Brought from the device on first access after a converged fit; like the reference, a fit that did not
		converge leaves no meaningful labels (N zeros). */
		DLL_DECLSPEC const std::vector<unsigned int>& labels() const override;

		bool converged() const override { return converged_; }

		/** Iterations (E-step + M-step pairs) executed by the last fit. */
		unsigned int number_iterations() const { return number_iterations_; }

		/** Frees the HBM-resident state of the last fit (the points, 8 D bytes each, stay on the device after fit() so that
		responsibilities(), labels() and the batched assign_responsibilities() can be served).  `keep_results`: bring the
		pending responsibilities and labels to the host first.  The batched prediction needs a new fit afterwards. */
		DLL_DECLSPEC void release_device(bool keep_results = true);
	private:
		Prng prng_;
		std::shared_ptr<const Clustering::CentroidsInitialiser> means_initialiser_;
		std::shared_ptr<const Clustering::ResponsibilitiesInitialiser> responsibilities_initialiser_;
		Eigen::VectorXd mixing_probabilities_;
		Eigen::MatrixXd means_; /**< D x K */
		mutable Eigen::MatrixXd responsibilities_; /**< N x K, materialised on demand */
		mutable bool responsibilities_on_host_;
		std::vector<Eigen::MatrixXd> covariances_; /**< K matrices D x D */
		std::vector<Eigen::MatrixXd> inverse_covariances_;
		Eigen::VectorXd sqrt_covariance_determinants_;
		mutable std::vector<unsigned int> labels_;
		mutable bool labels_on_host_;
		Eigen::Index sample_size_;
		double absolute_tolerance_;
		double relative_tolerance_;
		double log_likelihood_;
		unsigned int number_components_;
		unsigned int maximum_steps_;
		unsigned int number_iterations_;
		bool verbose_;
		bool maximise_first_;
		bool converged_;
		mutable std::unique_ptr<detail::EmDevice> device_; /**< HBM-resident state of the last fit */

		void initialise_centroids(const Clustering::CentroidsInitialiser& initialiser, DataView data, MatrixOut centroids);
		void process_covariances(Eigen::Index number_dimensions);
		void fetch_parameters(Eigen::Index number_dimensions);
	};
}
