// ml::EM on the B200 backend.  The control flow, defaults, error behaviour and result semantics
// follow ML/EM.cpp:18-174; the E-step, M-step, covariance refresh, sample covariance and label
// extraction (EM.cpp:190-304) run on the device behind include/mlb200.h.
#include "ML/EM.hpp"

#include <algorithm>
#include <cmath>
#include <iostream>
#include <limits>
#include <stdexcept>
#include <typeinfo>

#include "Backend.hpp"
#include "ML/LinearAlgebra.hpp"

namespace ml
{
	EM::EM(const unsigned int number_components)
		: means_initialiser_(std::make_shared<Clustering::Forgy>())
		, responsibilities_initialiser_(std::make_shared<Clustering::ClosestCentroid>(means_initialiser_))
		, mixing_probabilities_(number_components)
		, responsibilities_on_host_(true)
		, covariances_(number_components)
		, inverse_covariances_(number_components)
		, sqrt_covariance_determinants_(number_components)
		, labels_on_host_(true)
		, sample_size_(0)
		, absolute_tolerance_(1e-8)
		, relative_tolerance_(1e-8)
		, log_likelihood_(0)
		, number_components_(number_components)
		, maximum_steps_(1000)
		, number_iterations_(0)
		, verbose_(false)
		, maximise_first_(false)
		, converged_(false)
	{
		if (!number_components) {
			throw std::invalid_argument("EM: At least one component required");
		}
	}

	EM::~EM() = default;

	void EM::set_seed(unsigned int seed)
	{
		prng_.seed(seed);
	}

	void EM::set_absolute_tolerance(double absolute_tolerance)
	{
		if (absolute_tolerance < 0) {
			throw std::domain_error("EM: Negative absolute tolerance");
		}
		absolute_tolerance_ = absolute_tolerance;
	}

	void EM::set_relative_tolerance(double relative_tolerance)
	{
		if (relative_tolerance < 0) {
			throw std::domain_error("EM: Negative relative tolerance");
		}
		relative_tolerance_ = relative_tolerance;
	}

	void EM::set_maximum_steps(unsigned int maximum_steps)
	{
		if (maximum_steps < 2) {
			throw std::invalid_argument("EM: At least two steps required for convergence test");
		}
		maximum_steps_ = maximum_steps;
	}

	void EM::set_means_initialiser(std::shared_ptr<const Clustering::CentroidsInitialiser> means_initialiser)
	{
		if (!means_initialiser) {
			throw std::invalid_argument("EM: Null means initialiser");
		}
		means_initialiser_ = means_initialiser;
	}

	void EM::set_responsibilities_initialiser(std::shared_ptr<const Clustering::ResponsibilitiesInitialiser> responsibilities_initialiser)
	{
		if (!responsibilities_initialiser) {
			throw std::invalid_argument("EM: Null responsibilities initialiser");
		}
		responsibilities_initialiser_ = responsibilities_initialiser;
	}

	const Eigen::MatrixXd& EM::covariance(unsigned int k) const
	{
		if (k >= number_components_) {
			throw std::invalid_argument("EM: Bad component index");
		}
		return covariances_[k];
	}

	const Eigen::MatrixXd& EM::responsibilities() const
	{
		if (!responsibilities_on_host_ && device_) {
			// First access after a fit: one E-step at the parameters the fit's last E-step used,
			// written straight into the N x K host matrix.
			device_->emit(&responsibilities_, nullptr);
			responsibilities_on_host_ = true;
		}
		return responsibilities_;
	}

	const std::vector<unsigned int>& EM::labels() const
	{
		if (!labels_on_host_ && device_) {
			device_->emit(nullptr, &labels_);   // calculate_labels (EM.cpp:289-304) at the parameters of the last E-step
			labels_on_host_ = true;
		}
		if (static_cast<Eigen::Index>(labels_.size()) != sample_size_) {
			labels_.resize(static_cast<size_t>(sample_size_));   // EM.cpp:104; filled only by a converged fit
		}
		return labels_;
	}

	void EM::release_device(bool keep_results)
	{
		if (keep_results) {
			responsibilities();
			labels();
		}
		responsibilities_on_host_ = true;
		labels_on_host_ = true;
		device_.reset();
	}

	bool EM::fit(const DataView data)
	{
		converged_ = false;
		number_iterations_ = 0;
		const auto number_dimensions = static_cast<unsigned int>(data.rows());
		const auto sample_size = static_cast<unsigned int>(data.cols());
		if (!number_dimensions) {
			throw std::invalid_argument("EM: At least one dimension required");
		}
		if (sample_size < number_components_) {
			throw std::invalid_argument("EM: Not enough data ");
		}

		device_.reset();
		means_.resize(number_dimensions, number_components_);
		mixing_probabilities_.fill(1. / static_cast<double>(number_components_));
		labels_.clear();
		labels_on_host_ = true;
		sample_size_ = sample_size;
		responsibilities_.resize(0, 0);
		responsibilities_on_host_ = true;

		if (sample_size == number_components_) {
			// One component per point: exact fit, nothing to iterate (EM.cpp:108-118).
			responsibilities_ = Eigen::MatrixXd::Identity(sample_size, sample_size);
			labels_.resize(sample_size);
			for (unsigned int i = 0; i < sample_size; ++i) {
				std::copy_n(data.data() + static_cast<Eigen::Index>(i) * data.outerStride(), number_dimensions, means_.data() + static_cast<Eigen::Index>(i) * number_dimensions);
				covariances_[i].setZero(number_dimensions, number_dimensions);
				labels_[i] = i;
			}
			log_likelihood_ = std::numeric_limits<double>::infinity();
			converged_ = true;
			return converged_;
		}

		device_ = std::make_unique<detail::EmDevice>(data, number_components_);
		if (maximise_first_) {
			const Clustering::ResponsibilitiesInitialiser& initialiser = *responsibilities_initialiser_;
			if (typeid(initialiser) == typeid(Clustering::ClosestCentroid)) {
				// Clustering.cpp:72-89 without the N x K host matrix: initial centroids as the initialiser draws them, the
				// nearest-centroid pass by the K-means assignment kernel (same strict <, lowest index wins) on the points
				// already in HBM, then the M-step of the one-hot responsibilities.
				const auto& closest = static_cast<const Clustering::ClosestCentroid&>(initialiser);
				Eigen::MatrixXd centroids(number_dimensions, number_components_);
				initialise_centroids(*closest.centroids_initialiser(), data, centroids);
				detail::KmDevice nearest(device_->data(), number_components_);
				nearest.set_centroids(centroids);
				std::int64_t changed = 0;
				nearest.assign(changed);
				std::vector<unsigned int> initial_labels;
				nearest.get_labels(initial_labels);
				device_->maximise_from_labels(initial_labels);
			} else {
				Eigen::MatrixXd initial(sample_size, number_components_);
				responsibilities_initialiser_->init(data, prng_, number_components_, initial);
				device_->maximise_from(initial);
			}
		} else {
			initialise_centroids(*means_initialiser_, data, means_);
			const Eigen::MatrixXd sample_covariance(device_->sample_covariance());
			for (unsigned int k = 0; k < number_components_; ++k) {
				covariances_[k] = sample_covariance;
			}
			device_->set_parameters(means_, covariances_, mixing_probabilities_);
		}

		double old_log_likelihood = -std::numeric_limits<double>::infinity();
		for (unsigned int step = 0; step < maximum_steps_; ++step) {
			// expectation_step + maximisation_step, fused on the device
			log_likelihood_ = device_->step();
			number_iterations_ = step + 1;

			if (verbose_) {
				fetch_parameters(number_dimensions);
				std::cout << "Step " << step << "\n";
				std::cout << "Log-likelihood == " << log_likelihood_ << "\n";
				std::cout << "Mixing probabilities ==";
				for (unsigned int k = 0; k < number_components_; ++k) {
					std::cout << " " << mixing_probabilities_[k];
				}
				std::cout << "\n";
				for (unsigned int k = 0; k < number_components_; ++k) {
					std::cout << "Mean[" << k << "] ==";
					for (unsigned int l = 0; l < number_dimensions; ++l) {
						std::cout << " " << means_(l, k);
					}
					std::cout << "\n";
				}
				Eigen::MatrixXd head;
				device_->emit_rows(0, std::min(sample_size, 10u), head);
				std::cout << "Responsibilities (first 10 rows):\n" << head << std::endl;
			}

			if (step > 0) {
				const double ll_change = std::abs(log_likelihood_ - old_log_likelihood);
				if (ll_change < absolute_tolerance_ + relative_tolerance_ * std::max(std::abs(old_log_likelihood), std::abs(log_likelihood_))) {
					labels_on_host_ = false;   // calculate_labels (EM.cpp:289-304) runs on first access to labels()
					converged_ = true;
					break;
				}
			}
			old_log_likelihood = log_likelihood_;
		}

		fetch_parameters(number_dimensions);
		responsibilities_on_host_ = false;
		if (const char* eager = std::getenv("MLPP_EAGER_RESPONSIBILITIES")) {
			if (eager[0] == '1') {
				responsibilities();
			}
		}
		return converged_;
	}

	void EM::initialise_centroids(const Clustering::CentroidsInitialiser& initialiser, DataView data, MatrixOut centroids)
	{
		if (typeid(initialiser) == typeid(Clustering::KPP)) {
			// the built-in K-means++: distance passes on the device, draws here (Clustering.cpp:39-59)
			detail::kpp_on_device(*device_->data(), data, prng_, number_components_, centroids);
		} else {
			initialiser.init(data, prng_, number_components_, centroids);
		}
	}

	void EM::fetch_parameters(Eigen::Index number_dimensions)
	{
		device_->get_parameters(means_, covariances_, mixing_probabilities_);
		process_covariances(number_dimensions);
	}

	void EM::process_covariances(const Eigen::Index number_dimensions)
	{
		// Host copy of EM.cpp:274-287 for assign_responsibilities: Cholesky factor, inverse by solving
		// against the identity, sqrt|Sigma| as the product of the factor's diagonal.
		const Eigen::Index d = number_dimensions;
		std::vector<double> factor(static_cast<size_t>(d * d));
		for (unsigned int k = 0; k < number_components_; ++k) {
			const double* cov = covariances_[k].data();
			std::copy(cov, cov + d * d, factor.begin());
			double* l = factor.data();
			for (Eigen::Index j = 0; j < d; ++j) {
				double diagonal = l[j + j * d];
				for (Eigen::Index t = 0; t < j; ++t) {
					diagonal -= l[j + t * d] * l[j + t * d];
				}
				diagonal = std::sqrt(diagonal);
				l[j + j * d] = diagonal;
				for (Eigen::Index i = j + 1; i < d; ++i) {
					double value = l[i + j * d];
					for (Eigen::Index t = 0; t < j; ++t) {
						value -= l[i + t * d] * l[j + t * d];
					}
					l[i + j * d] = value / diagonal;
				}
			}
			inverse_covariances_[k].resize(d, d);
			double* inverse = inverse_covariances_[k].data();
			for (Eigen::Index c = 0; c < d; ++c) {
				double* x = inverse + c * d;
				for (Eigen::Index i = 0; i < d; ++i) {
					double value = (i == c) ? 1.0 : 0.0;
					for (Eigen::Index j = 0; j < i; ++j) {
						value -= l[i + j * d] * x[j];
					}
					x[i] = value / l[i + i * d];
				}
				for (Eigen::Index i = d - 1; i >= 0; --i) {
					double value = x[i];
					for (Eigen::Index j = i + 1; j < d; ++j) {
						value -= l[j + i * d] * x[j];
					}
					x[i] = value / l[i + i * d];
				}
			}
			double sqrt_determinant = 1;
			for (Eigen::Index i = 0; i < d; ++i) {
				sqrt_determinant *= l[i + i * d];
			}
			sqrt_covariance_determinants_[k] = sqrt_determinant;
		}
	}

	Eigen::MatrixXd EM::assign_responsibilities(DataView points) const
	{
		if (points.rows() != means().rows()) {
			throw std::invalid_argument("Wrong number of rows");
		}
		if (!device_) {
			throw std::logic_error("EM: no fitted device state");
		}
		Eigen::MatrixXd result;
		device_->predict(points, result);
		return result;
	}

	Eigen::VectorXd EM::log_likelihoods(DataView points) const
	{
		if (points.rows() != means().rows()) {
			throw std::invalid_argument("Wrong number of rows");
		}
		if (!device_) {
			throw std::logic_error("EM: no fitted device state");
		}
		Eigen::VectorXd result;
		device_->score(points, &result, nullptr);
		return result;
	}

	double EM::log_likelihood(DataView points) const
	{
		if (points.rows() != means().rows()) {
			throw std::invalid_argument("Wrong number of rows");
		}
		if (!device_) {
			throw std::logic_error("EM: no fitted device state");
		}
		double mean = 0;
		device_->score(points, nullptr, &mean);
		return mean;
	}

	Eigen::VectorXd EM::log_likelihoods() const
	{
		if (!device_) {
			throw std::logic_error("EM: no fitted device state");
		}
		Eigen::VectorXd result;
		device_->score_fitted(&result, nullptr);
		return result;
	}

	double EM::final_log_likelihood() const
	{
		if (!device_) {
			throw std::logic_error("EM: no fitted device state");
		}
		double mean = 0;
		device_->score_fitted(nullptr, &mean);
		return mean;
	}

	void EM::assign_responsibilities(PointView x, VectorOut u) const
	{
		if (x.size() != means().rows()) {
			throw std::invalid_argument("Wrong x size");
		}
		if (u.size() != static_cast<Eigen::Index>(number_components())) {
			throw std::invalid_argument("Wrong u size");
		}
		const Eigen::Index d = means_.rows();
		Eigen::VectorXd offset(d);
		double total = 0;
		for (unsigned int k = 0; k < number_components_; ++k) {
			for (Eigen::Index l = 0; l < d; ++l) {
				offset[l] = x[l] - means_(l, k);
			}
			u[k] = std::exp(-0.5 * LinearAlgebra::xAx_symmetric(inverse_covariances_[k], offset)) * mixing_probabilities_[k] / sqrt_covariance_determinants_[k];
		}
		for (unsigned int k = 0; k < number_components_; ++k) {
			total += u[k];
		}
		for (unsigned int k = 0; k < number_components_; ++k) {
			u[k] /= total;
		}
	}
}
