// ml::Clustering::KMeans on the B200 backend.  Control flow, defaults and error behaviour follow
// ML/KMeans.cpp:11-151; assignment_step and update_step (KMeans.cpp:153-192) run on the device.
// The data is uploaded once per fit() and shared by all initialisations of a multi-start fit.
#include "ML/KMeans.hpp"

#include <algorithm>
#include <cstdlib>
#include <iostream>
#include <limits>
#include <stdexcept>
#include <typeinfo>

#include "Backend.hpp"

namespace ml
{
	namespace Clustering
	{
		namespace
		{
			/** MLPP_KMEANS_LOCKSTEP=0: developer switch, the starts of a multi-start fit one after the other (same results;
			tools/bm_kmeans.py times both). */
			bool lockstep_enabled()
			{
				const char* env = std::getenv("MLPP_KMEANS_LOCKSTEP");
				return !(env && env[0] == '0');
			}
		}

		KMeans::KMeans(unsigned int number_clusters)
			: labels_on_host_(true)
			, centroids_initialiser_(std::make_shared<Forgy>())
			, absolute_tolerance_(1e-8)
			, inertia_(0)
			, maximum_steps_(1000)
			, number_initialisations_(1)
			, number_clusters_(number_clusters)
			, number_iterations_(0)
			, verbose_(false)
			, converged_(false)
		{
			if (!number_clusters) {
				throw std::invalid_argument("KMeans: number of clusters cannot be zero");
			}
		}

		KMeans::~KMeans() = default;

		const std::vector<unsigned int>& KMeans::labels() const
		{
			if (!labels_on_host_ && device_) {
				device_->get_labels(labels_);
				labels_on_host_ = true;
			}
			return labels_;
		}

		void KMeans::release_device(bool keep_results)
		{
			if (keep_results) {
				labels();
			}
			labels_on_host_ = true;
			device_.reset();
		}

		bool KMeans::fit(DataView data)
		{
			const auto number_dimensions = static_cast<unsigned int>(data.rows());
			const auto sample_size = static_cast<unsigned int>(data.cols());
			if (!number_dimensions) {
				throw std::invalid_argument("KMeans: At least one dimension required");
			}
			if (sample_size < number_clusters_) {
				throw std::invalid_argument("KMeans: Not enough data ");
			}
			converged_ = false;
			number_iterations_ = 0;
			device_.reset();
			centroids_.resize(number_dimensions, number_clusters_);
			labels_.clear();
			labels_on_host_ = true;

			if (sample_size == number_clusters_) {
				// Every point is its own cluster (KMeans.cpp:67-75); identical for every initialisation.
				labels_.resize(sample_size);
				for (unsigned int i = 0; i < sample_size; ++i) {
					std::copy_n(data.data() + static_cast<Eigen::Index>(i) * data.outerStride(), number_dimensions, centroids_.data() + static_cast<Eigen::Index>(i) * number_dimensions);
					labels_[i] = i;
				}
				inertia_ = 0;
				converged_ = true;
				return converged_;
			}

			device_ = std::make_unique<detail::KmDevice>(data, number_clusters_);
			detail::KmDevice& device = *device_;
			if (number_initialisations_ == 1) {
				fit_once(data, device);
			} else if (!verbose_ && lockstep_enabled() && detail::KmSetsDevice::supported(*device.data(), number_clusters_, 2)) {
				// Best of number_initialisations_ runs by inertia (KMeans.cpp:29-47), the runs advanced in lockstep.
				return fit_lockstep(data, device);
			} else {
				// Best of number_initialisations_ runs by inertia (KMeans.cpp:29-47).
				double min_inertia = std::numeric_limits<double>::infinity();
				Eigen::MatrixXd best_centroids;
				bool any_converged = false;
				for (unsigned int i = 0; i < number_initialisations_; ++i) {
					if (fit_once(data, device)) {
						if (inertia_ < min_inertia) {
							min_inertia = inertia_;
							best_centroids = centroids_;
						}
						any_converged = true;
					}
				}
				converged_ = any_converged;
				if (converged_) {
					centroids_ = best_centroids;
					device.set_centroids(centroids_);
					std::int64_t changed = 0;
					inertia_ = device.assign(changed);
				}
			}
			labels_on_host_ = false;   // downloaded on first access to labels()
			return converged_;
		}

		void KMeans::draw_initial_centroids(DataView data, detail::KmDevice& device)
		{
			const CentroidsInitialiser& initialiser = *centroids_initialiser_;
			if (typeid(initialiser) == typeid(KPP)) {
				// the built-in K-means++: distance passes on the device, draws here (Clustering.cpp:39-59)
				detail::kpp_on_device(*device.data(), data, prng_, number_clusters_, centroids_);
			} else {
				initialiser.init(data, prng_, number_clusters_, centroids_);
			}
		}

		bool KMeans::fit_lockstep(DataView data, detail::KmDevice& device)
		{
			// The reference runs fit_once number_initialisations_ times in a row (KMeans.cpp:34-42).  Only the initialiser
			// consumes the PRNG (KMeans.cpp:77), so the starts' initial centroids are drawn first, in the order the reference
			// draws them; after that the starts are independent Lloyd loops over the same points and are advanced together,
			// four to a pass over the data.  Every start keeps its own step counter and stopping tests (KMeans.cpp:80-109).
			const unsigned int total = number_initialisations_;
			std::vector<Eigen::MatrixXd> start_centroids(total);
			for (unsigned int i = 0; i < total; ++i) {
				draw_initial_centroids(data, device);
				start_centroids[i] = centroids_;
			}
			double min_inertia = std::numeric_limits<double>::infinity();
			Eigen::MatrixXd best_centroids;
			bool any_converged = false;
			for (unsigned int first = 0, count = 0; first < total; first += count) {
				count = std::min(4u, total - first);
				while (count > 1 && !detail::KmSetsDevice::supported(*device.data(), number_clusters_, count)) {
					--count;   // fewer starts per pass when four centroid images do not fit the shared memory
				}
				detail::KmSetsDevice sets(device.data(), number_clusters_, count);
				bool converged[4] = {false, false, false, false};
				double inertia[4] = {0, 0, 0, 0};
				unsigned int iterations[4] = {0, 0, 0, 0};
				for (unsigned int s = 0; s < count; ++s) {
					sets.set_centroids(s, start_centroids[first + s]);
				}
				unsigned int active = (1u << count) - 1u;
				for (unsigned int step = 0; step < maximum_steps_ && active; ++step) {
					std::int64_t changed[4] = {0, 0, 0, 0};
					sets.assign(active, inertia, changed);
					for (unsigned int s = 0; s < count; ++s) {
						if (!((active >> s) & 1u)) {
							continue;
						}
						iterations[s] = step + 1;
						if (step > 0 && changed[s] == 0) {
							// old_labels_ == labels_ (KMeans.cpp:84-89): the centroids are not updated again
							converged[s] = true;
							active &= ~(1u << s);
						}
					}
					if (!active) {
						break;
					}
					double shift[4] = {0, 0, 0, 0};
					sets.update(active, shift);
					if (step > 0) {
						unsigned int reassign = 0;
						for (unsigned int s = 0; s < count; ++s) {
							if (((active >> s) & 1u) && shift[s] < absolute_tolerance_) {
								reassign |= 1u << s;
							}
						}
						if (reassign) {
							// the closing assignment_step of KMeans.cpp:104-106
							sets.assign(reassign, inertia, changed);
							for (unsigned int s = 0; s < count; ++s) {
								if ((reassign >> s) & 1u) {
									converged[s] = true;
								}
							}
							active &= ~reassign;
						}
					}
				}
				// in the order of the reference's loop over the starts (KMeans.cpp:34-42)
				for (unsigned int s = 0; s < count; ++s) {
					if (converged[s]) {
						if (inertia[s] < min_inertia) {
							min_inertia = inertia[s];
							best_centroids.resize(centroids_.rows(), centroids_.cols());
							sets.get_centroids(s, best_centroids);
						}
						any_converged = true;
					}
				}
				if (first + count >= total) {
					// what the last fit_once leaves behind: its centroids, inertia, labels and step count
					const unsigned int s = count - 1;
					sets.get_centroids(s, centroids_);
					inertia_ = inertia[s];
					number_iterations_ = iterations[s];
					if (!any_converged) {
						sets.get_labels(s, labels_);
					}
				}
			}
			converged_ = any_converged;
			if (converged_) {
				centroids_ = best_centroids;
				device.set_centroids(centroids_);
				std::int64_t changed = 0;
				inertia_ = device.assign(changed);
				labels_on_host_ = false;   // downloaded on first access to labels()
			} else {
				labels_on_host_ = true;    // no start converged: the last start's labels, already here
				device.set_centroids(centroids_);   // what transform() and final_inertia() read: the returned centroids
			}
			return converged_;
		}

		bool KMeans::fit_once(DataView data, detail::KmDevice& device)
		{
			converged_ = false;
			draw_initial_centroids(data, device);
			device.set_centroids(centroids_);
			for (unsigned int step = 0; step < maximum_steps_; ++step) {
				std::int64_t changed = 0;
				inertia_ = device.assign(changed);
				number_iterations_ = step + 1;
				if (step > 0 && changed == 0) {
					// old_labels_ == labels_ (KMeans.cpp:84-89): the centroids are not updated again
					converged_ = true;
					break;
				}
				const double centroid_shift = device.update();
				if (verbose_) {
					device.get_centroids(centroids_);
					std::cout << "Step " << step << "\n";
					for (unsigned int k = 0; k < number_clusters_; ++k) {
						std::cout << "Centroid[" << k << "] ==";
						for (Eigen::Index l = 0; l < centroids_.rows(); ++l) {
							std::cout << " " << centroids_(l, k);
						}
						std::cout << "\n";
					}
					std::cout << std::endl;
				}
				if (step > 0 && centroid_shift < absolute_tolerance_) {
					inertia_ = device.assign(changed);
					converged_ = true;
					break;
				}
			}
			device.get_centroids(centroids_);
			return converged_;
		}

		void KMeans::set_seed(unsigned int seed)
		{
			prng_.seed(seed);
		}

		void KMeans::set_absolute_tolerance(double absolute_tolerance)
		{
			if (absolute_tolerance < 0) {
				throw std::domain_error("KMeans: Negative absolute tolerance");
			}
			absolute_tolerance_ = absolute_tolerance;
		}

		void KMeans::set_maximum_steps(unsigned int maximum_steps)
		{
			if (maximum_steps < 2) {
				throw std::invalid_argument("KMeans: At least two steps required for convergence test");
			}
			maximum_steps_ = maximum_steps;
		}

		void KMeans::set_number_initialisations(unsigned int number_initialisations)
		{
			if (number_initialisations < 1) {
				throw std::invalid_argument("KMeans: At least 1 initialisation required");
			}
			number_initialisations_ = number_initialisations;
		}

		void KMeans::set_centroids_initialiser(std::shared_ptr<const CentroidsInitialiser> centroids_initialiser)
		{
			if (!centroids_initialiser) {
				throw std::invalid_argument("KMeans: Null centroids initialiser");
			}
			centroids_initialiser_ = centroids_initialiser;
		}

		std::pair<std::vector<unsigned int>, std::vector<double>> KMeans::assign_labels(DataView points) const
		{
			if (points.rows() != centroids_.rows()) {
				throw std::invalid_argument("KMeans: wrong number of rows");
			}
			if (!device_) {
				throw std::logic_error("KMeans: no fitted device state");
			}
			std::pair<std::vector<unsigned int>, std::vector<double>> result;
			device_->predict(points, result.first, result.second);
			return result;
		}

		Eigen::MatrixXd KMeans::transform(DataView points) const
		{
			if (points.rows() != centroids_.rows()) {
				throw std::invalid_argument("KMeans: wrong number of rows");
			}
			if (!device_) {
				throw std::logic_error("KMeans: no fitted device state");
			}
			Eigen::MatrixXd result;
			device_->transform(points, result);
			return result;
		}

		Eigen::MatrixXd KMeans::transform() const
		{
			if (!device_) {
				throw std::logic_error("KMeans: no fitted device state");
			}
			Eigen::MatrixXd result;
			device_->transform_fitted(result);
			return result;
		}

		double KMeans::inertia(DataView points) const
		{
			if (points.rows() != centroids_.rows()) {
				throw std::invalid_argument("KMeans: wrong number of rows");
			}
			if (!device_) {
				throw std::logic_error("KMeans: no fitted device state");
			}
			return device_->inertia(points);
		}

		double KMeans::final_inertia() const
		{
			if (!device_) {
				throw std::logic_error("KMeans: no fitted device state");
			}
			return device_->fitted_inertia();
		}

		std::pair<unsigned int, double> KMeans::assign_label(PointView x) const
		{
			if (x.size() != centroids_.rows()) {
				throw std::invalid_argument("KMeans: wrong size of x");
			}
			const Eigen::Index dim = centroids_.rows();
			unsigned int label = 0;
			double smallest = std::numeric_limits<double>::infinity();
			for (unsigned int k = 0; k < number_clusters_; ++k) {
				const double* c = centroids_.data() + static_cast<Eigen::Index>(k) * dim;
				double distance = 0;
				for (Eigen::Index l = 0; l < dim; ++l) {
					const double diff = x[l] - c[l];
					distance += diff * diff;
				}
				if (distance < smallest) {
					smallest = distance;
					label = k;
				}
			}
			return std::make_pair(label, smallest);
		}
	}
}
