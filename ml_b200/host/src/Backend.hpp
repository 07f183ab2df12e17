#pragma once
// Private glue between the ML++ host classes and the C-ABI of include/mlb200.h: RAII handles, the
// process-wide GPU context, and the mapping of status codes to the exceptions the reference throws.
#include <cstdint>
#include <memory>
#include <random>
#include <vector>
#include <Eigen/Core>
#include "ML/dll.hpp"

extern "C" {
#include "mlb200.h"
}

namespace ml
{
	namespace detail
	{
		/** Throws std::invalid_argument for MLB_EINVAL and std::runtime_error for every other failure. */
		void check(int status, const char* where);

		/** The process-wide context: MLPP_CUDA_DEVICES = number of GPUs to shard over (1, 2, 4 or 8;
		default 1).  Created on first use; there is no CPU fallback, so a machine without a CUDA device
		gets a std::runtime_error from the first fit(). */
		mlb_ctx* shared_context();

		/** cppyml.utils.standardise_features (cppyml/cppyml/utils.py:8-28) on the device: every row of the D x N matrix
		minus its mean and, for N > 1, divided by its biased standard deviation. */
		DLL_DECLSPEC Eigen::MatrixXd standardise_features(Eigen::Ref<const Eigen::MatrixXd> data);

		/** The point matrix in HBM. */
		class DeviceData
		{
		public:
			explicit DeviceData(Eigen::Ref<const Eigen::MatrixXd> data);
			~DeviceData();
			DeviceData(const DeviceData&) = delete;
			DeviceData& operator=(const DeviceData&) = delete;
			mlb_data* handle() const { return handle_; }
			Eigen::Index rows() const { return rows_; }
			Eigen::Index cols() const { return cols_; }
			/** KPP distance pass for the newest centroid (D doubles); `nearest` (N) receives the squared distance of
			every point to the nearest centroid chosen so far. */
			void kpp_update(const double* centroid, bool first, std::vector<double>& nearest);
		private:
			mlb_data* handle_ = nullptr;
			Eigen::Index rows_ = 0, cols_ = 0;
		};

		/** What `std::discrete_distribution<Eigen::Index>(weights.begin(), weights.end())(prng)` returns and consumes
		(Clustering.cpp:55-56), without the two N-sized temporaries the library builds per draw: the same sequential sum,
		the same divisions, the same running partial sums, scanned until the first one not below the drawn number (which
		is where the library's binary search over the monotone partial sums ends).  Pinned against the library on the CPU
		(tests/cpp/host_tests.cpp). */
		Eigen::Index draw_discrete(const std::vector<double>& weights, std::default_random_engine& prng);

		/** KPP::init (ML/Clustering.cpp:39-59) with the distance passes on the device and the draws on the host:
		the same std::discrete_distribution over the same weights, so the same centroids and PRNG stream. */
		void kpp_on_device(DeviceData& device_data, Eigen::Ref<const Eigen::MatrixXd> data, std::default_random_engine& prng, unsigned int number_components, Eigen::Ref<Eigen::MatrixXd> centroids);

		/** Device state of one EM fit. */
		class EmDevice
		{
		public:
			EmDevice(Eigen::Ref<const Eigen::MatrixXd> data, unsigned int number_components);
			~EmDevice();
			EmDevice(const EmDevice&) = delete;
			EmDevice& operator=(const EmDevice&) = delete;
			Eigen::MatrixXd sample_covariance();
			void set_parameters(const Eigen::MatrixXd& means, const std::vector<Eigen::MatrixXd>& covariances, const Eigen::VectorXd& mixing_probabilities);
			void maximise_from(const Eigen::MatrixXd& responsibilities);
			/** M-step of the one-hot responsibilities of hard labels (ClosestCentroid start). */
			void maximise_from_labels(const std::vector<unsigned int>& labels);
			/** Responsibilities (m x K) of the columns of `points` (D x m) under the current parameters. */
			void predict(Eigen::Ref<const Eigen::MatrixXd> points, Eigen::MatrixXd& responsibilities);
			/** log p(x) of the columns of `points` (D x m) under the current parameters; either output may be null. */
			void score(Eigen::Ref<const Eigen::MatrixXd> points, Eigen::VectorXd* log_densities, double* mean);
			/** The same for the fitted points: this process's own points, and the mean over all points (collective under
			ml::Distributed). */
			void score_fitted(Eigen::VectorXd* log_densities, double* mean);
			const std::shared_ptr<DeviceData>& data() const { return data_; }
			double step();
			void get_parameters(Eigen::MatrixXd& means, std::vector<Eigen::MatrixXd>& covariances, Eigen::VectorXd& mixing_probabilities);
			void emit(Eigen::MatrixXd* responsibilities, std::vector<unsigned int>* labels);
			void emit_rows(Eigen::Index begin, Eigen::Index count, Eigen::MatrixXd& responsibilities);
		private:
			std::shared_ptr<DeviceData> data_;
			mlb_em* em_ = nullptr;
			unsigned int number_components_;
		};

		/** Device state of one K-means fit (shared by all initialisations of a multi-start fit). */
		class KmDevice
		{
		public:
			KmDevice(Eigen::Ref<const Eigen::MatrixXd> data, unsigned int number_clusters);
			/** On points that are already resident (shared with an EmDevice). */
			KmDevice(std::shared_ptr<DeviceData> data, unsigned int number_clusters);
			~KmDevice();
			KmDevice(const KmDevice&) = delete;
			KmDevice& operator=(const KmDevice&) = delete;
			void set_centroids(const Eigen::MatrixXd& centroids);
			void get_centroids(Eigen::MatrixXd& centroids);
			/** @return inertia; `changed` receives the number of labels that differ from the previous assignment. */
			double assign(std::int64_t& changed);
			/** @return squared Frobenius norm of the centroid shift. */
			double update();
			void get_labels(std::vector<unsigned int>& labels);
			/** Nearest centroid and squared distance for every column of `points` (D x m). */
			void predict(Eigen::Ref<const Eigen::MatrixXd> points, std::vector<unsigned int>& labels, std::vector<double>& squared_distances);
			const std::shared_ptr<DeviceData>& data() const { return data_; }
		private:
			std::shared_ptr<DeviceData> data_;
			mlb_km* km_ = nullptr;
		};

		/** Up to four starts of a multi-start K-means fit advanced in lockstep on one resident copy of the points
		(mlb_kms, KMeans.cpp:29-47): one pass of the assignment kernel scores every point against all active starts. */
		class KmSetsDevice
		{
		public:
			/** Whether `number_sets` starts of `number_clusters` centroids can share a pass on these points. */
			static bool supported(const DeviceData& data, unsigned int number_clusters, unsigned int number_sets);
			KmSetsDevice(std::shared_ptr<DeviceData> data, unsigned int number_clusters, unsigned int number_sets);
			~KmSetsDevice();
			KmSetsDevice(const KmSetsDevice&) = delete;
			KmSetsDevice& operator=(const KmSetsDevice&) = delete;
			unsigned int number_sets() const { return number_sets_; }
			void set_centroids(unsigned int set, const Eigen::MatrixXd& centroids);
			void get_centroids(unsigned int set, Eigen::MatrixXd& centroids);
			/** Assignment step of every start in `active` (bit s = start s): inertia[s], changed[s] for those starts. */
			void assign(unsigned int active, double* inertia, std::int64_t* changed);
			/** Update step of every start in `active`: squared centroid shift per start. */
			void update(unsigned int active, double* shift);
			void get_labels(unsigned int set, std::vector<unsigned int>& labels);
		private:
			std::shared_ptr<DeviceData> data_;
			mlb_kms* kms_ = nullptr;
			unsigned int number_sets_ = 0;
		};
	}
}
