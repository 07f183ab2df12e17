#include "Backend.hpp"
#include "ML/Distributed.hpp"

#include <algorithm>
#include <cstdlib>
#include <limits>
#include <mutex>
#include <numeric>
#include <stdexcept>
#include <string>

namespace ml
{
	namespace detail
	{
		void check(int status, const char* where)
		{
			if (status == MLB_OK) {
				return;
			}
			const std::string message = std::string(where) + ": " + mlb_last_error();
			if (status == MLB_EINVAL) {
				throw std::invalid_argument(message);
			}
			throw std::runtime_error(message);
		}

		namespace
		{
			/** The process-wide context is never destroyed: models (static objects of the application, Python objects
			collected at interpreter shutdown) may outlive any static of this library, and their destructors still need
			it.  The driver reclaims the device resources when the process ends. */
			struct ContextHolder
			{
				mlb_ctx* ctx = nullptr;
			};
		}

		namespace
		{
			ContextHolder& context_holder()
			{
				static ContextHolder holder;
				return holder;
			}

			std::mutex& context_mutex()
			{
				static std::mutex mutex;
				return mutex;
			}

			bool distributed_active = false;
		}

		mlb_ctx* shared_context()
		{
			ContextHolder& holder = context_holder();
			std::lock_guard<std::mutex> lock(context_mutex());
			if (!holder.ctx) {
				int number_devices = 1;
				if (const char* env = std::getenv("MLPP_CUDA_DEVICES")) {
					number_devices = std::atoi(env);
				}
				check(mlb_ctx_create(nullptr, number_devices, &holder.ctx), "ML++ B200 backend");
			}
			return holder.ctx;
		}

		Eigen::MatrixXd standardise_features(Eigen::Ref<const Eigen::MatrixXd> data)
		{
			Eigen::MatrixXd result(data.rows(), data.cols());
			if (data.size()) {
				check(mlb_standardise_features(shared_context(), data.data(), data.cols(), static_cast<int>(data.rows()), data.outerStride(), result.data(), data.rows()), "standardise_features");
			}
			return result;
		}

		DeviceData::DeviceData(Eigen::Ref<const Eigen::MatrixXd> data)
			: rows_(data.rows()), cols_(data.cols())
		{
			mlb_ctx* ctx = shared_context();
			int64_t total = data.cols();
			if (distributed_active) {
				// one process per GPU: `data` holds this rank's columns, the problem is the concatenation over the ranks
				check(mlb_ctx_sum_int64(ctx, data.cols(), &total), "point count over the ranks");
			}
			check(mlb_data_upload(ctx, data.data(), data.cols(), total, static_cast<int>(data.rows()), data.outerStride(), &handle_), "upload");
		}

		DeviceData::~DeviceData()
		{
			mlb_data_free(handle_);
		}

		void DeviceData::kpp_update(const double* centroid, bool first, std::vector<double>& nearest)
		{
			nearest.resize(static_cast<size_t>(cols_));
			check(mlb_data_kpp_update(handle_, centroid, first ? 1 : 0, nearest.data()), "KPP distance pass");
		}

		Eigen::Index draw_discrete(const std::vector<double>& weights, std::default_random_engine& prng)
		{
			const size_t n = weights.size();
			if (n < 2) {
				return 0;   // the library keeps no probabilities then and draws nothing
			}
			const double sum = std::accumulate(weights.begin(), weights.end(), 0.0);
			const double p = std::generate_canonical<double, std::numeric_limits<double>::digits>(prng);
			double cumulative = 0;
			for (size_t i = 0; i + 1 < n; ++i) {
				cumulative += weights[i] / sum;
				if (!(cumulative < p)) {
					return static_cast<Eigen::Index>(i);
				}
			}
			return static_cast<Eigen::Index>(n - 1);   // the last cumulative probability is set to one
		}

		void kpp_on_device(DeviceData& device_data, Eigen::Ref<const Eigen::MatrixXd> data, std::default_random_engine& prng, const unsigned int number_components, Eigen::Ref<Eigen::MatrixXd> centroids)
		{
			const Eigen::Index dim = data.rows();
			std::vector<double> weights(static_cast<size_t>(data.cols()), 1.0);   // first draw: uniform (Clustering.cpp:53)
			std::vector<double> newest(static_cast<size_t>(dim));
			for (unsigned int k = 0; k < number_components; ++k) {
				if (k > 0) {
					device_data.kpp_update(newest.data(), k == 1, weights);
				}
				const Eigen::Index index = draw_discrete(weights, prng);
				std::copy_n(data.data() + index * data.outerStride(), dim, newest.begin());
				std::copy_n(newest.begin(), dim, centroids.data() + static_cast<Eigen::Index>(k) * centroids.outerStride());
			}
		}

		EmDevice::EmDevice(Eigen::Ref<const Eigen::MatrixXd> data, unsigned int number_components)
			: data_(std::make_shared<DeviceData>(data)), number_components_(number_components)
		{
			check(mlb_em_create(shared_context(), data_->handle(), static_cast<int>(number_components), &em_), "EM");
		}

		EmDevice::~EmDevice()
		{
			mlb_em_destroy(em_);
		}

		Eigen::MatrixXd EmDevice::sample_covariance()
		{
			Eigen::MatrixXd covariance(data_->rows(), data_->rows());
			check(mlb_em_sample_covariance(em_, covariance.data()), "EM sample covariance");
			return covariance;
		}

		void EmDevice::set_parameters(const Eigen::MatrixXd& means, const std::vector<Eigen::MatrixXd>& covariances, const Eigen::VectorXd& mixing_probabilities)
		{
			const auto dd = static_cast<size_t>(data_->rows() * data_->rows());
			std::vector<double> packed(dd * covariances.size());
			for (size_t k = 0; k < covariances.size(); ++k) {
				std::copy(covariances[k].data(), covariances[k].data() + dd, packed.begin() + static_cast<std::ptrdiff_t>(k * dd));
			}
			check(mlb_em_set_params(em_, means.data(), packed.data(), mixing_probabilities.data()), "EM parameters");
		}

		void EmDevice::maximise_from(const Eigen::MatrixXd& responsibilities)
		{
			check(mlb_em_mstep_from_responsibilities(em_, responsibilities.data(), responsibilities.rows()), "EM maximisation step");
		}

		void EmDevice::maximise_from_labels(const std::vector<unsigned int>& labels)
		{
			if (static_cast<Eigen::Index>(labels.size()) != data_->cols()) {
				throw std::invalid_argument("EM maximisation step: wrong number of labels");
			}
			check(mlb_em_mstep_from_labels(em_, labels.data()), "EM maximisation step");
		}

		void EmDevice::predict(Eigen::Ref<const Eigen::MatrixXd> points, Eigen::MatrixXd& responsibilities)
		{
			responsibilities.resize(points.cols(), number_components_);
			check(mlb_em_predict(em_, points.data(), points.cols(), points.outerStride(), responsibilities.data(), std::max<Eigen::Index>(1, points.cols()), nullptr), "EM responsibilities of new points");
		}

		void EmDevice::score(Eigen::Ref<const Eigen::MatrixXd> points, Eigen::VectorXd* log_densities, double* mean)
		{
			if (log_densities) {
				log_densities->resize(points.cols());
			}
			check(mlb_em_score(em_, points.data(), points.cols(), points.outerStride(), log_densities ? log_densities->data() : nullptr, mean), "EM log-likelihood of new points");
		}

		void EmDevice::score_fitted(Eigen::VectorXd* log_densities, double* mean)
		{
			if (log_densities) {
				log_densities->resize(data_->cols());
			}
			check(mlb_em_score_fitted(em_, log_densities ? log_densities->data() : nullptr, mean), "EM log-likelihood of the fitted points");
		}

		double EmDevice::step()
		{
			double log_likelihood = 0;
			check(mlb_em_step(em_, &log_likelihood), "EM step");
			return log_likelihood;
		}

		void EmDevice::get_parameters(Eigen::MatrixXd& means, std::vector<Eigen::MatrixXd>& covariances, Eigen::VectorXd& mixing_probabilities)
		{
			const Eigen::Index d = data_->rows();
			const auto dd = static_cast<size_t>(d * d);
			std::vector<double> packed(dd * number_components_);
			means.resize(d, number_components_);
			mixing_probabilities.resize(number_components_);
			check(mlb_em_get_params(em_, means.data(), packed.data(), mixing_probabilities.data()), "EM parameters");
			covariances.resize(number_components_);
			for (size_t k = 0; k < covariances.size(); ++k) {
				covariances[k].resize(d, d);
				std::copy(packed.begin() + static_cast<std::ptrdiff_t>(k * dd), packed.begin() + static_cast<std::ptrdiff_t>((k + 1) * dd), covariances[k].data());
			}
		}

		void EmDevice::emit(Eigen::MatrixXd* responsibilities, std::vector<unsigned int>* labels)
		{
			if (responsibilities) {
				responsibilities->resize(data_->cols(), number_components_);
			}
			if (labels) {
				labels->resize(static_cast<size_t>(data_->cols()));
			}
			check(mlb_em_emit(em_, responsibilities ? responsibilities->data() : nullptr, data_->cols(), labels ? labels->data() : nullptr), "EM responsibilities");
		}

		void EmDevice::emit_rows(Eigen::Index begin, Eigen::Index count, Eigen::MatrixXd& responsibilities)
		{
			responsibilities.resize(count, number_components_);
			check(mlb_em_emit_range(em_, begin, count, responsibilities.data(), count, nullptr), "EM responsibilities");
		}

		KmDevice::KmDevice(Eigen::Ref<const Eigen::MatrixXd> data, unsigned int number_clusters)
			: KmDevice(std::make_shared<DeviceData>(data), number_clusters)
		{
		}

		KmDevice::KmDevice(std::shared_ptr<DeviceData> data, unsigned int number_clusters)
			: data_(std::move(data))
		{
			check(mlb_km_create(shared_context(), data_->handle(), static_cast<int>(number_clusters), &km_), "KMeans");
		}

		KmDevice::~KmDevice()
		{
			mlb_km_destroy(km_);
		}

		void KmDevice::set_centroids(const Eigen::MatrixXd& centroids)
		{
			check(mlb_km_set_centroids(km_, centroids.data()), "KMeans centroids");
		}

		void KmDevice::get_centroids(Eigen::MatrixXd& centroids)
		{
			check(mlb_km_get_centroids(km_, centroids.data()), "KMeans centroids");
		}

		double KmDevice::assign(std::int64_t& changed)
		{
			double inertia = 0;
			int64_t n_changed = 0;
			check(mlb_km_assign(km_, &inertia, &n_changed), "KMeans assignment step");
			changed = n_changed;
			return inertia;
		}

		double KmDevice::update()
		{
			double shift = 0;
			check(mlb_km_update(km_, &shift), "KMeans update step");
			return shift;
		}

		void KmDevice::predict(Eigen::Ref<const Eigen::MatrixXd> points, std::vector<unsigned int>& labels, std::vector<double>& squared_distances)
		{
			labels.resize(static_cast<size_t>(points.cols()));
			squared_distances.resize(static_cast<size_t>(points.cols()));
			check(mlb_km_predict(km_, points.data(), points.cols(), points.outerStride(), labels.data(), squared_distances.data()), "KMeans labels of new points");
		}

		void KmDevice::get_labels(std::vector<unsigned int>& labels)
		{
			labels.resize(static_cast<size_t>(data_->cols()));
			check(mlb_km_get_labels(km_, labels.data()), "KMeans labels");
		}

		bool KmSetsDevice::supported(const DeviceData& data, unsigned int number_clusters, unsigned int number_sets)
		{
			return mlb_kms_supported(data.handle(), static_cast<int>(number_clusters), static_cast<int>(number_sets)) != 0;
		}

		KmSetsDevice::KmSetsDevice(std::shared_ptr<DeviceData> data, unsigned int number_clusters, unsigned int number_sets)
			: data_(std::move(data)), number_sets_(number_sets)
		{
			check(mlb_kms_create(shared_context(), data_->handle(), static_cast<int>(number_clusters), static_cast<int>(number_sets), &kms_), "KMeans start sets");
		}

		KmSetsDevice::~KmSetsDevice()
		{
			mlb_kms_destroy(kms_);
		}

		void KmSetsDevice::set_centroids(unsigned int set, const Eigen::MatrixXd& centroids)
		{
			check(mlb_kms_set_centroids(kms_, static_cast<int>(set), centroids.data()), "KMeans centroids");
		}

		void KmSetsDevice::get_centroids(unsigned int set, Eigen::MatrixXd& centroids)
		{
			check(mlb_kms_get_centroids(kms_, static_cast<int>(set), centroids.data()), "KMeans centroids");
		}

		void KmSetsDevice::assign(unsigned int active, double* inertia, std::int64_t* changed)
		{
			int64_t n_changed[4] = {0, 0, 0, 0};
			check(mlb_kms_assign(kms_, active, inertia, n_changed), "KMeans assignment step");
			for (unsigned int s = 0; s < number_sets_; ++s) {
				if ((active >> s) & 1u) {
					changed[s] = n_changed[s];
				}
			}
		}

		void KmSetsDevice::update(unsigned int active, double* shift)
		{
			check(mlb_kms_update(kms_, active, shift), "KMeans update step");
		}

		void KmSetsDevice::get_labels(unsigned int set, std::vector<unsigned int>& labels)
		{
			labels.resize(static_cast<size_t>(data_->cols()));
			check(mlb_kms_get_labels(kms_, static_cast<int>(set), labels.data()), "KMeans labels");
		}
	}
}

namespace ml
{
	namespace Distributed
	{
		std::array<unsigned char, 128> unique_id()
		{
			std::array<unsigned char, 128> id{};
			detail::check(mlb_nccl_unique_id(id.data()), "NCCL unique id");
			return id;
		}

		void init(int device, int rank, int world, const std::array<unsigned char, 128>& id)
		{
			std::lock_guard<std::mutex> lock(detail::context_mutex());
			if (detail::context_holder().ctx) {
				throw std::logic_error("ml::Distributed::init: the process already has a GPU context (call init before the first fit)");
			}
			detail::check(mlb_ctx_create_rank(device, rank, world, id.data(), &detail::context_holder().ctx), "ml::Distributed::init");
			detail::distributed_active = true;
		}

		bool active()
		{
			return detail::distributed_active;
		}

		std::pair<Eigen::Index, Eigen::Index> shard_range(Eigen::Index n_total, int world, int rank)
		{
			int64_t begin = 0, end = 0;
			detail::check(mlb_shard_range(n_total, world, rank, &begin, &end), "ml::Distributed::shard_range");
			return std::make_pair(static_cast<Eigen::Index>(begin), static_cast<Eigen::Index>(end));
		}
	}
}
