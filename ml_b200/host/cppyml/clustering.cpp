// cppyml.clustering: the Python surface of the reference's cppyml/clustering.cpp:75-184 over the
// B200 host classes.  Same class names, methods, properties, argument names and array conventions:
// fit() takes a float64 C-contiguous (N, D) array without conversion (a point per row) and views it
// as the column-major D x N matrix the C++ API wants; `means` is (D, K); `responsibilities` is
// (N, K); KMeans.centroids is (K, D); KMeans.labels is a list.
//
// pybind11/eigen.h needs the real Eigen headers; so that the module also builds where Eigen is not
// installed, arrays are converted by hand through pybind11/numpy.h (same shapes, same dtypes).
#include <pybind11/pybind11.h>
#include <pybind11/numpy.h>
#include <pybind11/stl.h>

#include <cmath>
#include <cstring>
#include <stdexcept>

#include "ML/Clustering.hpp"
#include "ML/Distributed.hpp"
#include "ML/EM.hpp"
#include "ML/KMeans.hpp"
#include "../src/Backend.hpp"

namespace py = pybind11;

namespace
{
	using MatrixXdR = Eigen::Matrix<double, Eigen::Dynamic, Eigen::Dynamic, Eigen::RowMajor>;

	/** The (N, D) row-major array as a D x N column-major matrix, without copying. */
	Eigen::Map<const Eigen::MatrixXd> as_columns(const py::array& data)
	{
		if (!py::isinstance<py::array_t<double>>(data) || data.ndim() != 2 || !(data.flags() & py::array::c_style)) {
			throw py::type_error("incompatible function arguments. data must be a C-contiguous float64 numpy array of shape (N, D); no conversion is performed");
		}
		return Eigen::Map<const Eigen::MatrixXd>(static_cast<const double*>(data.data()), data.shape(1), data.shape(0));
	}

	Eigen::VectorXd as_vector(const py::array_t<double, py::array::c_style | py::array::forcecast>& x)
	{
		if (x.ndim() != 1) {
			throw py::type_error("x must be a 1-D array");
		}
		Eigen::VectorXd v(x.shape(0));
		std::memcpy(v.data(), x.data(), sizeof(double) * static_cast<size_t>(x.shape(0)));
		return v;
	}

	/** Column-major matrix -> numpy array of the same shape (Fortran order, like pybind11/eigen.h produces). */
	py::array_t<double> to_numpy(const Eigen::MatrixXd& m)
	{
		py::array_t<double, py::array::f_style> out({m.rows(), m.cols()});
		std::memcpy(out.mutable_data(), m.data(), sizeof(double) * static_cast<size_t>(m.size()));
		return out;
	}

	py::array_t<unsigned int> to_numpy(const std::vector<unsigned int>& v)
	{
		py::array_t<unsigned int> out(static_cast<py::ssize_t>(v.size()));
		std::memcpy(out.mutable_data(), v.data(), sizeof(unsigned int) * v.size());
		return out;
	}

	/** (K, D) C-contiguous array -> D x K column-major matrix (the same memory). */
	Eigen::MatrixXd centroids_from_rows(const py::array_t<double, py::array::c_style | py::array::forcecast>& rows)
	{
		if (rows.ndim() != 2) {
			throw py::type_error("centroids must be a 2-D array of shape (K, D)");
		}
		Eigen::MatrixXd m(rows.shape(1), rows.shape(0));
		std::memcpy(m.data(), rows.data(), sizeof(double) * static_cast<size_t>(m.size()));
		return m;
	}

	py::array_t<double> to_numpy(const Eigen::VectorXd& v)
	{
		py::array_t<double> out(v.size());
		std::memcpy(out.mutable_data(), v.data(), sizeof(double) * static_cast<size_t>(v.size()));
		return out;
	}
}

namespace ml
{
	/** ml::EM with row-major entry points for Python. */
	class EMPy : public EM
	{
	public:
		explicit EMPy(unsigned int number_components)
			: EM(number_components)
		{}

		bool fit_row_major(const py::array& data)
		{
			const auto columns = as_columns(data);
			fitted_points_ = columns.cols();
			py::gil_scoped_release release;   // no Python callbacks happen inside fit
			return fit(columns);
		}

		py::array_t<double> calculate_responsibilities(const py::array_t<double, py::array::c_style | py::array::forcecast>& x) const
		{
			const Eigen::VectorXd point = as_vector(x);
			Eigen::VectorXd u(number_components());
			EM::assign_responsibilities(point, u);
			return to_numpy(u);
		}

		/** (m, D) points -> (m, K) responsibilities, on the device. */
		py::array_t<double> calculate_responsibilities_batch(const py::array& points) const
		{
			const auto columns = as_columns(points);
			Eigen::MatrixXd result;
			{
				py::gil_scoped_release release;
				result = EM::assign_responsibilities(columns);
			}
			return to_numpy(result);
		}

		/** log p(x) of every row of `data` (m, D), or of the fitted points when `data` is None, on the device. */
		py::array_t<double> score_samples_py(const py::object& data) const
		{
			Eigen::VectorXd result;
			if (data.is_none()) {
				py::gil_scoped_release release;
				result = log_likelihoods();
			} else {
				const auto columns = as_columns(data);
				py::gil_scoped_release release;
				result = log_likelihoods(columns);
			}
			return to_numpy(result);
		}

		/** Mean log p(x) over the rows of `data`, or over the fitted points when `data` is None. */
		double score_py(const py::object& data) const
		{
			if (data.is_none()) {
				py::gil_scoped_release release;
				return final_log_likelihood();
			}
			const auto columns = as_columns(data);
			py::gil_scoped_release release;
			return log_likelihood(columns);
		}

		/** -2 n score(data) + penalty_per_parameter * p, p the free parameters of a full-covariance mixture (sklearn's
		GaussianMixture._n_parameters: K D means, K D (D + 1) / 2 covariance entries, K - 1 weights). */
		double information_criterion(const py::object& data, bool bayesian) const
		{
			const double n = static_cast<double>(data.is_none() ? fitted_points_ : as_columns(data).cols());
			const double d = static_cast<double>(means().rows()), k = static_cast<double>(number_components());
			const double p = k * d + k * d * (d + 1) / 2 + k - 1;
			return -2 * n * score_py(data) + (bayesian ? std::log(n) : 2.0) * p;
		}

	private:
		Eigen::Index fitted_points_ = 0;
	};

	namespace Clustering
	{
		/** ml::Clustering::KMeans with row-major entry points for Python. */
		class KMeansPy : public KMeans
		{
		public:
			explicit KMeansPy(unsigned int number_clusters)
				: KMeans(number_clusters)
			{}

			bool fit_row_major(const py::array& data)
			{
				const auto columns = as_columns(data);
				py::gil_scoped_release release;
				return fit(columns);
			}

			/** (K, D), C order: the memory of the D x K column-major centroid matrix. */
			py::array_t<double> centroids_row_major() const
			{
				const Eigen::MatrixXd& c = centroids();
				py::array_t<double> out({c.cols(), c.rows()});
				std::memcpy(out.mutable_data(), c.data(), sizeof(double) * static_cast<size_t>(c.size()));
				return out;
			}

			std::pair<unsigned int, double> assign_label_py(const py::array_t<double, py::array::c_style | py::array::forcecast>& x) const
			{
				return assign_label(as_vector(x));
			}

			/** (m, D) points -> (labels uint32 (m,), squared distances (m,)), on the device. */
			std::pair<py::array_t<unsigned int>, py::array_t<double>> assign_labels_py(const py::array& points) const
			{
				const auto columns = as_columns(points);
				std::pair<std::vector<unsigned int>, std::vector<double>> result;
				{
					py::gil_scoped_release release;
					result = assign_labels(columns);
				}
				py::array_t<unsigned int> labels(static_cast<py::ssize_t>(result.first.size()));
				py::array_t<double> distances(static_cast<py::ssize_t>(result.second.size()));
				std::memcpy(labels.mutable_data(), result.first.data(), sizeof(unsigned int) * result.first.size());
				std::memcpy(distances.mutable_data(), result.second.data(), sizeof(double) * result.second.size());
				return std::make_pair(labels, distances);
			}

			/** Euclidean distance of every row of `data` (m, D), or of every fitted point when `data` is None, to every
			centroid: (m, K), on the device. */
			py::array_t<double> transform_py(const py::object& data) const
			{
				Eigen::MatrixXd result;
				if (data.is_none()) {
					py::gil_scoped_release release;
					result = transform();
				} else {
					const auto columns = as_columns(data);
					py::gil_scoped_release release;
					result = transform(columns);
				}
				return to_numpy(result);
			}

			/** -inertia of the rows of `data`, or of the fitted points at the returned centroids when `data` is None. */
			double score_py(const py::object& data) const
			{
				if (data.is_none()) {
					py::gil_scoped_release release;
					return -final_inertia();
				}
				const auto columns = as_columns(data);
				py::gil_scoped_release release;
				return -inertia(columns);
			}
		};
	}
}

void init_clustering(py::module_& m)
{
	auto m_clustering = m.def_submodule("clustering", "Gaussian-mixture EM and K-means.");

	py::class_<ml::Clustering::CentroidsInitialiser, std::shared_ptr<ml::Clustering::CentroidsInitialiser>>(m_clustering, "CentroidsInitialiser")
		.doc() = "Base class of the strategies that pick K starting centroids.";

	py::class_<ml::Clustering::ResponsibilitiesInitialiser, std::shared_ptr<ml::Clustering::ResponsibilitiesInitialiser>>(m_clustering, "ResponsibilitiesInitialiser")
		.doc() = "Base class of the strategies that pick starting responsibilities (N x K).";

	py::class_<ml::Clustering::Forgy, std::shared_ptr<ml::Clustering::Forgy>, ml::Clustering::CentroidsInitialiser>(m_clustering, "Forgy")
		.def(py::init<>())
		.doc() = "K distinct data points, drawn without replacement, become the centroids.";

	py::class_<ml::Clustering::RandomPartition, std::shared_ptr<ml::Clustering::RandomPartition>, ml::Clustering::CentroidsInitialiser>(m_clustering, "RandomPartition")
		.def(py::init<>())
		.doc() = "Every point joins one of K groups at random; the group means become the centroids.";

	py::class_<ml::Clustering::KPP, std::shared_ptr<ml::Clustering::KPP>, ml::Clustering::CentroidsInitialiser>(m_clustering, "KPP")
		.def(py::init<>())
		.doc() = "k-means++ seeding: each new centroid is a data point drawn with probability proportional to its squared distance from the centroids chosen so far (distance passes on the GPU).";

	py::class_<ml::Clustering::ExplicitCentroids, std::shared_ptr<ml::Clustering::ExplicitCentroids>, ml::Clustering::CentroidsInitialiser>(m_clustering, "ExplicitCentroids")
		.def(py::init([](const py::array_t<double, py::array::c_style | py::array::forcecast>& centroids) {
			return std::make_shared<ml::Clustering::ExplicitCentroids>(centroids_from_rows(centroids));
		}), py::arg("centroids"))
		.doc() = "The given (K, D) array, verbatim, as the starting centroids (an addition to the reference's initialisers).";

	py::class_<ml::Clustering::ClosestCentroid, std::shared_ptr<ml::Clustering::ClosestCentroid>, ml::Clustering::ResponsibilitiesInitialiser>(m_clustering, "ClosestCentroid")
		.def(py::init<std::shared_ptr<ml::Clustering::CentroidsInitialiser>>(), py::arg("centroids_initialiser"))
		.doc() = "One-hot responsibilities: each point belongs to the nearest of the centroids its centroids_initialiser picks.";

	py::class_<ml::EMPy, std::shared_ptr<ml::EMPy>>(m_clustering, "EM")
		.def(py::init<unsigned int>(), py::arg("number_components"), "Args:\n    number_components: how many Gaussians the mixture has (at least 1).")
		.def("set_seed", &ml::EMPy::set_seed, py::arg("seed"), "Seeds the pseudo-random generator the initialisers draw from.")
		.def("set_absolute_tolerance", &ml::EMPy::set_absolute_tolerance, py::arg("absolute_tolerance"), "Absolute part of the stopping threshold (>= 0).")
		.def("set_relative_tolerance", &ml::EMPy::set_relative_tolerance, py::arg("relative_tolerance"), "Relative part of the stopping threshold on the log-likelihood change (>= 0).")
		.def("set_maximum_steps", &ml::EMPy::set_maximum_steps, py::arg("maximum_steps"), "Upper bound on the number of iterations (at least 2).")
		.def("set_means_initialiser", &ml::EMPy::set_means_initialiser, py::arg("means_initialiser"), "Chooses how the starting means are picked.")
		.def("set_responsibilities_initialiser", &ml::EMPy::set_responsibilities_initialiser, py::arg("responsibilities_initialiser"), "Chooses how the starting responsibilities are picked (used with set_maximise_first(True)).")
		.def("set_verbose", &ml::EMPy::set_verbose, py::arg("verbose"), "Prints the state after every iteration when True.")
		.def("set_maximise_first", &ml::EMPy::set_maximise_first, py::arg("maximise_first"), "When True the fit starts with an M-step on initial responsibilities instead of from initial means.")
		.def("fit", &ml::EMPy::fit_row_major, py::arg("data").noconvert(),
			"Runs EM on the GPU.\n\nArgs:\n    data: float64 C-contiguous array of shape (N, D), one point per row; used as is, never converted.\n\nReturns:\n    Whether the log-likelihood change fell below the tolerance before maximum_steps.")
		.def_property_readonly("number_components", &ml::EMPy::number_components, "K, as given to the constructor.")
		.def_property_readonly("means", [](const ml::EMPy& em) { return to_numpy(em.means()); }, "Means after the fit, shape (D, K).")
		.def_property_readonly("responsibilities", [](py::object self) {
			// A read-only view of the model's own N x K matrix (what pybind11/eigen.h returns for a `const MatrixXd&`
			// property in the reference): no second copy of a matrix that is 25.6 GB at N = 1e8, K = 32.
			const ml::EMPy& em = self.cast<const ml::EMPy&>();
			const Eigen::MatrixXd* r = nullptr;
			{
				py::gil_scoped_release release;
				r = &em.responsibilities();
			}
			py::array_t<double> view({r->rows(), r->cols()}, {static_cast<py::ssize_t>(sizeof(double)), static_cast<py::ssize_t>(sizeof(double) * r->rows())}, r->data(), self);
			py::detail::array_proxy(view.ptr())->flags &= ~py::detail::npy_api::NPY_ARRAY_WRITEABLE_;
			return view;
		}, "Responsibilities of the last E-step, shape (N, K): a read-only view of the model's matrix, brought to the host on first access.")
		.def_property_readonly("log_likelihood", [](const ml::EMPy& em) { return em.log_likelihood(); }, "Mean log-likelihood per point at the last E-step.")
		.def_property_readonly("mixing_probabilities", [](const ml::EMPy& em) { return to_numpy(em.mixing_probabilities()); }, "Mixture weights, shape (K,).")
		.def_property_readonly("number_iterations", &ml::EMPy::number_iterations, "Iterations run by the last fit.")
		.def_property_readonly("converged", &ml::EMPy::converged, "Whether the last fit converged.")
		.def_property_readonly("labels_array", [](const ml::EMPy& em) { return to_numpy(em.labels()); }, "Most responsible component of every fitted point as a uint32 array (meaningful after a converged fit); brought to the host on first access.")
		.def("covariance", [](const ml::EMPy& em, unsigned int k) { return to_numpy(em.covariance(k)); }, py::arg("k"),
			"Args:\n    k: component index in [0, K).\n\nReturns:\n    The (D, D) covariance of that component.")
		.def("assign_responsibilities", &ml::EMPy::calculate_responsibilities, py::arg("x"),
			"Args:\n    x: one point, D values.\n\nReturns:\n    The K responsibilities of the fitted components for x.")
		.def("release_device", &ml::EMPy::release_device, py::arg("keep_results") = true, "Frees the GPU memory the last fit still holds (the points and the pending results); with keep_results the responsibilities and labels are brought to the host first.")
		.def("assign_responsibilities_batch", &ml::EMPy::calculate_responsibilities_batch, py::arg("data").noconvert(),
			"Responsibilities of the fitted components for every row of data (computed on the GPU).\n\nArgs:\n    data: A 2D float64 C-contiguous array with data points in rows.\n\nReturns:\n    2D array, one row of responsibilities per data point.")
		.def("score_samples", &ml::EMPy::score_samples_py, py::arg("data").noconvert() = py::none(),
			"Log-likelihood log p(x) of every point under the fitted mixture (computed on the GPU), as sklearn's GaussianMixture.score_samples.\n\nArgs:\n    data: A 2D float64 C-contiguous array of shape (m, D) with points in rows, or None for the fitted points (still on the GPU).\n\nReturns:\n    Array of shape (m,).")
		.def("score", &ml::EMPy::score_py, py::arg("data").noconvert() = py::none(),
			"Mean log-likelihood per point under the fitted mixture, as sklearn's GaussianMixture.score.  With data=None it is the log-likelihood of the parameters the fit returned (the log_likelihood property belongs to the parameters before the last M-step).\n\nArgs:\n    data: A 2D float64 C-contiguous array of shape (m, D), or None for the fitted points.")
		.def("bic", [](const ml::EMPy& em, const py::object& data) { return em.information_criterion(data, true); }, py::arg("data").noconvert() = py::none(),
			"Bayesian information criterion -2 n score(data) + p ln n, p = K D + K D (D + 1) / 2 + K - 1 free parameters (sklearn's definition).\n\nArgs:\n    data: A 2D float64 C-contiguous array of shape (n, D), or None for the fitted points.")
		.def("aic", [](const ml::EMPy& em, const py::object& data) { return em.information_criterion(data, false); }, py::arg("data").noconvert() = py::none(),
			"Akaike information criterion -2 n score(data) + 2 p (sklearn's definition).\n\nArgs:\n    data: A 2D float64 C-contiguous array of shape (n, D), or None for the fitted points.")
		.doc() = "Full-covariance Gaussian mixture fitted by expectation-maximisation on B200 GPUs.";

	py::class_<ml::Clustering::KMeansPy, std::shared_ptr<ml::Clustering::KMeansPy>>(m_clustering, "KMeans")
		.def(py::init<unsigned int>(), py::arg("number_clusters"), "Args:\n    number_clusters: K, at least 1.")
		.def("set_seed", &ml::Clustering::KMeansPy::set_seed, py::arg("seed"), "Seeds the pseudo-random generator the initialiser draws from.")
		.def("set_absolute_tolerance", &ml::Clustering::KMeansPy::set_absolute_tolerance, py::arg("absolute_tolerance"), "Absolute part of the stopping threshold (>= 0).")
		.def("set_maximum_steps", &ml::Clustering::KMeansPy::set_maximum_steps, py::arg("maximum_steps"), "Upper bound on the number of iterations (at least 2).")
		.def("set_centroids_initialiser", &ml::Clustering::KMeansPy::set_centroids_initialiser, py::arg("centroids_initialiser"), "Chooses how the starting centroids are picked.")
		.def("set_number_initialisations", &ml::Clustering::KMeansPy::set_number_initialisations, py::arg("centroids_initialiser"), "Number of independent starts; the converged one with the smallest inertia wins.")
		.def("set_verbose", &ml::Clustering::KMeansPy::set_verbose, py::arg("verbose"), "Prints the state after every iteration when True.")
		.def("fit", &ml::Clustering::KMeansPy::fit_row_major, py::arg("data").noconvert(),
			"Runs Lloyd iterations on the GPU.\n\nArgs:\n    data: float64 C-contiguous array of shape (N, D), one point per row; used as is, never converted.\n\nReturns:\n    Whether the labels or the centroids stopped moving before maximum_steps.")
		.def_property_readonly("number_clusters", &ml::Clustering::KMeansPy::number_clusters, "K, as given to the constructor.")
		.def_property_readonly("centroids", &ml::Clustering::KMeansPy::centroids_row_major, "Centroids after the fit, shape (K, D).")
		.def_property_readonly("labels", &ml::Clustering::KMeansPy::labels, "Cluster index of every fitted point (a list, as in the reference; brought to the host on first access).")
		.def_property_readonly("labels_array", [](const ml::Clustering::KMeansPy& km) { return to_numpy(km.labels()); }, "The same as a uint32 numpy array (an addition: a Python list of 1e8 integers takes gigabytes).")
		.def_property_readonly("inertia", [](const ml::Clustering::KMeansPy& km) { return km.inertia(); }, "Sum of the squared distances of the points to their centroids.")
		.def_property_readonly("converged", &ml::Clustering::KMeansPy::converged, "Whether the last fit converged.")
		.def_property_readonly("number_iterations", &ml::Clustering::KMeansPy::number_iterations, "Assignment steps run by the last fit.")
		.def("assign_label", &ml::Clustering::KMeansPy::assign_label_py, py::arg("x"),
			"Args:\n    x: one point, D values.\n\nReturns:\n    (index of the nearest centroid, squared distance to it).")
		.def("release_device", &ml::Clustering::KMeansPy::release_device, py::arg("keep_results") = true, "Frees the GPU memory the last fit still holds; with keep_results the labels are brought to the host first.")
		.def("assign_labels", &ml::Clustering::KMeansPy::assign_labels_py, py::arg("data").noconvert(),
			"Assigns every row of data to its closest cluster (computed on the GPU).\n\nArgs:\n    data: A 2D float64 C-contiguous array with data points in rows.\n\nReturns:\n    Tuple of the array of cluster labels and the array of squared Euclidean distances to the cluster centroids.")
		.def("transform", &ml::Clustering::KMeansPy::transform_py, py::arg("data").noconvert() = py::none(),
			"Euclidean distance of every point to every centroid (computed on the GPU), as sklearn's KMeans.transform.\n\nArgs:\n    data: A 2D float64 C-contiguous array of shape (m, D) with points in rows, or None for the fitted points (still on the GPU).\n\nReturns:\n    Array of shape (m, K).  For the fitted points that is N K 8 bytes, and the call briefly holds twice that in host memory (the result is copied into the array).")
		.def("score", &ml::Clustering::KMeansPy::score_py, py::arg("data").noconvert() = py::none(),
			"Opposite of the inertia, the sum of the squared distances of the points to their nearest centroids (computed on the GPU), as sklearn's KMeans.score.  With data=None it is the inertia of the fitted points at the centroids the fit returned (the inertia property belongs to the last assignment of the fit, which precedes the last update when the fit stops at maximum_steps).\n\nArgs:\n    data: A 2D float64 C-contiguous array of shape (m, D), or None for the fitted points.")
		.doc() = "Lloyd's K-means on B200 GPUs.";

	m.def("_standardise_features", [](const py::array& features) {
		// (N, D) row-major in, (N, D) row-major out: the same memory as the D x N column-major matrices of the C++ side
		const auto columns = as_columns(features);
		Eigen::MatrixXd result;
		{
			py::gil_scoped_release release;
			result = ml::detail::standardise_features(columns);
		}
		py::array_t<double> out({result.cols(), result.rows()});
		std::memcpy(out.mutable_data(), result.data(), sizeof(double) * static_cast<size_t>(result.size()));
		return out;
	}, py::arg("features").noconvert(), "Device part of cppyml.utils.standardise_features.");

	auto m_distributed = m.def_submodule("distributed", "One process per GPU: every rank fits its own rows, parameters are exchanged over NCCL (an addition to the reference).");
	m_distributed.def("unique_id", []() {
		const auto id = ml::Distributed::unique_id();
		return py::bytes(reinterpret_cast<const char*>(id.data()), id.size());
	}, "The 128-byte NCCL id rank 0 creates and ships to the other ranks.");
	m_distributed.def("init", [](int device, int rank, int world, const py::bytes& id) {
		const std::string raw = id;
		if (raw.size() != 128) {
			throw py::value_error("the NCCL id must have 128 bytes");
		}
		std::array<unsigned char, 128> buffer{};
		std::memcpy(buffer.data(), raw.data(), 128);
		ml::Distributed::init(device, rank, world, buffer);
	}, py::arg("device"), py::arg("rank"), py::arg("world"), py::arg("unique_id"), "Makes this process rank `rank` of `world` on CUDA device `device`; call before the first fit.");
	m_distributed.def("shard_range", [](std::int64_t n_total, int world, int rank) {
		const auto range = ml::Distributed::shard_range(n_total, world, rank);
		return py::make_tuple(range.first, range.second);
	}, py::arg("n_total"), py::arg("world"), py::arg("rank"), "Half-open range [begin, end) of the rows rank `rank` passes to fit().");
}
