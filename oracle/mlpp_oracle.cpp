// ORACLE — TEST INFRASTRUCTURE ONLY.  Not part of the product path.
//
// A single-threaded CPU restatement, operation by operation, of the clustering hot path of
// romanwerpachowski/ML ("ML++"):
//     ML/EM.cpp            EM::fit, expectation_step, maximisation_step, process_covariances,
//                          calculate_sample_covariance, calculate_labels, assign_responsibilities
//     ML/KMeans.cpp        KMeans::fit, fit_once, assign_label, assignment_step, update_step
//     ML/Clustering.cpp    Forgy, RandomPartition, KPP, ClosestCentroid
//     ML/LinearAlgebra.cpp xAx_symmetric, xxT, add_a_xxT
// Each function cites the reference lines it follows.  Only tests/, __graft_entry__.smoke() and
// bench.py's cpu_baseline / --impl reference legs may load this library, and only as the checker
// or the timed CPU baseline — never as something the product path falls back on.
//
// Why C++ and not plain C: the reference's initialisers draw from libstdc++ <random>
// (std::default_random_engine = minstd_rand0, std::sample, std::uniform_int_distribution,
// std::discrete_distribution).  Using the very same std:: facilities with the same g++ is the only
// way to reproduce its PRNG stream bit for bit.  Everything else is plain loops over raw arrays.
//
// PARITY STATUS: pinned bit for bit (with -ffp-contract=off; 1e-13 with release flags) against the reference's own
// sources compiled with a first-party Eigen stand-in (oracle/_ref, tests/test_oracle_vs_reference.py).  The reference
// against REAL Eigen cannot be compiled here (Eigen 3 is neither installed nor
// vendored; SConstruct:24), so the parts of the arithmetic that live inside Eigen are restated from
// Eigen's documented algorithms with *sequential* summation:
//     - dense products / reductions (EM.cpp:211, 216, 229, 238, 267-268; squaredNorm call sites),
//     - LLT::compute (Eigen's unblocked left-looking Cholesky, used for n < 32; the blocked variant
//       for n >= 32 differs only in summation order),
//     - LLT::solve(Identity) (forward then backward substitution),
//     - selfadjointView<Upper> * x for D >= 15 (LinearAlgebra.cpp:29).
// Eigen's internal (vectorised) summation order is "parity unpinned"; differences are O(1e-13)
// relative.  The oracle IS pinned by the reference's own tests restated in tests/ (ground-truth
// recovery, K=1 mean, N==K exact fit, label/inertia identities) and by the sklearn cross-check of
// cppyml/tests/test_clustering.py:47-67 (log-likelihood equal to sklearn's within 1e-10).
//
// Matrices are column-major, exactly like Eigen::MatrixXd: data is D x N (a point per column).
//
// Build (see oracle/Makefile):  g++ -O2 -march=native -std=c++17 -shared -fPIC
// (the reference's release flags, SConstruct:21,25: -O2 -flto -march=native).

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <iterator>
#include <limits>
#include <numeric>
#include <random>
#include <vector>

namespace {

using Index = std::ptrdiff_t;  // Eigen::Index

// Column-major dense matrix, the minimum needed here.
struct Mat {
    Index rows = 0, cols = 0;
    std::vector<double> a;
    void resize(Index r, Index c) { rows = r; cols = c; a.resize(static_cast<size_t>(r * c)); }
    void set_zero() { std::fill(a.begin(), a.end(), 0.0); }
    double& operator()(Index i, Index j) { return a[static_cast<size_t>(i + j * rows)]; }
    double operator()(Index i, Index j) const { return a[static_cast<size_t>(i + j * rows)]; }
    double* col(Index j) { return a.data() + j * rows; }
    const double* col(Index j) const { return a.data() + j * rows; }
};

// Read-only view of column-major data with an outer stride (Eigen::Ref<const MatrixXd>).
struct DataRef {
    const double* p;
    Index rows, cols, ld;
    const double* col(Index j) const { return p + j * ld; }
};

inline double squared_distance(const double* x, const double* c, Index d)
{
    // (x - c).squaredNorm()            Clustering.cpp:47,78,81; KMeans.cpp:158
    double s = 0;
    for (Index l = 0; l < d; ++l) {
        const double t = x[l] - c[l];
        s += t * t;
    }
    return s;
}

// ---------------------------------------------------------------- LinearAlgebra.cpp

// LinearAlgebra.cpp:8-31
double xAx_symmetric(const Mat& A, const double* x)
{
    const Index dim = A.rows;
    if (dim < 15) {
        double sum = 0;
        for (Index i = 0; i < dim; ++i) {
            const double x_i = x[i];
            sum += A(i, i) * x_i * x_i;
            for (Index j = 0; j < i; ++j) {
                sum += 2 * A(j, i) * x_i * x[j];
            }
        }
        return sum;
    }
    // x^T * A.selfadjointView<Upper>() * x, evaluated as (A_sym x) . x, upper triangle only.
    double result = 0;
    for (Index i = 0; i < dim; ++i) {
        double t = 0;
        for (Index j = 0; j < dim; ++j) {
            const double a_ij = (j >= i) ? A(i, j) : A(j, i);
            t += a_ij * x[j];
        }
        result += t * x[i];
    }
    return result;
}

// LinearAlgebra.cpp:33-52
void xxT(const double* x, Index dim, Mat& dest)
{
    if (dest.rows != dim || dest.cols != dim) dest.resize(dim, dim);
    for (Index i = 0; i < dim; ++i) {
        const double x_i = x[i];
        dest(i, i) = x_i * x_i;
        for (Index j = 0; j < i; ++j) {
            const double x_i_x_j = x_i * x[j];
            dest(i, j) = x_i_x_j;
            dest(j, i) = x_i_x_j;
        }
    }
}

// LinearAlgebra.cpp:54-73
void add_a_xxT(const double* x, Mat& dest, double a)
{
    const Index dim = dest.rows;
    if (dim < 14) {
        for (Index i = 0; i < dim; ++i) {
            const double x_i = x[i];
            dest(i, i) += a * x_i * x_i;
            for (Index j = 0; j < i; ++j) {
                const double a_x_i_x_j = a * x_i * x[j];
                dest(i, j) += a_x_i_x_j;
                dest(j, i) += a_x_i_x_j;
            }
        }
    } else {
        // dest.noalias() += a * x * x^T : Eigen evaluates (a*x) once, then a column at a time.
        std::vector<double> ax(static_cast<size_t>(dim));
        for (Index i = 0; i < dim; ++i) ax[static_cast<size_t>(i)] = a * x[i];
        for (Index j = 0; j < dim; ++j) {
            const double x_j = x[j];
            for (Index i = 0; i < dim; ++i) dest(i, j) += x_j * ax[static_cast<size_t>(i)];
        }
    }
}

// ---------------------------------------------------------------- Clustering.cpp

enum InitKind : int { INIT_FORGY = 0, INIT_RANDOM_PARTITION = 1, INIT_KPP = 2, INIT_EXPLICIT = 3 };

// Clustering.cpp:16-25
void forgy_init(const DataRef& data, std::default_random_engine& prng, unsigned k, Mat& centroids)
{
    std::vector<Index> all_indices(static_cast<size_t>(data.cols));
    std::iota(all_indices.begin(), all_indices.end(), 0);
    std::vector<Index> sampled_indices;
    std::sample(all_indices.begin(), all_indices.end(), std::back_inserter(sampled_indices), k, prng);
    for (unsigned i = 0; i < k; ++i) {
        std::memcpy(centroids.col(i), data.col(sampled_indices[i]), sizeof(double) * static_cast<size_t>(data.rows));
    }
}

// Clustering.cpp:27-37
void random_partition_init(const DataRef& data, std::default_random_engine& prng, unsigned k, Mat& centroids)
{
    centroids.set_zero();
    std::vector<unsigned> counters(k, 0);
    std::uniform_int_distribution<unsigned int> dist(0, k - 1);
    for (Index i = 0; i < data.cols; ++i) {
        const auto c = dist(prng);
        const double num = static_cast<double>(++counters[c]);
        double* cc = centroids.col(c);
        const double* x = data.col(i);
        for (Index l = 0; l < data.rows; ++l) cc[l] += (x[l] - cc[l]) / num;
    }
}

// Clustering.cpp:39-59
void kpp_init(const DataRef& data, std::default_random_engine& prng, unsigned k, Mat& centroids)
{
    std::vector<double> weights(static_cast<size_t>(data.cols));
    for (unsigned n = 0; n < k; ++n) {
        if (n) {
            for (Index i = 0; i < data.cols; ++i) {
                double min_distance_squared = std::numeric_limits<double>::infinity();
                for (unsigned c = 0; c < n; ++c) {
                    const double distance_squared = squared_distance(data.col(i), centroids.col(c), data.rows);
                    min_distance_squared = std::min(min_distance_squared, distance_squared);
                }
                weights[static_cast<size_t>(i)] = min_distance_squared;
            }
        } else {
            std::fill(weights.begin(), weights.end(), 1);
        }
        std::discrete_distribution<Index> dist(weights.begin(), weights.end());
        const auto new_mean_idx = dist(prng);
        std::memcpy(centroids.col(n), data.col(new_mean_idx), sizeof(double) * static_cast<size_t>(data.rows));
    }
}

void centroids_init(int kind, const DataRef& data, std::default_random_engine& prng, unsigned k,
                    const double* explicit_means, Mat& centroids)
{
    switch (kind) {
    case INIT_FORGY: forgy_init(data, prng, k, centroids); break;
    case INIT_RANDOM_PARTITION: random_partition_init(data, prng, k, centroids); break;
    case INIT_KPP: kpp_init(data, prng, k, centroids); break;
    default:
        // A user-supplied CentroidsInitialiser (Clustering.hpp:58-72) that copies fixed means.
        std::memcpy(centroids.a.data(), explicit_means, sizeof(double) * centroids.a.size());
    }
}

// Clustering.cpp:72-89
void closest_centroid_init(int centroid_kind, const DataRef& data, std::default_random_engine& prng, unsigned k,
                           const double* explicit_means, Mat& responsibilities)
{
    Mat centroids;
    centroids.resize(data.rows, k);
    centroids_init(centroid_kind, data, prng, k, explicit_means, centroids);
    responsibilities.set_zero();
    for (Index i = 0; i < data.cols; ++i) {
        double min_distance_squared = squared_distance(data.col(i), centroids.col(0), data.rows);
        unsigned closest_mean_index = 0;
        for (unsigned c = 1; c < k; ++c) {
            const double distance_squared = squared_distance(data.col(i), centroids.col(c), data.rows);
            if (distance_squared < min_distance_squared) {
                min_distance_squared = distance_squared;
                closest_mean_index = c;
            }
        }
        responsibilities(i, closest_mean_index) = 1;
    }
}

// ---------------------------------------------------------------- Eigen::LLT restated

// Eigen's unblocked lower Cholesky (left-looking, a column at a time).  Returns false if a pivot
// is not positive, leaving `L` partially factorised exactly as Eigen would.
bool llt_compute(const Mat& A, Mat& L)
{
    const Index n = A.rows;
    L = A;
    for (Index k = 0; k < n; ++k) {
        double x = L(k, k);
        double sq = 0;
        for (Index j = 0; j < k; ++j) sq += L(k, j) * L(k, j);
        if (k > 0) x -= sq;
        if (!(x > 0)) return false;
        x = std::sqrt(x);
        L(k, k) = x;
        for (Index i = k + 1; i < n; ++i) {
            double dot = 0;
            for (Index j = 0; j < k; ++j) dot += L(i, j) * L(k, j);
            double v = L(i, k);
            if (k > 0) v -= dot;
            L(i, k) = v / x;
        }
    }
    return true;
}

// llt.solve(Identity): L Y = I, then L^T X = Y, column by column.
void llt_solve_identity(const Mat& L, Mat& X)
{
    const Index n = L.rows;
    X.resize(n, n);
    X.set_zero();
    for (Index c = 0; c < n; ++c) {
        double* x = X.col(c);
        x[c] = 1;
        for (Index i = 0; i < n; ++i) {
            double v = x[i];
            for (Index j = 0; j < i; ++j) v -= L(i, j) * x[j];
            x[i] = v / L(i, i);
        }
        for (Index i = n - 1; i >= 0; --i) {
            double v = x[i];
            for (Index j = i + 1; j < n; ++j) v -= L(j, i) * x[j];
            x[i] = v / L(i, i);
        }
    }
}

// ---------------------------------------------------------------- EM.cpp

constexpr double PI = 3.14159265358979323846;  // EM.cpp:13

struct EM {
    // EM.cpp:18-37 (defaults)
    std::default_random_engine prng;
    unsigned number_components;
    int means_init_kind = INIT_FORGY;
    int resp_init_centroid_kind = INIT_FORGY;  // ClosestCentroid keeps the constructor-time Forgy (EM.cpp:19-20)
    const double* explicit_means = nullptr;
    double absolute_tolerance = 1e-8;
    double relative_tolerance = 1e-8;
    unsigned maximum_steps = 1000;
    bool maximise_first = false;

    std::vector<double> mixing_probabilities;
    Mat means;
    Mat responsibilities;
    std::vector<double> work_vector;
    std::vector<Mat> covariances, inverse_covariances, cholesky;
    std::vector<double> sqrt_covariance_determinants;
    std::vector<unsigned> labels;
    double log_likelihood = 0;
    bool converged = false;
    unsigned iterations = 0;              // not stored by the reference; step + 1 at the break
    std::vector<double> step_seconds;     // timing hook for the CPU baseline

    explicit EM(unsigned k)
        : number_components(k), mixing_probabilities(k), covariances(k), inverse_covariances(k), cholesky(k),
          sqrt_covariance_determinants(k) {}

    // EM.cpp:274-287
    void process_covariances()
    {
        for (unsigned k = 0; k < number_components; ++k) {
            llt_compute(covariances[k], cholesky[k]);
            llt_solve_identity(cholesky[k], inverse_covariances[k]);
            double sqrt_covariance_determinant = 1;
            for (Index i = 0; i < covariances[k].rows; ++i) sqrt_covariance_determinant *= cholesky[k](i, i);
            sqrt_covariance_determinants[k] = sqrt_covariance_determinant;
        }
    }

    // EM.cpp:265-272
    static Mat calculate_sample_covariance(const DataRef& data)
    {
        const Index d = data.rows, n = data.cols;
        std::vector<double> mean(static_cast<size_t>(d), 0.0);
        for (Index l = 0; l < d; ++l) {
            double s = 0;
            for (Index i = 0; i < n; ++i) s += data.col(i)[l];
            mean[static_cast<size_t>(l)] = s / static_cast<double>(n);
        }
        Mat centred;
        centred.resize(d, n);
        for (Index i = 0; i < n; ++i)
            for (Index l = 0; l < d; ++l) centred(l, i) = data.col(i)[l] - mean[static_cast<size_t>(l)];
        Mat covariance;
        covariance.resize(d, d);
        for (Index a = 0; a < d; ++a)
            for (Index b = 0; b < d; ++b) {
                double s = 0;
                for (Index i = 0; i < n; ++i) s += centred(a, i) * centred(b, i);
                covariance(a, b) = s / static_cast<double>(n - 1);
            }
        return covariance;
    }

    // EM.cpp:190-219
    void expectation_step(const DataRef& data)
    {
        const Index number_dimensions = data.rows;
        const Index sample_size = data.cols;
        static const double log_2_pi = std::log(2. * PI);
        const double log_likelihood_normalisation_constant = static_cast<double>(number_dimensions) * log_2_pi / 2;
        for (unsigned k = 0; k < number_components; ++k) {
            const double* mean = means.col(k);
            double* component_weights = responsibilities.col(k);
            const Mat& inverse_covariance = inverse_covariances[k];
            for (Index i = 0; i < sample_size; ++i) {
                const double* x = data.col(i);
                for (Index l = 0; l < number_dimensions; ++l) work_vector[static_cast<size_t>(l)] = x[l] - mean[l];
                component_weights[i] = std::exp(-0.5 * xAx_symmetric(inverse_covariance, work_vector.data()));
            }
            const double scale = mixing_probabilities[k] / sqrt_covariance_determinants[k];
            for (Index i = 0; i < sample_size; ++i) component_weights[i] *= scale;
        }
        // responsibilities_.rowwise().sum().array().log().mean() - const      EM.cpp:211
        double sum_logs = 0;
        for (Index i = 0; i < sample_size; ++i) {
            double row_sum = 0;
            for (unsigned k = 0; k < number_components; ++k) row_sum += responsibilities(i, k);
            sum_logs += std::log(row_sum);
        }
        log_likelihood = sum_logs / static_cast<double>(sample_size) - log_likelihood_normalisation_constant;
        // EM.cpp:214-218
        for (Index i = 0; i < sample_size; ++i) {
            double sum_weights = 0;
            for (unsigned k = 0; k < number_components; ++k) sum_weights += responsibilities(i, k);
            for (unsigned k = 0; k < number_components; ++k) responsibilities(i, k) /= sum_weights;
        }
    }

    // EM.cpp:221-263
    void maximisation_step(const DataRef& data)
    {
        const Index number_dimensions = data.rows;
        const Index sample_size = data.cols;
        // means_ = data * responsibilities_  (unnormalised)                   EM.cpp:229
        means.set_zero();
        for (unsigned k = 0; k < number_components; ++k) {
            double* mean = means.col(k);
            const double* w = responsibilities.col(k);
            for (Index i = 0; i < sample_size; ++i) {
                const double* x = data.col(i);
                const double r = w[i];
                for (Index l = 0; l < number_dimensions; ++l) mean[l] += x[l] * r;
            }
        }
        for (unsigned k = 0; k < number_components; ++k) {
            Mat& covariance = covariances[k];
            for (double& v : covariance.a) v *= 0;
            const double* component_weights = responsibilities.col(k);
            double sum_component_weights = 0;
            for (Index i = 0; i < sample_size; ++i) sum_component_weights += component_weights[i];
            double* mean = means.col(k);
            for (Index l = 0; l < number_dimensions; ++l) mean[l] /= sum_component_weights;
            for (Index i = 0; i < sample_size; ++i) {
                const double* x = data.col(i);
                for (Index l = 0; l < number_dimensions; ++l) work_vector[static_cast<size_t>(l)] = x[l] - mean[l];
                add_a_xxT(work_vector.data(), covariance, component_weights[i]);
            }
            for (double& v : covariance.a) v /= sum_component_weights;
            static constexpr double epsilon = 1e-15;
            for (Index l = 0; l < number_dimensions; ++l) covariance(l, l) += epsilon;
            mixing_probabilities[k] = sum_component_weights / static_cast<double>(sample_size);
        }
        process_covariances();
    }

    // EM.cpp:289-304
    void calculate_labels()
    {
        for (Index i = 0; i < responsibilities.rows; ++i) {
            double max_responsibility = -1;
            Index label = -1;
            for (Index k = 0; k < responsibilities.cols; ++k) {
                if (responsibilities(i, k) > max_responsibility) {
                    max_responsibility = responsibilities(i, k);
                    label = k;
                }
            }
            labels[static_cast<size_t>(i)] = static_cast<unsigned>(label);
        }
    }

    // EM.cpp:176-188
    void assign_responsibilities(const double* x, double* u) const
    {
        const Index d = means.rows;
        std::vector<double> w(static_cast<size_t>(d));
        double sum = 0;
        for (unsigned k = 0; k < number_components; ++k) {
            for (Index l = 0; l < d; ++l) w[static_cast<size_t>(l)] = x[l] - means(l, k);
            u[k] = std::exp(-0.5 * xAx_symmetric(inverse_covariances[k], w.data())) * mixing_probabilities[k]
                / sqrt_covariance_determinants[k];
        }
        for (unsigned k = 0; k < number_components; ++k) sum += u[k];
        for (unsigned k = 0; k < number_components; ++k) u[k] /= sum;
    }

    // EM.cpp:91-174
    bool fit(const DataRef& data)
    {
        converged = false;
        iterations = 0;
        const auto number_dimensions = static_cast<unsigned>(data.rows);
        const auto sample_size = static_cast<unsigned>(data.cols);
        means.resize(number_dimensions, number_components);
        responsibilities.resize(sample_size, number_components);
        std::fill(mixing_probabilities.begin(), mixing_probabilities.end(), 1. / static_cast<double>(number_components));
        labels.resize(sample_size);
        if (sample_size == number_components) {
            responsibilities.set_zero();
            for (unsigned i = 0; i < sample_size; ++i) {
                responsibilities(i, i) = 1;
                std::memcpy(means.col(i), data.col(i), sizeof(double) * number_dimensions);
                covariances[i].resize(number_dimensions, number_dimensions);
                covariances[i].set_zero();
                log_likelihood = std::numeric_limits<double>::infinity();
                labels[i] = i;
            }
            converged = true;
            return converged;
        }
        work_vector.resize(number_dimensions);
        if (maximise_first) {
            closest_centroid_init(resp_init_centroid_kind, data, prng, number_components, explicit_means, responsibilities);
            for (unsigned k = 0; k < number_components; ++k) {
                covariances[k].resize(number_dimensions, number_dimensions);
                covariances[k].set_zero();
            }
            maximisation_step(data);
        } else {
            centroids_init(means_init_kind, data, prng, number_components, explicit_means, means);
            const Mat sample_covariance = calculate_sample_covariance(data);
            for (unsigned k = 0; k < number_components; ++k) covariances[k] = sample_covariance;
            process_covariances();
        }
        double old_log_likelihood = -std::numeric_limits<double>::infinity();
        for (unsigned step = 0; step < maximum_steps; ++step) {
            const auto t0 = std::chrono::steady_clock::now();
            expectation_step(data);
            maximisation_step(data);
            step_seconds.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
            iterations = step + 1;
            if (step > 0) {
                const double ll_change = std::abs(log_likelihood - old_log_likelihood);
                if (ll_change < absolute_tolerance
                        + relative_tolerance * std::max(std::abs(old_log_likelihood), std::abs(log_likelihood))) {
                    calculate_labels();
                    converged = true;
                    break;
                }
            }
            old_log_likelihood = log_likelihood;
        }
        return converged;
    }
};

// ---------------------------------------------------------------- KMeans.cpp

struct KMeans {
    std::vector<unsigned> labels, old_labels;
    Mat centroids, old_centroids;
    std::vector<double> work_vector;
    std::default_random_engine prng;
    int init_kind = INIT_FORGY;
    const double* explicit_means = nullptr;
    double absolute_tolerance = 1e-8;
    double inertia = 0;
    unsigned maximum_steps = 1000;
    unsigned num_inits = 1;
    unsigned num_clusters;
    bool converged = false;
    unsigned iterations = 0;          // assignment steps executed by the last fit_once
    std::vector<double> step_seconds;

    explicit KMeans(unsigned k) : work_vector(k), num_clusters(k) {}

    // KMeans.cpp:153-165
    std::pair<unsigned, double> assign_label(const double* x) const
    {
        double min_squared_distance = std::numeric_limits<double>::infinity();
        unsigned label = 0;
        for (unsigned k = 0; k < num_clusters; ++k) {
            const double sq = squared_distance(x, centroids.col(k), centroids.rows);
            if (sq < min_squared_distance) {
                min_squared_distance = sq;
                label = k;
            }
        }
        return std::make_pair(label, min_squared_distance);
    }

    // KMeans.cpp:167-178
    void assignment_step(const DataRef& data)
    {
        old_labels.swap(labels);
        inertia = 0;
        for (Index i = 0; i < data.cols; ++i) {
            const auto label_and_distance = assign_label(data.col(i));
            labels[static_cast<size_t>(i)] = label_and_distance.first;
            inertia += label_and_distance.second;
        }
    }

    // KMeans.cpp:180-192
    void update_step(const DataRef& data)
    {
        std::fill(work_vector.begin(), work_vector.end(), 0.0);
        std::swap(old_centroids, centroids);
        centroids.set_zero();
        for (Index i = 0; i < data.cols; ++i) {
            const unsigned label = labels[static_cast<size_t>(i)];
            const double num = (++work_vector[label]);
            double* c = centroids.col(label);
            const double* x = data.col(i);
            for (Index l = 0; l < data.rows; ++l) c[l] += (x[l] - c[l]) / num;
        }
    }

    // KMeans.cpp:50-114
    bool fit_once(const DataRef& data)
    {
        converged = false;
        iterations = 0;
        const auto number_dimensions = static_cast<unsigned>(data.rows);
        const auto sample_size = static_cast<unsigned>(data.cols);
        centroids.resize(number_dimensions, num_clusters);
        old_centroids.resize(number_dimensions, num_clusters);
        labels.resize(sample_size);
        old_labels.resize(sample_size);
        if (sample_size == num_clusters) {
            for (unsigned i = 0; i < sample_size; ++i) {
                std::memcpy(centroids.col(i), data.col(i), sizeof(double) * number_dimensions);
                labels[i] = i;
            }
            inertia = 0;
            converged = true;
            return converged;
        }
        centroids_init(init_kind, data, prng, num_clusters, explicit_means, centroids);
        for (unsigned step = 0; step < maximum_steps; ++step) {
            const auto t0 = std::chrono::steady_clock::now();
            assignment_step(data);
            iterations = step + 1;
            if (step > 0) {
                if (old_labels == labels) {
                    converged = true;
                    break;
                }
            }
            update_step(data);
            step_seconds.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
            if (step > 0) {
                double centroid_shift = 0;
                for (size_t e = 0; e < centroids.a.size(); ++e) {
                    const double t = centroids.a[e] - old_centroids.a[e];
                    centroid_shift += t * t;
                }
                if (centroid_shift < absolute_tolerance) {
                    assignment_step(data);
                    converged = true;
                    break;
                }
            }
        }
        return converged;
    }

    // KMeans.cpp:25-48
    bool fit(const DataRef& data)
    {
        if (num_inits == 1) return fit_once(data);
        converged = false;
        double min_inertia = std::numeric_limits<double>::infinity();
        Mat best_centroids;
        for (unsigned i = 0; i < num_inits; ++i) {
            if (fit_once(data)) {
                if (inertia < min_inertia) {
                    min_inertia = inertia;
                    best_centroids = centroids;
                }
                converged = true;
            }
        }
        if (converged) {
            centroids = best_centroids;
            assignment_step(data);
        }
        return converged;
    }
};

}  // namespace

// ======================================================================= C interface (ctypes)

extern "C" {

struct mlpp_oracle_em_options {
    unsigned seed;              // used only if set_seed != 0 (a default-constructed engine otherwise)
    int set_seed;
    double absolute_tolerance;
    double relative_tolerance;
    unsigned maximum_steps;
    int means_init_kind;        // 0 Forgy, 1 RandomPartition, 2 KPP, 3 explicit means
    int resp_init_centroid_kind;
    int maximise_first;
    const double* explicit_means;  // D x K column-major, for kind 3
};

struct mlpp_oracle_em_result {
    double* means;              // D x K             (may be NULL)
    double* covariances;        // K blocks of D x D (may be NULL)
    double* mixing_probabilities;  // K              (may be NULL)
    double* responsibilities;   // N x K column-major (may be NULL)
    unsigned* labels;           // N                 (may be NULL)
    double* inverse_covariances;   // K blocks of D x D (may be NULL)
    double* sqrt_covariance_determinants;  // K (may be NULL)
    double* step_seconds;       // maximum_steps entries (may be NULL)
    double log_likelihood;
    int converged;
    unsigned iterations;
};

// ml::EM::fit on column-major D x N data with outer stride ld.  Returns 0, or 1 for the argument
// errors on which the reference throws std::invalid_argument (EM.cpp:96-101, 18-37).
int mlpp_oracle_em_fit(const double* data, int64_t d, int64_t n, int64_t ld, unsigned k,
                       const mlpp_oracle_em_options* opt, mlpp_oracle_em_result* out)
{
    if (k == 0 || d <= 0 || n < static_cast<int64_t>(k)) return 1;
    EM em(k);
    if (opt->set_seed) em.prng.seed(opt->seed);
    em.absolute_tolerance = opt->absolute_tolerance;
    em.relative_tolerance = opt->relative_tolerance;
    em.maximum_steps = opt->maximum_steps;
    em.means_init_kind = opt->means_init_kind;
    em.resp_init_centroid_kind = opt->resp_init_centroid_kind;
    em.maximise_first = opt->maximise_first != 0;
    em.explicit_means = opt->explicit_means;
    const DataRef ref{data, d, n, ld};
    em.fit(ref);
    const size_t D = static_cast<size_t>(d), K = k, N = static_cast<size_t>(n);
    if (out->means) std::memcpy(out->means, em.means.a.data(), sizeof(double) * D * K);
    for (size_t c = 0; c < K; ++c) {
        if (out->covariances && em.covariances[c].a.size() == D * D)
            std::memcpy(out->covariances + c * D * D, em.covariances[c].a.data(), sizeof(double) * D * D);
        if (out->inverse_covariances && em.inverse_covariances[c].a.size() == D * D)
            std::memcpy(out->inverse_covariances + c * D * D, em.inverse_covariances[c].a.data(), sizeof(double) * D * D);
    }
    if (out->mixing_probabilities) std::memcpy(out->mixing_probabilities, em.mixing_probabilities.data(), sizeof(double) * K);
    if (out->sqrt_covariance_determinants)
        std::memcpy(out->sqrt_covariance_determinants, em.sqrt_covariance_determinants.data(), sizeof(double) * K);
    if (out->responsibilities) std::memcpy(out->responsibilities, em.responsibilities.a.data(), sizeof(double) * N * K);
    if (out->labels) std::memcpy(out->labels, em.labels.data(), sizeof(unsigned) * N);
    if (out->step_seconds)
        for (size_t s = 0; s < em.step_seconds.size() && s < opt->maximum_steps; ++s) out->step_seconds[s] = em.step_seconds[s];
    out->log_likelihood = em.log_likelihood;
    out->converged = em.converged ? 1 : 0;
    out->iterations = em.iterations;
    return 0;
}

// EM::assign_responsibilities (EM.cpp:176-188) from explicit post-fit parameters.
void mlpp_oracle_em_assign_responsibilities(const double* x, int64_t d, unsigned k, const double* means,
                                            const double* inverse_covariances, const double* mixing_probabilities,
                                            const double* sqrt_covariance_determinants, double* u)
{
    EM em(k);
    em.means.resize(d, k);
    std::memcpy(em.means.a.data(), means, sizeof(double) * static_cast<size_t>(d) * k);
    for (unsigned c = 0; c < k; ++c) {
        em.inverse_covariances[c].resize(d, d);
        std::memcpy(em.inverse_covariances[c].a.data(), inverse_covariances + static_cast<size_t>(c) * d * d,
                    sizeof(double) * static_cast<size_t>(d * d));
        em.mixing_probabilities[c] = mixing_probabilities[c];
        em.sqrt_covariance_determinants[c] = sqrt_covariance_determinants[c];
    }
    em.assign_responsibilities(x, u);
}

struct mlpp_oracle_kmeans_options {
    unsigned seed;
    int set_seed;
    double absolute_tolerance;
    unsigned maximum_steps;
    unsigned number_initialisations;
    int init_kind;
    const double* explicit_means;
};

struct mlpp_oracle_kmeans_result {
    double* centroids;      // D x K (may be NULL)
    unsigned* labels;       // N (may be NULL)
    double* step_seconds;   // maximum_steps entries (may be NULL)
    double inertia;
    int converged;
    unsigned iterations;
};

int mlpp_oracle_kmeans_fit(const double* data, int64_t d, int64_t n, int64_t ld, unsigned k,
                           const mlpp_oracle_kmeans_options* opt, mlpp_oracle_kmeans_result* out)
{
    if (k == 0 || d <= 0 || n < static_cast<int64_t>(k)) return 1;
    KMeans km(k);
    if (opt->set_seed) km.prng.seed(opt->seed);
    km.absolute_tolerance = opt->absolute_tolerance;
    km.maximum_steps = opt->maximum_steps;
    km.num_inits = opt->number_initialisations;
    km.init_kind = opt->init_kind;
    km.explicit_means = opt->explicit_means;
    const DataRef ref{data, d, n, ld};
    km.fit(ref);
    if (out->centroids) std::memcpy(out->centroids, km.centroids.a.data(), sizeof(double) * static_cast<size_t>(d) * k);
    if (out->labels) std::memcpy(out->labels, km.labels.data(), sizeof(unsigned) * static_cast<size_t>(n));
    if (out->step_seconds)
        for (size_t s = 0; s < km.step_seconds.size() && s < opt->maximum_steps; ++s) out->step_seconds[s] = km.step_seconds[s];
    out->inertia = km.inertia;
    out->converged = km.converged ? 1 : 0;
    out->iterations = km.iterations;
    return 0;
}

// KMeans::assign_label (KMeans.cpp:153-165) against explicit centroids.
unsigned mlpp_oracle_kmeans_assign_label(const double* x, int64_t d, unsigned k, const double* centroids, double* sq_out)
{
    KMeans km(k);
    km.centroids.resize(d, k);
    std::memcpy(km.centroids.a.data(), centroids, sizeof(double) * static_cast<size_t>(d) * k);
    const auto r = km.assign_label(x);
    if (sq_out) *sq_out = r.second;
    return r.first;
}

// KMeans::assign_label for m points (column-major D x m) with the distance summed as a chain of fused multiply-adds,
// s = fma(t, t, s) over the dimensions in order: the evaluation of the device's exact refinement (kmeans.cu,
// exact_distance), which differs from the unfused sum above in the last bits.  Same scan: strict <, lowest index wins.
void mlpp_oracle_kmeans_assign_fused(const double* x, int64_t d, int64_t m, unsigned k, const double* centroids, unsigned* labels,
                                     double* sq_out)
{
    for (int64_t i = 0; i < m; ++i) {
        const double* xi = x + i * d;
        double best = std::numeric_limits<double>::infinity();
        unsigned label = 0;
        for (unsigned c = 0; c < k; ++c) {
            const double* cc = centroids + static_cast<int64_t>(c) * d;
            double sq = 0;
            for (int64_t l = 0; l < d; ++l) {
                const double t = xi[l] - cc[l];
                sq = std::fma(t, t, sq);
            }
            if (sq < best) {
                best = sq;
                label = c;
            }
        }
        labels[i] = label;
        sq_out[i] = best;
    }
}

// The initialisers on their own (Clustering.cpp:16-59), for PRNG-stream parity tests of the
// product's host classes.  `seed` as in set_seed(); a default-constructed engine if !set_seed.
void mlpp_oracle_centroids_init(int kind, const double* data, int64_t d, int64_t n, int64_t ld, unsigned k,
                                unsigned seed, int set_seed, double* centroids)
{
    std::default_random_engine prng;
    if (set_seed) prng.seed(seed);
    Mat c;
    c.resize(d, k);
    const DataRef ref{data, d, n, ld};
    centroids_init(kind, ref, prng, k, nullptr, c);
    std::memcpy(centroids, c.a.data(), sizeof(double) * c.a.size());
}

// LinearAlgebra.cpp helpers, for the identities of Tests/test_LinearAlgebra.cpp.
double mlpp_oracle_xAx_symmetric(const double* A, int64_t dim, const double* x)
{
    Mat m;
    m.resize(dim, dim);
    std::memcpy(m.a.data(), A, sizeof(double) * static_cast<size_t>(dim * dim));
    return xAx_symmetric(m, x);
}

void mlpp_oracle_xxT(const double* x, int64_t dim, double* dest)
{
    Mat m;
    xxT(x, dim, m);
    std::memcpy(dest, m.a.data(), sizeof(double) * static_cast<size_t>(dim * dim));
}

void mlpp_oracle_add_a_xxT(const double* x, int64_t dim, double* dest, double a)
{
    Mat m;
    m.resize(dim, dim);
    std::memcpy(m.a.data(), dest, sizeof(double) * static_cast<size_t>(dim * dim));
    add_a_xxT(x, m, a);
    std::memcpy(dest, m.a.data(), sizeof(double) * static_cast<size_t>(dim * dim));
}

// ---------------------------------------------------------------- test-data generators
// The data sets the reference's own tests and benchmarks draw, with the same libstdc++ calls, so
// that the pins of SURVEY.md §4 run on identical numbers.

// Tests/test_EM.cpp:10-34 and Tests/test_KMeans.cpp:10-37: 400 points, D=3, two diagonal
// Gaussians, default-seeded engine.  data is 3 x 400 column-major; ground_truth may be NULL.
void mlpp_oracle_testdata_two_gaussians(double* data, unsigned* ground_truth)
{
    std::default_random_engine rng;
    std::uniform_real_distribution<double> u01(0, 1);
    std::normal_distribution<double> standard_normal;
    const unsigned num_dimensions = 3, sample_size = 400;
    constexpr double p0 = 0.25;
    const double means[3][2] = {{0.4, -1.2}, {0.11, 2.2}, {0.5, 1.6}};
    const double sigmas[3][2] = {{0.05, 0.2}, {0.04, 0.1}, {0.01, 0.2}};
    for (unsigned i = 0; i < sample_size; ++i) {
        const unsigned k = u01(rng) < p0 ? 0 : 1;
        if (ground_truth) ground_truth[i] = k;
        for (unsigned l = 0; l < num_dimensions; ++l) {
            data[l + i * num_dimensions] = standard_normal(rng) * sigmas[l][k] + means[l][k];
        }
    }
}

// Benchmarks/bm_EM.cpp:11-34, bm_KMeans.cpp, Demo/clustering_demo.cpp:14-37: the "mouse" data,
// D=2, three uniform discs, default-seeded engine.  data is 2 x n column-major.
void mlpp_oracle_testdata_mouse(double* data, unsigned* classes, unsigned sample_size)
{
    std::default_random_engine rng;
    std::uniform_real_distribution<double> u01(0, 1);
    const double face_radius = 1;
    const double ear_radius = 0.3;
    const std::vector<double> radii{face_radius, ear_radius, ear_radius};
    std::discrete_distribution<unsigned int> component_distr{face_radius * face_radius, 2 * ear_radius * ear_radius,
                                                             2 * ear_radius * ear_radius};
    const double ear_angle = 45 * PI / 180.;
    std::vector<double> center_xs{0, -(face_radius + ear_radius) * std::sin(ear_angle), (face_radius + ear_radius) * std::sin(ear_angle)};
    std::vector<double> center_ys{0, (face_radius + ear_radius) * std::cos(ear_angle), (face_radius + ear_radius) * std::cos(ear_angle)};
    for (unsigned i = 0; i < sample_size; ++i) {
        const unsigned k = component_distr(rng);
        if (classes) classes[i] = k;
        const double phi = 2 * PI * u01(rng);
        const double r = std::sqrt(u01(rng)) * radii[k];
        data[0 + 2 * static_cast<size_t>(i)] = center_xs[k] + r * std::cos(phi);
        data[1 + 2 * static_cast<size_t>(i)] = center_ys[k] + r * std::sin(phi);
    }
}

}  // extern "C"
