#pragma once
// ml::Clustering::KMeans: Lloyd's algorithm with the reference's public surface
// (ML/KMeans.hpp:19-101) on the B200 backend.  Additions: number_iterations(); assign_labels(points), the
// batched form of assign_label(x) on the device; transform(points) and transform(), the distance of every point to
// every centroid, and inertia(points) and final_inertia(), the inertia at the returned centroids, for new points or the
// fitted ones, on the device.
#include "Clustering.hpp"
#include <memory>
#include <vector>
#include <utility>
#include <Eigen/Core>
#include "dll.hpp"

namespace ml
{
    namespace detail { class KmDevice; }

    namespace Clustering
    {
        class KMeans : public Model
        {
        public:
            /** @throw std::invalid_argument If `number_clusters` is zero. */
            DLL_DECLSPEC KMeans(unsigned int number_clusters);
            DLL_DECLSPEC ~KMeans() override;
            KMeans(const KMeans&) = delete;
            KMeans& operator=(const KMeans&) = delete;

            DLL_DECLSPEC bool fit(DataView data) override;

            unsigned int number_clusters() const override { return number_clusters_; }

            /** Brought from the device on first access after a fit (400 MB at N = 1e8). */
            DLL_DECLSPEC const std::vector<unsigned int>& labels() const override;

            const Eigen::MatrixXd& centroids() const override { return centroids_; }

            DLL_DECLSPEC void set_seed(unsigned int seed);

            /** Tolerance on the squared Frobenius norm of the centroid shift.
            @throw std::domain_error If negative. */
            DLL_DECLSPEC void set_absolute_tolerance(double absolute_tolerance);

            /** @throw std::invalid_argument If less than 2. */
            DLL_DECLSPEC void set_maximum_steps(unsigned int maximum_steps);

            /** @throw std::invalid_argument If zero. */
            DLL_DECLSPEC void set_number_initialisations(unsigned int number_initialisations);

            /** @throw std::invalid_argument If null. */
            DLL_DECLSPEC void set_centroids_initialiser(std::shared_ptr<const CentroidsInitialiser> centroids_initialiser);

            void set_verbose(bool verbose) { verbose_ = verbose; }

            /** Nearest centroid of x and the squared distance to it.
            @throw std::invalid_argument If x has the wrong size. */
            DLL_DECLSPEC std::pair<unsigned int, double> assign_label(PointView x) const;

            /** The same for every column of `points` (D x m) at once, on the device.
            @throw std::invalid_argument If `points` has the wrong number of rows.
            @throw std::logic_error If there is no fitted device state (no fit yet, or the N == K exact fit). */
            DLL_DECLSPEC std::pair<std::vector<unsigned int>, std::vector<double>> assign_labels(DataView points) const;

            /** Sum of squared distances of the points to their centroids, from the last assignment of the fit (when the fit
            stops at maximum_steps, that assignment came before the last update: see final_inertia()). */
            double inertia() const { return inertia_; }

            /** Euclidean distance of every column of `points` (D x m) to every centroid, m x K, on the device.
            @throw std::invalid_argument If `points` has the wrong number of rows.
            @throw std::logic_error If there is no fitted device state (no fit yet, the N == K exact fit, or after
            release_device()). */
            DLL_DECLSPEC Eigen::MatrixXd transform(DataView points) const;

            /** The same for the fitted points (this process's own points under ml::Distributed): N x K, N K 8 bytes of host
            memory (205 GB at N = 1e8, K = 256; the cppyml binding copies the result into its numpy array, so through Python
            the peak is twice that).
            @throw std::logic_error If there is no fitted device state. */
            DLL_DECLSPEC Eigen::MatrixXd transform() const;

            /** Sum over the columns of `points` of the squared distance to the nearest centroid, on the device.
            @throw std::invalid_argument If `points` has the wrong number of rows.
            @throw std::logic_error If there is no fitted device state. */
            DLL_DECLSPEC double inertia(DataView points) const;

            /** The inertia of the fitted points at the centroids the fit returned: inertia() whenever the fit ended on an
            assignment to those centroids.  Under ml::Distributed: over all ranks' points, and collective.
            @throw std::logic_error If there is no fitted device state. */
            DLL_DECLSPEC double final_inertia() const;

            bool converged() const override { return converged_; }

            /** Assignment steps executed by the last (single-initialisation) fit. */
            unsigned int number_iterations() const { return number_iterations_; }

            /** Frees the HBM-resident state of the last fit (the points stay on the device after fit() so that labels()
            and assign_labels() can be served).  `keep_results`: bring the pending labels to the host first. */
            DLL_DECLSPEC void release_device(bool keep_results = true);
        private:
            mutable std::vector<unsigned int> labels_;
            mutable bool labels_on_host_;
            Eigen::MatrixXd centroids_;
            Prng prng_;
            std::shared_ptr<const CentroidsInitialiser> centroids_initialiser_;
            double absolute_tolerance_;
            double inertia_;
            unsigned int maximum_steps_;
            unsigned int number_initialisations_;
            unsigned int number_clusters_;
            unsigned int number_iterations_;
            bool verbose_;
            bool converged_;
            mutable std::unique_ptr<detail::KmDevice> device_; /**< HBM-resident state of the last fit */

            bool fit_once(DataView data, detail::KmDevice& device);
            /** Draws the initial centroids of one start (KMeans.cpp:77). */
            void draw_initial_centroids(DataView data, detail::KmDevice& device);
            /** The starts of a multi-start fit in lockstep groups of up to four (same results as one after the other). */
            bool fit_lockstep(DataView data, detail::KmDevice& device);
        };
    }
}
