// Drop-in replacement for L/include/limu/sensors/lidar/helpers/registration.hpp:10-15
// (lidar::align_clouds, lidar::ICP): same signatures; the correspondence search, residual/Jacobian,
// normal-equation reduction AND the Gauss-Newton loop run in one persistent kernel on the B200.
#ifndef REGISTRATION_HPP
#define REGISTRATION_HPP

#include "common.hpp"
#include "voxel_hash_map.hpp"

namespace lidar
{
    using SE3d = Sophus::SE3d;

    // registration.cpp:43-92
    inline SE3d align_clouds(const utils::Vec3dVector &source, const utils::Vec3dVector &target, double th)
    {
        double pose[7];
        const int64_t n = static_cast<int64_t>(source.size() < target.size() ? source.size() : target.size());
        limu_dropin::check(limu_align(limu_dropin::context(), n ? source.front().data() : nullptr, n ? target.front().data() : nullptr, n, th,
                                      nullptr, nullptr, nullptr, pose), "align_clouds");
        return limu_dropin::from_pose7(pose);
    }

    // registration.cpp:94-130
    inline SE3d ICP(VoxelHashMap &local_map, const utils::Vec3dVector &points,
                    const SE3d &init_guess, const double max_corresp_dist, const double kernel,
                    const int &icp_max_iteration, const double &est_threshold)
    {
        double init[7], pose[7];
        limu_dropin::to_pose7(init_guess, init);
        limu_dropin::check(limu_icp(local_map.handle(), points.empty() ? nullptr : points.front().data(), static_cast<int64_t>(points.size()), init,
                                    max_corresp_dist, kernel, icp_max_iteration, est_threshold, pose, nullptr, nullptr, nullptr, nullptr), "ICP");
        return limu_dropin::from_pose7(pose);
    }

    // lidar::ICP from every guess of init_guesses in one launch (limu_icp_multi; no counterpart in the reference): relocalization against
    // an existing map. Returns the pose each guess converged to and its record (iterations, converged, inliers, rms); best_index (optional)
    // receives the hypothesis with the most inliers, then the smaller rms, then the lower index (-1 without guesses).
    struct ICPMultiResult
    {
        std::vector<SE3d> poses;
        std::vector<limu_icp_hypothesis> hypotheses;
        int best = -1;
    };
    inline ICPMultiResult ICP_multi(VoxelHashMap &local_map, const utils::Vec3dVector &points, const std::vector<SE3d> &init_guesses,
                                    const double max_corresp_dist, const double kernel, const int &icp_max_iteration, const double &est_threshold)
    {
        const size_t k = init_guesses.size();
        std::vector<double> init(7 * k), poses(7 * k);
        for (size_t i = 0; i < k; ++i) limu_dropin::to_pose7(init_guesses[i], init.data() + 7 * i);
        ICPMultiResult r;
        r.hypotheses.resize(k);
        int32_t best = -1;
        limu_dropin::check(limu_icp_multi(local_map.handle(), points.empty() ? nullptr : points.front().data(), static_cast<int64_t>(points.size()),
                                          init.data(), static_cast<int32_t>(k), max_corresp_dist, kernel, icp_max_iteration, est_threshold,
                                          LIMU_ICP_REFERENCE, poses.data(), r.hypotheses.data(), &best), "ICP_multi");
        r.poses.reserve(k);
        for (size_t i = 0; i < k; ++i) r.poses.push_back(limu_dropin::from_pose7(poses.data() + 7 * i));
        r.best = best;
        return r;
    }

    // Global relocalization without a coarse pose (limu_relocalize; no counterpart in the reference): every candidate of the planar grid
    // of nx x ny x nyaw poses around `center` (x, y steps step_xy, yaw steps step_yaw; z, roll and pitch from center) is scored on the
    // device, the n_refine best (most inliers, then the smaller rms, then the lower grid index) are refined by ICP_multi and returned in that
    // order: candidates[i] holds the grid index, the coarse pose and score, and the refined pose and record; poses[i] is the refined pose.
    // best: ICP_multi's rule over the refined results.
    struct RelocalizeResult
    {
        std::vector<limu_reloc_candidate> candidates;
        std::vector<SE3d> poses;
        int best = -1;
    };
    inline RelocalizeResult relocalize(VoxelHashMap &local_map, const utils::Vec3dVector &points, const SE3d &center, const int nx, const int ny,
                                       const int nyaw, const double step_xy, const double step_yaw, const int n_refine, const double max_corresp_dist,
                                       const double kernel, const int &icp_max_iteration, const double &est_threshold)
    {
        limu_reloc_grid grid{};
        limu_dropin::to_pose7(center, grid.center);
        grid.nx = nx; grid.ny = ny; grid.nyaw = nyaw; grid.step_xy = step_xy; grid.step_yaw = step_yaw;
        RelocalizeResult r;
        r.candidates.resize(static_cast<size_t>(n_refine > 0 && n_refine <= 4096 ? n_refine : 1));
        int32_t n_out = 0, best = -1;
        limu_dropin::check(limu_relocalize(local_map.handle(), points.empty() ? nullptr : points.front().data(), static_cast<int64_t>(points.size()),
                                           &grid, n_refine, max_corresp_dist, kernel, icp_max_iteration, est_threshold, LIMU_ICP_REFERENCE,
                                           r.candidates.data(), &n_out, &best), "relocalize");
        r.candidates.resize(static_cast<size_t>(n_out));
        r.poses.reserve(r.candidates.size());
        for (const limu_reloc_candidate &c : r.candidates) r.poses.push_back(limu_dropin::from_pose7(c.pose));
        r.best = best;
        return r;
    }
}
#endif
