// bundle_adjustment_manager.h -- RSCalibration::BAManager with the reference's interface
// (Main_Calibration/bundle_adjustment_manager.h:7-17): ctor(intrinsics map, distortion map), StartBA(), Write().
// StartBA() hands the problem to the CUDA library through the ba_cuda_* C ABI instead of building a
// ceres::Problem (bundle_adjustment_manager.cpp:19-95).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "ba_cuda.h"
#include "bundle_adjustment.h"

namespace RSCalibration {

class BAManager {
 private:
  BALProblem bal_problem;
  std::map<std::string, cv::Mat> camera_intrinsics_map, dist_coeffs_map;
  // run-time configuration; defaults = the reference's hard-coded values
  std::string correspondence_path_ = "../Common/Correspondence/hongo/correspondence.txt";
  std::string transform_xml_path_ = "../Common/Correspondence/hongo/Camera_Transform.xml";
  std::string extrinsics_dir_ = "../Common/Calibration/Extrinsics";
  std::string point3d_path_ = "../Common/Correspondence/hongo/point3d.txt";
  std::vector<std::string> serial_numbers_ = std::vector<std::string>(SERIAL_NUMBERS, SERIAL_NUMBERS + CAMERAS);
  bool fix_base_marker_ = true;   // Main dispatch (manager.cpp:26,28,58); false = Test2's two-functor dispatch
  bool rotation_as_rvec_ = false; // Test2 writes R<i> as the 3x1 rvec (Test2_BundleAdjustment/main.cpp:128)
  bool loaded_ = false;
  int device_ = 0;
  int loss_function_ = BA_LOSS_NONE;
  double loss_scale_ = 1.0;
  ba_cuda_summary summary_{};
  std::vector<ba_cuda_iteration> iterations_;
  void Load();
  std::vector<double> Intrinsics4() const;   // fx, fy, ppx, ppy per camera, looked up by serial number

 public:
  BAManager(const std::map<std::string, cv::Mat>& camera_intrinsics_map, const std::map<std::string, cv::Mat>& dist_coeffs_map);
  void StartBA();
  void Write();

  // additions (not in the reference): what was compile-time or hard-coded there
  struct Config {
    std::string correspondence_path, transform_xml_path, extrinsics_dir, point3d_path;
    std::vector<std::string> serial_numbers;
    double marker_side = MARKER_SIDE;
    bool fix_base_marker = true, rotation_as_rvec = false;
    int device = 0;
    int loss_function = BA_LOSS_NONE;   // the reference passes NULL to AddResidualBlock (manager.cpp:38,51,68,82)
    double loss_scale = 1.0;
  };
  BAManager(const std::map<std::string, cv::Mat>& camera_intrinsics_map, const std::map<std::string, cv::Mat>& dist_coeffs_map,
            const Config& config);
  const ba_cuda_summary& summary() const { return summary_; }
  const std::vector<ba_cuda_iteration>& iterations() const { return iterations_; }
  // ceres::Covariance + GetCovarianceBlock after StartBA(), at the solved parameters and with its loss: the 6x6 covariance
  // of every camera pose (CAMERAS x 36, row-major; camera 0 is not a parameter: zeros) and of every frame pose
  // (num_times x 36).  Either output may be NULL.  Returns BA_OK or the ba_status of ba_cuda_covariance
  // (BA_ERR_RANK_DEFICIENT when the problem has a gauge freedom, e.g. no marker fixed); the message is ba_cuda_last_error().
  int Covariance(std::vector<double>* camera_cov, std::vector<double>* frame_cov);
  BALProblem& problem() { return bal_problem; }
};

}  // namespace RSCalibration
