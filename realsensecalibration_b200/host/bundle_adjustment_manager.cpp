#include "bundle_adjustment_manager.h"

#include <cstdlib>
#include <fstream>
#include <iostream>

#include "cv_storage.h"

namespace RSCalibration {

using std::cerr;
using std::cout;
using std::endl;

static void Die(const std::string& what) {  // the reference prints, PAUSEs and exit(1)s (manager.cpp:8-13)
  cerr << what << endl;
  std::exit(1);
}

void BAManager::Load() {
  if (!bal_problem.loadFile(correspondence_path_.c_str())) Die("unable to open correspondence file ");
  loaded_ = true;
}

BAManager::BAManager(const std::map<std::string, cv::Mat>& camera_intrinsics_map, const std::map<std::string, cv::Mat>& dist_coeffs_map)
    : camera_intrinsics_map(camera_intrinsics_map), dist_coeffs_map(dist_coeffs_map) {
  Load();
}

BAManager::BAManager(const std::map<std::string, cv::Mat>& camera_intrinsics_map, const std::map<std::string, cv::Mat>& dist_coeffs_map,
                     const Config& c)
    : camera_intrinsics_map(camera_intrinsics_map), dist_coeffs_map(dist_coeffs_map) {
  if (!c.correspondence_path.empty()) correspondence_path_ = c.correspondence_path;
  if (!c.transform_xml_path.empty()) transform_xml_path_ = c.transform_xml_path;
  if (!c.extrinsics_dir.empty()) extrinsics_dir_ = c.extrinsics_dir;
  if (!c.point3d_path.empty()) point3d_path_ = c.point3d_path;
  if (!c.serial_numbers.empty()) serial_numbers_ = c.serial_numbers;
  fix_base_marker_ = c.fix_base_marker;
  rotation_as_rvec_ = c.rotation_as_rvec;
  device_ = c.device;
  loss_function_ = c.loss_function; loss_scale_ = c.loss_scale;
  bal_problem.set_marker_side(c.marker_side);
  Load();
}

// Replaces bundle_adjustment_manager.cpp:16-96.  The per-observation functor dispatch on
// (camera_idx == 0, marker_idx == 0) is done inside ba_cuda_set_model_b (fix_cam0 = 1, fix_marker0 = Main/Test2);
// intrinsics are looked up by SERIAL_NUMBERS[camera_idx] exactly as manager.cpp:34,47,64,78 do; the solver
// options are Ceres' defaults with DENSE_SCHUR and progress to stdout (manager.cpp:90-92).
std::vector<double> BAManager::Intrinsics4() const {
  const int C = bal_problem.num_cameras();
  if ((int)serial_numbers_.size() < C) Die("BAManager: fewer serial numbers than cameras");
  std::vector<double> intr(4 * (size_t)C);
  for (int c = 0; c < C; ++c) {
    auto it = camera_intrinsics_map.find(serial_numbers_[c]);
    if (it == camera_intrinsics_map.end() || it->second.empty()) Die("BAManager: no intrinsics for camera " + serial_numbers_[c]);
    const cv::Mat& K = it->second;
    intr[4 * c + 0] = K.at<double>(0, 0); intr[4 * c + 1] = K.at<double>(1, 1);   // fx, fy   (bundle_adjustment.h:66-67)
    intr[4 * c + 2] = K.at<double>(0, 2); intr[4 * c + 3] = K.at<double>(1, 2);   // ppx, ppy (bundle_adjustment.h:68-69)
  }
  return intr;
}

void BAManager::StartBA() {
  const int C = bal_problem.num_cameras();
  const std::vector<double> intr = Intrinsics4();
  ba_cuda_problem* p = nullptr;
  auto check = [&](int rc, const char* what) {
    if (rc != BA_OK) { std::string m = std::string(what) + ": " + ba_cuda_last_error(); ba_cuda_destroy(p); Die(m); }
  };
  check(ba_cuda_create(&p, device_), "ba_cuda_create");
  check(ba_cuda_set_model_b(p, C, bal_problem.num_times(), bal_problem.num_markers(), bal_problem.num_observations(),
                            bal_problem.time_index(), bal_problem.camera_index(), bal_problem.marker_index(), bal_problem.observations(),
                            intr.data(), bal_problem.marker_side(), 1, fix_base_marker_ ? 1 : 0), "ba_cuda_set_model_b");
  check(ba_cuda_set_parameters(p, bal_problem.parameters(), bal_problem.num_parameters()), "ba_cuda_set_parameters");
  ba_cuda_options options;
  ba_cuda_options_init(&options);
  options.rcs_solver = BA_RCS_DENSE_CHOLESKY;      // options.linear_solver_type = DENSE_SCHUR
  options.minimizer_progress_to_stdout = 1;        // options.minimizer_progress_to_stdout = true
  options.loss_function = loss_function_; options.loss_scale = loss_scale_;   // NULL loss unless configured otherwise
  check(ba_cuda_solve(p, &options, &summary_), "ba_cuda_solve");
  // Ceres optimises the caller's parameter blocks in place; here the result is copied back into parameters_
  check(ba_cuda_get_parameters(p, bal_problem.mutable_parameters(), bal_problem.num_parameters()), "ba_cuda_get_parameters");
  const int n = ba_cuda_get_iterations(p, nullptr, 0);
  iterations_.resize(n > 0 ? n : 0);
  if (n > 0) ba_cuda_get_iterations(p, iterations_.data(), n);
  ba_cuda_destroy(p);
  // summary.FullReport() (manager.cpp:95), the fields this path produces
  static const char* kTerm[] = {"CONVERGENCE", "NO_CONVERGENCE", "FAILURE"};
  static const char* kWhy[] = {"", "Gradient tolerance reached.", "Parameter tolerance reached.", "Function tolerance reached.",
                               "Minimum trust region radius reached.", "Maximum number of iterations reached.",
                               "Number of consecutive invalid steps more than max_num_consecutive_invalid_steps.",
                               "Initial residual and Jacobian evaluation failed."};
  cout << "\nSolver Summary (B200 ba_cuda)\n\n"
       << "Parameters          " << summary_.num_free_parameters << "\nResiduals           " << summary_.num_residuals
       << "\nLinear solver       DENSE_SCHUR (reduced system " << summary_.rcs_dim << " x " << summary_.rcs_dim << ")\n\nCost:\nInitial   "
       << summary_.initial_cost << "\nFinal     " << summary_.final_cost << "\nChange    " << summary_.initial_cost - summary_.final_cost
       << "\n\nMinimizer iterations  " << summary_.num_iterations << "\nSuccessful steps      " << summary_.num_successful_steps
       << "\nUnsuccessful steps    " << summary_.num_unsuccessful_steps << "\n\nTime (s): total " << summary_.total_time_s
       << "\nTermination: " << kTerm[summary_.termination_type] << " (" << kWhy[summary_.termination_reason] << ")\n" << endl;
}

int BAManager::Covariance(std::vector<double>* camera_cov, std::vector<double>* frame_cov) {
  const int C = bal_problem.num_cameras(), M = bal_problem.num_markers();
  const std::vector<double> intr = Intrinsics4();
  const size_t nk = 6 * ((size_t)C + M);
  std::vector<double> kept(nk * nk), frames(36 * (size_t)bal_problem.num_times());
  ba_cuda_options options;
  ba_cuda_options_init(&options);
  options.loss_function = loss_function_; options.loss_scale = loss_scale_;   // the loss StartBA() solved with
  ba_cuda_problem* p = nullptr;
  int rc = ba_cuda_create(&p, device_);
  if (rc == BA_OK)
    rc = ba_cuda_set_model_b(p, C, bal_problem.num_times(), M, bal_problem.num_observations(), bal_problem.time_index(),
                             bal_problem.camera_index(), bal_problem.marker_index(), bal_problem.observations(), intr.data(),
                             bal_problem.marker_side(), 1, fix_base_marker_ ? 1 : 0);
  if (rc == BA_OK) rc = ba_cuda_set_parameters(p, bal_problem.parameters(), bal_problem.num_parameters());
  if (rc == BA_OK) rc = ba_cuda_covariance(p, &options, 0.0, kept.data(), frames.data(), nullptr);
  ba_cuda_destroy(p);
  if (rc != BA_OK) return rc;
  if (camera_cov) {   // GetCovarianceBlock(camera_c, camera_c)
    camera_cov->assign(36 * (size_t)C, 0.0);
    for (int c = 0; c < C; ++c)
      for (int a = 0; a < 6; ++a)
        for (int b = 0; b < 6; ++b) (*camera_cov)[36 * (size_t)c + 6 * a + b] = kept[(6 * (size_t)c + a) * nk + 6 * c + b];
  }
  if (frame_cov) frame_cov->swap(frames);
  return BA_OK;
}

// bundle_adjustment_manager.cpp:98-175: Camera_Transform.xml (R<i> 3x3, t<i> 3x1, 17 digits), the inverse pose
// files Extrinsics/mat<i>.txt and point3d.txt (default ofstream precision).  Rodrigues, [R^T | -R^T t] and the
// composed corner points come from the GPU (ba_cuda_model_b_outputs).
void BAManager::Write() {
  const int C = bal_problem.num_cameras();
  cout << "Marker Transform" << endl;
  for (int marker_idx = 0; marker_idx < bal_problem.num_markers(); marker_idx++) {
    double* m = bal_problem.marker_transform(marker_idx);
    cout << marker_idx << " Rvec: " << m[0] << " " << m[1] << " " << m[2] << " tvec: " << m[3] << " " << m[4] << " " << m[5] << endl;
  }
  std::vector<double> rot(9 * (size_t)C), inv(12 * (size_t)C), corners(12 * (size_t)bal_problem.num_observations()), intr(4 * (size_t)C, 1.0);
  ba_cuda_problem* p = nullptr;
  bool ok = ba_cuda_create(&p, device_) == BA_OK &&
            ba_cuda_set_model_b(p, C, bal_problem.num_times(), bal_problem.num_markers(), bal_problem.num_observations(),
                                bal_problem.time_index(), bal_problem.camera_index(), bal_problem.marker_index(), bal_problem.observations(),
                                intr.data(), bal_problem.marker_side(), 1, fix_base_marker_ ? 1 : 0) == BA_OK &&
            ba_cuda_set_parameters(p, bal_problem.parameters(), bal_problem.num_parameters()) == BA_OK &&
            ba_cuda_model_b_outputs(p, rot.data(), inv.data(), corners.data()) == BA_OK;
  if (!ok) { std::string m = std::string("BAManager::Write: ") + ba_cuda_last_error(); ba_cuda_destroy(p); Die(m); }
  ba_cuda_destroy(p);

  storage::XmlWriter fs(transform_xml_path_);
  if (!fs.isOpened()) Die("unable to open Camera_Transform.xml");
  for (int i = 0; i < C; i++) {
    double* cam = bal_problem.camera_parameters(i);
    cv::Mat camera_rot(3, 3, &rot[9 * (size_t)i]), camera_tvec(3, 1, cam + 3), camera_rvec(3, 1, cam);
    fs.Write("R" + std::to_string(i), rotation_as_rvec_ ? camera_rvec : camera_rot);
    fs.Write("t" + std::to_string(i), camera_tvec);
    std::ofstream f_hongo(extrinsics_dir_ + "/mat" + std::to_string(i) + ".txt");
    for (int row = 0; row < 3; row++)
      for (int col = 0; col < 4; col++) f_hongo << inv[12 * (size_t)i + 4 * row + col] << endl;
  }
  fs.release();

  std::ofstream fout(point3d_path_);
  const size_t n_points = corners.size() / 3;
  fout << n_points << " " << bal_problem.num_times() << " " << bal_problem.num_cameras() << endl;
  for (int time_idx = 0; time_idx < bal_problem.num_times(); time_idx++) {
    fout << time_idx;
    for (int camera_idx = 0; camera_idx < C; camera_idx++) fout << " " << bal_problem.num_observations_per_time_camera(time_idx, camera_idx);
    fout << endl;
  }
  for (size_t i = 0; i < n_points; i++) fout << corners[3 * i] << " " << corners[3 * i + 1] << " " << corners[3 * i + 2] << endl;
}

}  // namespace RSCalibration
