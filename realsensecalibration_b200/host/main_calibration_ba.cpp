// main_calibration_ba.cpp -- the bundle-adjustment stage of Main_Calibration's main() (main.cpp:35-43) on the
// files the earlier stages leave behind, driven through the source-compatible host classes:
//   BAManager(intrinsics, dist) -> StartBA() -> Write() -> ReprojectionCheck::Reproject(...)
// usage: ba_main_calibration <Common dir> <output dir> [test1 | test2 | covariance]
// covariance: the hongo run, followed by one line per camera with the standard deviations of its pose parameters
// (rvec, tvec; per unit of pixel noise) from ceres::Covariance's counterpart (BAManager::Covariance).
// Everything before it in the reference's main() (image capture, ArUco detection, solvePnP) is out of scope; the
// detected corners Reproject needs are the observations stored in correspondence.txt.
#include <cmath>
#include <cstdio>
#include <iostream>

#include "bundle_adjustment_manager.h"
#include "cv_storage.h"
#include "reprojection_check.h"
#include "test1_bundle_adjustmenter.h"

using namespace RSCalibration;

static bool GetIntrinsics(const std::string& common, const std::vector<std::string>& serials, std::map<std::string, cv::Mat>& K,
                          std::map<std::string, cv::Mat>& dist) {  // IO::GetIntrinsics, my_io.cpp:5-31
  for (const std::string& sn : serials) {
    std::map<std::string, cv::Mat> m;
    if (!storage::ReadXml(common + "/Calibration/Intrinsics/" + sn + ".xml", m)) { std::cerr << "unable to open intrinsics file." << std::endl; return false; }
    K[sn] = m["intrinsics"];
    dist[sn] = m["distCoeffs"];
  }
  return true;
}

int main(int argc, char** argv) {
  if (argc < 3) { std::fprintf(stderr, "usage: %s <Common dir> <output dir> [test1]\n", argv[0]); return 2; }
  const std::string common = argv[1], out = argv[2];
  if (argc > 3 && std::string(argv[3]) == "test1") {  // Test1_BundleAdjustment/main.cpp:56-87
    std::map<std::string, cv::Mat> K, dist;
    if (!GetIntrinsics(common, {"825312072048"}, K, dist)) return 1;
    RSCalibrationTest1::BALProblem pb;
    if (!pb.LoadFile((common + "/Correspondence/two_cam_data.txt").c_str())) { std::cerr << "ERROR: unable to open file \n"; return 1; }
    ba_cuda_summary s;
    if (SolveTest1(pb, K["825312072048"], &s) != BA_OK) { std::cerr << ba_cuda_last_error() << std::endl; return 1; }
    std::printf("test1: iterations %d initial %.12e final %.12e camera %.17g %.17g %.17g %.17g %.17g %.17g\n", s.num_iterations, s.initial_cost,
                s.final_cost, pb.mutable_cameras()[0], pb.mutable_cameras()[1], pb.mutable_cameras()[2], pb.mutable_cameras()[3],
                pb.mutable_cameras()[4], pb.mutable_cameras()[5]);
    return 0;
  }
  // test2: Test2_BundleAdjustment/main.cpp:53-152 on its fixture -- two cameras, marker 0 free (two-functor dispatch), R<i>
  // written as the rotation vector, and the check reading that file back (the configuration the committed outputs were made
  // with: 48 mm markers, cameras 819612072493 / 825312072048, SURVEY.md 8c)
  const bool test2 = argc > 3 && std::string(argv[3]) == "test2";
  const std::vector<std::string> serials = test2 ? std::vector<std::string>{"819612072493", "825312072048"}
                                                 : std::vector<std::string>(SERIAL_NUMBERS, SERIAL_NUMBERS + CAMERAS);
  std::map<std::string, cv::Mat> camera_intrinsics_map, dist_coeffs_map;
  if (!GetIntrinsics(common, serials, camera_intrinsics_map, dist_coeffs_map)) return 1;
  BAManager::Config cfg;
  cfg.correspondence_path = common + (test2 ? "/Correspondence/test2/correspondence_test.txt" : "/Correspondence/hongo/correspondence.txt");
  if (test2) { cfg.serial_numbers = serials; cfg.marker_side = 0.048; cfg.fix_base_marker = false; cfg.rotation_as_rvec = true; }
  cfg.transform_xml_path = out + "/Camera_Transform.xml";
  cfg.extrinsics_dir = out;
  cfg.point3d_path = out + "/point3d.txt";
  BAManager ba_manager(camera_intrinsics_map, dist_coeffs_map, cfg);
  ba_manager.StartBA();
  ba_manager.Write();
  // detected corners per (time, camera) in file order == what Correspondencer hands to Reproject (main.cpp:43)
  BALProblem& pb = ba_manager.problem();
  std::vector<std::vector<std::vector<cv::Point2f>>> image_points_per_time(pb.num_times(), std::vector<std::vector<cv::Point2f>>(pb.num_cameras()));
  for (int i = 0; i < pb.num_observations(); i++)
    for (int j = 0; j < 4; j++)
      image_points_per_time[pb.time_index()[i]][pb.camera_idx(i)].emplace_back(
          cv::Point2f((float)pb.observations()[8 * i + 2 * j], (float)pb.observations()[8 * i + 2 * j + 1]));
  const ReprojectionCheck::Result r =
      ReprojectionCheck::Reproject(cfg.point3d_path, cfg.transform_xml_path, serials, image_points_per_time, camera_intrinsics_map);
  if (!r.ok) return 1;
  std::cout << "Reprojection Error (After BA): " << r.reprojection_error << std::endl;
  std::cout << "Average Reprojection Error per One Coordinate: " << r.rms_per_coordinate << std::endl;
  std::printf("summary: iterations %d initial %.15e final %.15e reprojection %.12e rms %.8f\n", ba_manager.summary().num_iterations,
              ba_manager.summary().initial_cost, ba_manager.summary().final_cost, r.reprojection_error, r.rms_per_coordinate);
  if (argc > 3 && std::string(argv[3]) == "covariance") {
    std::vector<double> cam;
    if (ba_manager.Covariance(&cam, nullptr) != BA_OK) { std::cerr << ba_cuda_last_error() << std::endl; return 1; }
    for (int c = 0; c < pb.num_cameras(); ++c) {
      std::printf("covariance: camera %d sd", c);
      for (int k = 0; k < 6; ++k) std::printf(" %.6e", std::sqrt(cam[36 * (size_t)c + 7 * k]));
      std::printf("\n");
    }
  }
  return 0;
}
