// System.cc -- see System.h.  Mirrors src/System.cc:25-244 (construction, TrackRGBD, SaveResults) over the C ABI.
#include "System.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <sstream>

#include "vdo_b200.h"

namespace VDO_SLAM {
namespace {
// "Key: value  # comment" lines of an OpenCV FileStorage YAML (the only form the reference's settings files use)
map<string, double> read_settings(const string &path, bool &ok) {
  map<string, double> kv;
  ifstream f(path.c_str());
  ok = f.is_open();
  string line;
  while (ok && getline(f, line)) {
    const size_t h = line.find('#');
    if (h != string::npos) line.erase(h);
    const size_t c = line.find(':');
    if (c == string::npos || line.compare(0, 5, "%YAML") == 0) continue;
    string key = line.substr(0, c), val = line.substr(c + 1);
    key.erase(0, key.find_first_not_of(" \t")); key.erase(key.find_last_not_of(" \t") + 1);
    char *end = nullptr;
    const double v = strtod(val.c_str(), &end);
    if (end != val.c_str()) kv[key] = v;
  }
  return kv;
}
double get(const map<string, double> &kv, const char *k, double dflt = 0.0) {
  map<string, double>::const_iterator it = kv.find(k);
  return it == kv.end() ? dflt : it->second;      // cv::FileNode of a missing key converts to 0 as well
}

// ---- the float 4x4 algebra of the reference's cv::Mat expressions (same two OpenCV gemm branches as csrc/results_io.cpp) ----
typedef System::Mat16 M4;
M4 eye4() { M4 m{}; m.v[0] = m.v[5] = m.v[10] = m.v[15] = 1.f; return m; }
M4 mul4(const M4 &A, const M4 &B) {            // 4x4 * 4x4: gemm's small-matrix branch, float accumulation left to right
  M4 C{};
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      float s = A.v[4 * i] * B.v[j];
      s = s + A.v[4 * i + 1] * B.v[4 + j];
      s = s + A.v[4 * i + 2] * B.v[8 + j];
      s = s + A.v[4 * i + 3] * B.v[12 + j];
      C.v[4 * i + j] = s;
    }
  return C;
}
M4 inv4(const M4 &T) {                          // Converter::toInvMatrix (src/Converter.cc:151-166): -R.t()*t in double, one rounding
  M4 I = eye4();
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) I.v[4 * i + j] = T.v[4 * j + i];
    double s = 0;
    for (int k = 0; k < 3; ++k) s += (double)T.v[4 * k + i] * (double)T.v[4 * k + 3];
    I.v[4 * i + 3] = (float)(-s);
  }
  return I;
}
M4 from_mat(const cv::Mat &m) {
  M4 o = eye4();
  if (m.empty() || m.rows < 3 || m.cols < 4 || m.type() != CV_32F) return o;
  for (int i = 0; i < m.rows && i < 4; ++i) for (int j = 0; j < 4; ++j) o.v[4 * i + j] = m.at<float>(i, j);
  return o;
}
// Tracking::ObjPoseParsingKT (src/Tracking.cc:2010-2080): KITTI ground-truth row -> object pose in the camera frame (R = Ry*Rx*Rz, x = z = 0)
M4 obj_pose_kt(const vector<float> &g) {
  M4 P = eye4();
  if (g.size() < 10) return P;
  const float y = g[9] + (3.1415926 / 2), x = 0.0, z = 0.0;
  const float cy = cos(y), sy = sin(y), cx = cos(x), sx = sin(x), cz = cos(z), sz = sin(z);
  P.v[0] = cy * cz + sy * sx * sz; P.v[1] = -cy * sz + sy * sx * cz; P.v[2] = sy * cx;
  P.v[4] = cx * sz; P.v[5] = cx * cz; P.v[6] = -sx;
  P.v[8] = -sy * cz + cy * sx * sz; P.v[9] = sy * sz + cy * sx * cz; P.v[10] = cy * cx;
  P.v[3] = g[6]; P.v[7] = g[7]; P.v[11] = g[8];
  return P;
}
// Tracking::ObjPoseParsingOX (src/Tracking.cc:2082-2130): OMD row -> pose in the world frame from a quaternion (x, y, z, w at columns 5..8)
M4 obj_pose_ox(const vector<float> &g) {
  M4 P = eye4();
  if (g.size() < 9) return P;
  const float qx = g[5], qy = g[6], qz = g[7], qw = g[8];
  P.v[0] = 1 - 2 * qz * qz - 2 * qy * qy; P.v[1] = -2 * qz * qw + 2 * qy * qx; P.v[2] = 2 * qy * qw + 2 * qz * qx;
  P.v[4] = 2 * qx * qy + 2 * qw * qz; P.v[5] = 1 - 2 * qz * qz - 2 * qx * qx; P.v[6] = 2 * qz * qy - 2 * qx * qw;
  P.v[8] = 2 * qx * qz - 2 * qw * qy; P.v[9] = 2 * qy * qz + 2 * qw * qx; P.v[10] = 1 - 2 * qy * qy - 2 * qx * qx;
  P.v[3] = g[2]; P.v[7] = g[3]; P.v[11] = g[4];
  return P;
}
template <typename T> vector<T> tracker_get(vdo_tracker *t, const char *name) {
  int n = 0;
  vector<T> out;
  if (vdo_tracker_get(t, name, nullptr, 0, &n) != VDO_OK || n <= 0) return out;
  out.resize(n);
  vdo_tracker_get(t, name, out.data(), n, &n);
  return out;
}
template <typename T> vector<T> map_get(vdo_tracker *t, const char *name) {
  int n = 0;
  vector<T> out;
  if (vdo_tracker_map_get(t, name, nullptr, 0, &n) != VDO_OK || n <= 0) return out;
  out.resize(n);
  vdo_tracker_map_get(t, name, out.data(), n, &n);
  return out;
}
}  // namespace

System::System(const string &strSettingsFile, const eSensor sensor) : mSensor(sensor), mpCtx(nullptr), mpTracker(nullptr), mbRGB(true), mbKitti(true), mnDataset(2) {
  bool ok = false;
  const map<string, double> kv = read_settings(strSettingsFile, ok);
  if (!ok) {
    cerr << "Failed to open settings file at: " << strSettingsFile << endl;
    exit(-1);
  }
  mpParams = new vdo_tracker_params;
  vdo_tracker_params &p = *mpParams;
  vdo_tracker_params_default(&p);
  p.fx = (float)get(kv, "Camera.fx"); p.fy = (float)get(kv, "Camera.fy"); p.cx = (float)get(kv, "Camera.cx"); p.cy = (float)get(kv, "Camera.cy");
  // Camera.width / Camera.height are NOT read by the reference (the size comes from the images): the tracker is created from the first frame
  p.width = p.height = 0;
  p.bf = (float)get(kv, "Camera.bf"); p.depth_factor = (float)get(kv, "DepthMapFactor");
  p.th_depth_bg = (float)get(kv, "ThDepthBG"); p.th_depth_obj = (float)get(kv, "ThDepthOBJ");
  p.max_track_bg = (int)get(kv, "MaxTrackPointBG"); p.max_track_obj = (int)get(kv, "MaxTrackPointOBJ");
  p.sf_mg_thres = (float)get(kv, "SFMgThres"); p.sf_ds_thres = (float)get(kv, "SFDsThres");
  p.n_features = (int)get(kv, "ORBextractor.nFeatures"); p.scale_factor = (float)get(kv, "ORBextractor.scaleFactor");
  p.n_levels = (int)get(kv, "ORBextractor.nLevels"); p.ini_th_fast = (int)get(kv, "ORBextractor.iniThFAST"); p.min_th_fast = (int)get(kv, "ORBextractor.minThFAST");
  mnDataset = (int)get(kv, "ChooseData");              // src/Tracking.cc:114-130: 1 OMD, 2 KITTI, 3 VirtualKITTI
  if (mnDataset < 1 || mnDataset > 3) {
    cerr << "ChooseData must be 1 (OMD), 2 (KITTI) or 3 (VirtualKITTI); got " << mnDataset << endl;
    exit(-1);
  }
  p.dataset = mnDataset;
  p.is_kitti = (mnDataset == 2) ? 1 : 0;
  p.window_size = (int)get(kv, "WINDOW_SIZE"); p.overlap_size = (int)get(kv, "OVERLAP_SIZE");
  mbRGB = (int)get(kv, "Camera.RGB") != 0;
  mbKitti = p.is_kitti != 0;
  const int useSample = (int)get(kv, "UseSampleFeature");
  if (useSample != 0 && useSample != 1) {
    cerr << "UseSampleFeature must be 0 (detected features) or 1 (sampled features); got " << useSample << endl;
    exit(-1);
  }
  p.use_sample_feature = useSample;
  // SampleSeed is not a key of the reference: missing or 0 seeds every frame's sampler with time(NULL) like src/Frame.cc:674; any other value
  // fixes the seed so that a run can be repeated (the tracker reports the seeds it used through vdo_tracker_get("sample_seed"))
  const double seed = get(kv, "SampleSeed");
  if (!(seed >= 0.0 && seed <= 4294967295.0) || seed != floor(seed)) {
    cerr << "SampleSeed must be an integer in [0, 4294967295]; got " << seed << endl;
    exit(-1);
  }
  p.sample_seed = (unsigned)seed;
  if (vdo_ctx_create(0, &mpCtx) != VDO_OK) {
    cerr << "vdo_b200: no usable CUDA device (there is no CPU fallback)" << endl;
    exit(-1);
  }
}

System::~System() {
  if (mpTracker) vdo_tracker_destroy(mpTracker);
  vdo_ctx_destroy(mpCtx);
  delete mpParams;
}

cv::Mat System::TrackRGBD(const cv::Mat &im, cv::Mat &depthmap, const cv::Mat &flowmap, const cv::Mat &masksem, const cv::Mat &mTcw_gt,
                          const vector<vector<float> > &vObjPose_gt, const double &, cv::Mat &, const int &nImage) {
  if (mSensor != RGBD) {
    cerr << "ERROR: you called TrackRGBD but input sensor was not set to RGBD." << endl;
    exit(-1);
  }
  const int rows = im.rows, cols = im.cols;
  if (rows <= 0 || cols <= 0 || !depthmap.isContinuous() || !flowmap.isContinuous() || !masksem.isContinuous() || depthmap.type() != CV_32F ||
      flowmap.type() != CV_32FC2 || masksem.type() != CV_32SC1 || depthmap.rows != rows || depthmap.cols != cols || flowmap.rows != rows || flowmap.cols != cols ||
      masksem.rows != rows || masksem.cols != cols) {
    cerr << "ERROR: TrackRGBD expects continuous CV_32F depth, CV_32FC2 flow and CV_32SC1 mask, all of the image size (" << cols << "x" << rows << ")." << endl;
    exit(-1);
  }
  if (!mpTracker) {                                    // the reference takes the frame size from the first image
    mpParams->width = cols; mpParams->height = rows;
    if (vdo_tracker_create(mpCtx, mpParams, &mpTracker) != VDO_OK) {
      cerr << "vdo_b200: tracker creation failed: " << vdo_last_error(mpCtx) << endl;
      exit(-1);
    }
  } else if (cols != mpParams->width || rows != mpParams->height) {
    cerr << "ERROR: TrackRGBD frame size changed from " << mpParams->width << "x" << mpParams->height << " to " << cols << "x" << rows << "." << endl;
    exit(-1);
  }
  // cvtColor(RGB/BGR(A) -> GRAY) of src/Tracking.cc:209-222 in OpenCV's 8-bit fixed point: (R*4899 + G*9617 + B*1868 + 2^13) >> 14
  mGray.resize((size_t)rows * cols);
  const int ch = im.channels();
  for (int r = 0; r < rows; ++r) {
    const unsigned char *src = im.data + (size_t)r * im.step;
    unsigned char *dst = &mGray[(size_t)r * cols];
    if (ch == 1) memcpy(dst, src, cols);
    else
      for (int c = 0; c < cols; ++c) {
        const unsigned char *px = src + (size_t)c * ch;
        const int R = mbRGB ? px[0] : px[2], G = px[1], B = mbRGB ? px[2] : px[0];
        dst[c] = (unsigned char)((R * 4899 + G * 9617 + B * 1868 + (1 << 13)) >> 14);
      }
  }
  vector<int> gt(vObjPose_gt.size());
  for (size_t i = 0; i < vObjPose_gt.size(); ++i) gt[i] = vObjPose_gt[i].size() > 1 ? (int)vObjPose_gt[i][1] : -1;
  cv::Mat Tcw = cv::Mat::eye(4, 4, CV_32F);
  float T[16];
  // the mask is declared const in the reference's signature yet mutated through the shared cv::Mat buffer (mSegMap = maskSEM); same here
  const int rc = vdo_tracker_track(mpTracker, cols, rows, mGray.data(), (float *)depthmap.data, (const float *)flowmap.data, (int *)masksem.data, (int)gt.size(),
                                   gt.empty() ? nullptr : gt.data(), 1, T);
  if (rc != VDO_OK) {
    cerr << "vdo_b200: TrackRGBD failed (" << rc << "): " << vdo_tracker_last_error(mpTracker) << endl;
    exit(-1);
  }
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) Tcw.at<float>(i, j) = T[4 * i + j];
  UpdateGroundTruthMap(mTcw_gt, vObjPose_gt);
  // StopFrame = nImage - 1: whole-sequence optimisation after the last frame (src/Tracking.cc:168, 1162-1176, 1198; KITTI only)
  if ((int)mvCamPoseGT.size() == nImage && mbKitti && nImage > 2) {
    vdo_lm_stats st;
    if (vdo_tracker_batch_optimize(mpTracker, 1, nullptr, &st, nullptr) != VDO_OK)
      cerr << "vdo_b200: FullBatchOptimization failed: " << vdo_tracker_last_error(mpTracker) << endl;
  }
  return Tcw;
}

// The ground-truth side of the map the reference keeps for its result files (src/Tracking.cc:318-341 pose chain and object-pose parsing,
// :784-850 per-object ground-truth motion, :1113-1131 pushes): vmCameraPose_GT, vmObjPosePre, vmRigidMotion_GT, aligned entry by entry
// with the tracker's vmRigidMotion (entry 0 = camera, then the objects with bObjStat == true in nModLabel order).
void System::UpdateGroundTruthMap(const cv::Mat &mTcw_gt, const vector<vector<float> > &vObjPose_gt) {
  const M4 in = from_mat(mTcw_gt);
  const bool first = mvCamPoseGT.empty();
  M4 cur_Tcw_gt;
  if (first) { cur_Tcw_gt = inv4(in); mOriginInv = in; }
  else cur_Tcw_gt = mul4(inv4(in), mOriginInv);
  vector<int> sem(vObjPose_gt.size());
  vector<M4> pose(vObjPose_gt.size());
  for (size_t i = 0; i < vObjPose_gt.size(); ++i) {
    sem[i] = vObjPose_gt[i].size() > 1 ? (int)vObjPose_gt[i][1] : -1;
    pose[i] = (mnDataset == 1) ? obj_pose_ox(vObjPose_gt[i]) : obj_pose_kt(vObjPose_gt[i]);
  }
  if (first) {
    mvCamPoseGT.push_back(eye4());                                      // :1250
  } else {
    mvCamPoseGT.push_back(inv4(cur_Tcw_gt));                           // :1114-1115
    const vector<int> semPos = tracker_get<int>(mpTracker, "nSemPosition"), stat = tracker_get<int>(mpTracker, "bObjStat");
    const vector<float> vel = tracker_get<float>(mpTracker, "mVelocity");
    M4 velocity = eye4();
    if (vel.size() == 16) memcpy(velocity.v, vel.data(), 64);
    vector<M4> posePre(1, inv4(velocity)), motGT(1, mul4(mLastTcwGT, inv4(cur_Tcw_gt)));     // :1083-1086, :1120-1121
    const M4 lastTwc = inv4(mLastTcwGT), curTwc = inv4(cur_Tcw_gt);
    for (size_t i = 0; i < semPos.size() && i < stat.size(); ++i) {
      if (!stat[i]) continue;
      M4 Lwp = eye4(), Lwc = eye4();
      for (size_t k = 0; k < mLastSemGT.size(); ++k) if (mLastSemGT[k] == semPos[i]) { Lwp = (mnDataset == 1) ? mLastPoseGT[k] : mul4(lastTwc, mLastPoseGT[k]); break; }
      for (size_t k = 0; k < sem.size(); ++k) if (sem[k] == semPos[i]) { Lwc = (mnDataset == 1) ? pose[k] : mul4(curTwc, pose[k]); break; }
      posePre.push_back(Lwp);                                          // vObjPosePre = L_w_p (:850)
      motGT.push_back(mul4(inv4(Lwp), Lwc));                           // vObjMod_gt = L_w_p^-1 * L_w_c (:847-848)
    }
    mvObjPosePre.push_back(posePre); mvRigidMotionGT.push_back(motGT);
  }
  mLastTcwGT = cur_Tcw_gt; mLastSemGT = sem; mLastPoseGT = pose;
}

void System::SaveResults(const string &filename) {
  cout << endl << "Saving Results into TXT File..." << endl;
  if (!mpTracker) { cerr << "vdo_b200: SaveResults before the first frame" << endl; return; }
  // `filename` is a directory prefix: the reference appends the seven file names to it (src/System.cc:74-77, 128, 148, 166)
  const vector<int> per = map_get<int>(mpTracker, "n_per_frame"), labels = map_get<int>(mpTracker, "vnRMLabel");
  const vector<float> mot = map_get<float>(mpTracker, "vmRigidMotion"), mot_rf = map_get<float>(mpTracker, "vmRigidMotion_RF"), cen = map_get<float>(mpTracker, "vmRigidCentre");
  const vector<float> cam = map_get<float>(mpTracker, "vmCameraPose"), cam_rf = map_get<float>(mpTracker, "vmCameraPose_RF");
  vector<float> pre, gtm, camgt;
  size_t entries = 0;
  for (size_t i = 0; i < per.size(); ++i) entries += (size_t)per[i];
  for (size_t i = 0; i < per.size() && i < mvObjPosePre.size(); ++i)
    for (int j = 0; j < per[i]; ++j) {
      const M4 a = j < (int)mvObjPosePre[i].size() ? mvObjPosePre[i][j] : eye4(), b = j < (int)mvRigidMotionGT[i].size() ? mvRigidMotionGT[i][j] : eye4();
      pre.insert(pre.end(), a.v, a.v + 16); gtm.insert(gtm.end(), b.v, b.v + 16);
    }
  for (size_t i = 0; i < mvCamPoseGT.size(); ++i) camgt.insert(camgt.end(), mvCamPoseGT[i].v, mvCamPoseGT[i].v + 16);
  bool ok = pre.size() == 16 * entries && mot.size() == 16 * entries && mot_rf.size() == 16 * entries && cen.size() == 3 * entries && labels.size() == entries;
  if (!ok) cerr << "vdo_b200: SaveResults: the map and the ground-truth bookkeeping disagree on the number of entries" << endl;
  const int nf = (int)per.size();
  struct Out { const char *name; int rc; } outs[7] = {
      {"obj_mot_stereo_new.txt", ok ? vdo_results_write_object_motions((filename + "obj_mot_stereo_new.txt").c_str(), 0, nf, per.data(), labels.data(), mot.data(), pre.data()) : -1},
      {"obj_mot_stereo_rf_new.txt", ok ? vdo_results_write_object_motions((filename + "obj_mot_stereo_rf_new.txt").c_str(), 0, nf, per.data(), labels.data(), mot_rf.data(), pre.data()) : -1},
      {"obj_mot_gt.txt", ok ? vdo_results_write_object_motions((filename + "obj_mot_gt.txt").c_str(), 0, nf, per.data(), labels.data(), gtm.data(), nullptr) : -1},
      {"obj_centre.txt", ok ? vdo_results_write_object_centres((filename + "obj_centre.txt").c_str(), 0, nf, per.data(), labels.data(), cen.data()) : -1},
      {"initial_stereo_new.txt", vdo_results_write_poses((filename + "initial_stereo_new.txt").c_str(), 0, (int)cam.size() / 16, cam.data())},
      {"refined_stereo_new.txt", vdo_results_write_poses((filename + "refined_stereo_new.txt").c_str(), 0, (int)cam_rf.size() / 16, cam_rf.data())},
      {"cam_pose_gt_stereo.txt", vdo_results_write_poses((filename + "cam_pose_gt_stereo.txt").c_str(), 0, (int)camgt.size() / 16, camgt.data())}};
  for (int i = 0; i < 7; ++i)
    if (outs[i].rc != VDO_OK) cerr << "vdo_b200: SaveResults could not write " << filename << outs[i].name << " (" << outs[i].rc << ")" << endl;
  // time analysis (src/System.cc:196-237): mean wall-clock per tracking component and per windowed optimisation
  const vector<float> st = tracker_get<float>(mpTracker, "stage_ms");
  const vector<int> lba = tracker_get<int>(mpTracker, "local_ba");
  const double frames = mvCamPoseGT.empty() ? 1.0 : (double)mvCamPoseGT.size();
  cout << "Time of all components: " << endl;
  for (size_t j = 0; j < st.size(); ++j) cout << "(" << j << "): " << st[j] / frames << " ";
  cout << endl;
  if (lba.size() == 2 && st.size() == 9) cout << "Time of local bundle adjustment: " << (lba[0] ? st[8] / lba[0] : 0.0) << endl;
}

}  // namespace VDO_SLAM
