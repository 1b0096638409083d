// tracker.cpp -- host side of the per-frame path: the sequencing of Tracking::GrabImageRGBD + Tracking::Track
// (src/Tracking.cc:164-648, 650-1212) over the device stages of this library.  It owns two resident frames (current / last),
// the per-frame vectors the reference keeps in `Frame` (include/Frame.h:110-196) and the slice of `Map` (include/Map.h:34-84)
// the batch optimisers read.  Everything numerical happens in the stages it calls (depth prep, ORB front end, static filter,
// object sampling, mask propagation, initial model, joint flow/pose LM, scene flow, object classification, renewal); the code
// here is control flow, index bookkeeping and 4x4 float algebra with cv::Mat rounding (float gemm = double accumulation,
// one rounding).  Ground-truth error metrics, drawing and file output of the reference are not part of the hot path.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <ctime>
#include <string>
#include <vector>

#include "../../include/vdo_b200.h"

namespace {
using M4 = std::array<float, 16>;
M4 eye4() { M4 m{}; m[0] = m[5] = m[10] = m[15] = 1.f; return m; }
// cv::Mat A * B of two 4x4 CV_32F (e.g. `mCurrentFrame.mTcw * Converter::toInvMatrix(mLastFrame.mTcw)`, src/Tracking.cc:700-706):
// OpenCV's gemm takes its small-matrix branch (no flags, inner dimension <= 4) and evaluates a0*b0 + a1*b1 + a2*b2 + a3*b3 in
// FLOAT, left to right.  Pinned bit for bit against cv2.gemm (tests/test_results_io.py for the same formula in results_io.cpp;
// the oracle pipeline calls cv2.gemm itself, so the tracker parity tests pin this one).
M4 mul4(const M4& A, const M4& B) {
  M4 C{};
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      float s = A[4 * i] * B[j];
      s = s + A[4 * i + 1] * B[4 + j];
      s = s + A[4 * i + 2] * B[8 + j];
      s = s + A[4 * i + 3] * B[12 + j];
      C[4 * i + j] = s;
    }
  return C;
}
// Converter::toInvMatrix (src/Converter.cc:151-166): [R^T | -R^T t]
M4 inv4(const M4& T) {
  M4 I = eye4();
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) I[4 * i + j] = T[4 * j + i];
    double s = 0;
    for (int k = 0; k < 3; ++k) s += (double)T[4 * k + i] * (double)T[4 * k + 3];
    I[4 * i + 3] = (float)(-s);
  }
  return I;
}

struct FrameState {
  vdo_frame* img = nullptr;
  M4 Tcw = eye4();
  std::vector<float> keys;                                              // mvKeys (x, y)
  std::vector<float> statKeysTmp, corres, flowNext, statDepthTmp, stat3DTmp;   // mvStatKeysTmp, mvCorres, mvFlowNext, mvStatDepthTmp, mvStat3DPointTmp
  std::vector<float> statKeys, statDepth;                               // mvStatKeys, mvStatDepth
  std::vector<float> sampKeys;                                          // Option II: the constructor's filtered samples (RenewFrameInfo's top-up source)
  std::vector<int> staInlierID;                                         // nStaInlierID
  std::vector<float> objKeys, objCorres, objFlowNext, objDepth, obj3D;  // mvObjKeys, mvObjCorres, mvObjFlowNext, mvObjDepth, mvObj3DPoint
  std::vector<int> semObjLabel, objLabel, dynInlierID;                  // vSemObjLabel, vObjLabel, nDynInlierID
  std::vector<float> flow3d;                                            // vFlow_3d
  std::vector<int> nModLabel, nSemPosition, semPosiGt;                  // nModLabel, nSemPosition, nSemPosi_gt
  std::vector<unsigned char> bObjStat;
  std::vector<M4> vObjMod;
  std::vector<float> vObjCentre3D;                                      // 3 per object (src/Tracking.cc:856-866)
  std::vector<std::vector<int>> vnObjID, vnObjInlierID;
  void clear_dynamic() {
    keys.clear(); statKeysTmp.clear(); corres.clear(); flowNext.clear(); statDepthTmp.clear(); stat3DTmp.clear(); statKeys.clear(); statDepth.clear(); sampKeys.clear();
    staInlierID.clear(); objKeys.clear(); objCorres.clear(); objFlowNext.clear(); objDepth.clear(); obj3D.clear(); semObjLabel.clear(); objLabel.clear();
    dynInlierID.clear(); flow3d.clear(); nModLabel.clear(); nSemPosition.clear(); semPosiGt.clear(); bObjStat.clear(); vObjMod.clear(); vObjCentre3D.clear(); vnObjID.clear();
    vnObjInlierID.clear();
  }
};

struct MapSlice {        // what Tracking::Track pushes per frame (src/Tracking.cc:1016-1070)
  std::vector<std::vector<float>> featSta, depSta, p3dSta, featDyn, depDyn, p3dDyn;
  std::vector<std::vector<int>> assoSta, assoDyn, featLabel, rmLabel, smLabel;
  std::vector<M4> cameraPose, cameraPose_RF;              // vmCameraPose (updated by the windowed BA) / vmCameraPose_RF (by the full batch)
  std::vector<std::vector<M4>> rigidMotion, rigidMotion_RF;
  std::vector<std::vector<float>> rigidCentre;            // vmRigidCentre: 3 floats per entry (entry 0 = camera = 0)
};
}  // namespace

struct vdo_tracker {
  vdo_ctx* ctx = nullptr;
  vdo_tracker_params p{};
  FrameState fr[2];
  int cur = 0;                 // index of the current frame; last = 1 - cur
  bool first = true;
  int f_id = 0, max_id = 1;
  bool has_velocity = false;
  M4 velocity = eye4();
  std::vector<float> tmpObjKeys, tmpObjDepth, tmpObjFlowNext, tmpObjCorres; std::vector<int> tmpSemObjLabel;   // mvTmp*
  std::vector<int> temperalMatch, temperalMatchSubset;
  MapSlice map;
  std::string err;
  double stage_ms[9] = {0};
  int frames = 0, local_ba_runs = 0, local_ba_iters = 0;
  unsigned sample_seed = 0;    // seed of the last frame's sampled background keypoints (0: none drawn)
  // scratch
  std::vector<float> s_f[12]; std::vector<int> s_i[8]; std::vector<unsigned char> s_b[2]; std::vector<double> s_d[2];
};

namespace {
struct StageTimer {
  double* acc; std::chrono::steady_clock::time_point t0;
  explicit StageTimer(double* a) : acc(a), t0(std::chrono::steady_clock::now()) {}
  ~StageTimer() { *acc += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};
#define TK(call) do { int rc_ = (call); if (rc_ != VDO_OK) { t->err = std::string(#call) + " failed"; return rc_; } } while (0)

void get3d_camera(float u, float v, float z, const vdo_tracker_params& p, float* X) {      // Optimizer::Get3DinCamera (src/Optimizer.cc:2995-3013)
  const float invfx = 1.0f / p.fx, invfy = 1.0f / p.fy;
  X[0] = (u - p.cx) * z * invfx; X[1] = (v - p.cy) * z * invfy; X[2] = z;
}
// Frame::UnprojectStereoStat / UnprojectStereoObject (src/Frame.cc:484-555): world point of a last-frame key
void unproject_world(float u, float v, float z, const vdo_tracker_params& p, const M4& Tcw, float* X) {
  const float invfx = 1.0f / p.fx, invfy = 1.0f / p.fy;
  const float x = (u - p.cx) * z * invfx, y = (v - p.cy) * z * invfy;
  for (int r = 0; r < 3; ++r) {
    const double twl = (double)(float)(-((double)Tcw[r] * (double)Tcw[3] + (double)Tcw[4 + r] * (double)Tcw[7] + (double)Tcw[8 + r] * (double)Tcw[11]));
    X[r] = (float)((double)Tcw[r] * (double)x + (double)Tcw[4 + r] * (double)y + (double)Tcw[8 + r] * (double)z + twl);
  }
}

// Frame::Frame (src/Frame.cc:61-260): ORB keypoints, static candidates, semi-dense object samples
int build_frame(vdo_tracker* t, FrameState& F) {
  const vdo_tracker_params& p = t->p;
  const int max_kp = p.n_features * 2 + 4096;
  auto& x = t->s_f[0]; auto& y = t->s_f[1]; auto& resp = t->s_f[2]; auto& ang = t->s_f[3]; auto& oct = t->s_i[0]; auto& sz = t->s_i[1];
  x.resize(max_kp); y.resize(max_kp); resp.resize(max_kp); ang.resize(max_kp); oct.resize(max_kp); sz.resize(max_kp);
  int n = 0;
  TK(vdo_orb_extract(F.img, p.n_features, p.scale_factor, p.n_levels, p.ini_th_fast, p.min_th_fast, max_kp, x.data(), y.data(), oct.data(), resp.data(), ang.data(),
                     sz.data(), &n, nullptr));
  F.keys.resize(2 * (size_t)n);
  for (int i = 0; i < n; ++i) { F.keys[2 * i] = x[i]; F.keys[2 * i + 1] = y[i]; }
  if (n == 0) return VDO_OK;                                    // Frame.cc:83-84: nothing else is filled
  const bool sampled = p.use_sample_feature != 0;
  const int ns = sampled ? VDO_SAMPLE_KEYPOINTS : n;
  auto& keep = t->s_i[2]; auto& cx = t->s_f[4]; auto& cy = t->s_f[5]; auto& fu = t->s_f[6]; auto& fv = t->s_f[7]; auto& dp = t->s_f[8];
  keep.resize(ns); cx.resize(ns); cy.resize(ns); fu.resize(ns); fv.resize(ns); dp.resize(ns);
  int m = 0;
  if (sampled) {                                                // Option II (Frame.cc:130-194)
    const unsigned seed = p.sample_seed ? p.sample_seed : (unsigned)std::time(nullptr);   // cv::RNG rng((unsigned)time(NULL)), Frame.cc:674
    t->sample_seed = seed;
    x.resize(ns); y.resize(ns);                                 // the ORB keypoints are in F.keys already
    TK(vdo_frame_sample_static(F.img, seed, p.th_depth_bg, ns, x.data(), y.data(), cx.data(), cy.data(), fu.data(), fv.data(), dp.data(), &m, nullptr));
    for (int i = 0; i < m; ++i) keep[i] = i;
  } else {
    TK(vdo_frame_filter_static(F.img, n, x.data(), y.data(), p.th_depth_bg, keep.data(), cx.data(), cy.data(), fu.data(), fv.data(), dp.data(), &m));
  }
  F.statKeysTmp.resize(2 * (size_t)m); F.corres.resize(2 * (size_t)m); F.flowNext.resize(2 * (size_t)m); F.statDepthTmp.resize(m);
  for (int i = 0; i < m; ++i) {
    F.statKeysTmp[2 * i] = x[keep[i]]; F.statKeysTmp[2 * i + 1] = y[keep[i]];
    F.corres[2 * i] = cx[i]; F.corres[2 * i + 1] = cy[i]; F.flowNext[2 * i] = fu[i]; F.flowNext[2 * i + 1] = fv[i];
    F.statDepthTmp[i] = dp[i] > 0 ? dp[i] : -1.f;
  }
  if (sampled) F.sampKeys = F.statKeysTmp;                     // RenewFrameInfo overwrites mvStatKeysTmp but tops up from this list
  const int step = 4, cap = ((p.width + step - 1) / step) * ((p.height + step - 1) / step);
  auto& ox = t->s_i[3]; auto& oy = t->s_i[4]; auto& lab = t->s_i[5];
  auto& ocx = t->s_f[4]; auto& ocy = t->s_f[5]; auto& ofx = t->s_f[6]; auto& ofy = t->s_f[7]; auto& od = t->s_f[8];
  ox.resize(cap); oy.resize(cap); lab.resize(cap); ocx.resize(cap); ocy.resize(cap); ofx.resize(cap); ofy.resize(cap); od.resize(cap);
  int k = 0;
  TK(vdo_frame_sample_objects(F.img, p.th_depth_obj, step, cap, ox.data(), oy.data(), ocx.data(), ocy.data(), ofx.data(), ofy.data(), od.data(), lab.data(), &k));
  F.objKeys.resize(2 * (size_t)k); F.objCorres.resize(2 * (size_t)k); F.objFlowNext.resize(2 * (size_t)k); F.objDepth.resize(k); F.semObjLabel.resize(k);
  for (int i = 0; i < k; ++i) {
    F.objKeys[2 * i] = (float)ox[i]; F.objKeys[2 * i + 1] = (float)oy[i]; F.objCorres[2 * i] = ocx[i]; F.objCorres[2 * i + 1] = ocy[i];
    F.objFlowNext[2 * i] = ofx[i]; F.objFlowNext[2 * i + 1] = ofy[i]; F.objDepth[i] = od[i]; F.semObjLabel[i] = lab[i];
  }
  return VDO_OK;
}

// Optimizer::PoseOptimizationFlow2Cam / Flow2 host wrapper for a batch of problems that index the LAST frame's arrays
struct FlowJob { int mode; const std::vector<int>* idx; M4 T_init; };
int run_flow(vdo_tracker* t, const FrameState& L, bool objects, const std::vector<FlowJob>& jobs, std::vector<M4>& T_out, std::vector<double>& flow_out,
             std::vector<unsigned char>& inlier, std::vector<int>& offs, std::vector<double>& stats) {
  const int np = (int)jobs.size();
  offs.assign(np + 1, 0);
  for (int j = 0; j < np; ++j) offs[j + 1] = offs[j] + (int)jobs[j].idx->size();
  const int tot = offs[np];
  auto& pts = t->s_f[9]; auto& dep = t->s_f[10]; auto& flo = t->s_f[11];
  pts.resize(2 * (size_t)tot + 2); dep.resize((size_t)tot + 1); flo.resize(2 * (size_t)tot + 2);
  const std::vector<float>& K = objects ? L.objKeys : L.statKeys; const std::vector<float>& D = objects ? L.objDepth : L.statDepth;
  const std::vector<float>& F = objects ? L.objFlowNext : L.flowNext;
  std::vector<int> mode(np); std::vector<float> Kc(4 * (size_t)np), Tl(16 * (size_t)np), Ti(16 * (size_t)np), To(16 * (size_t)np);
  for (int j = 0; j < np; ++j) {
    mode[j] = jobs[j].mode;
    const float k4[4] = {t->p.fx, t->p.fy, t->p.cx, t->p.cy};
    std::memcpy(&Kc[4 * j], k4, 16); std::memcpy(&Tl[16 * j], L.Tcw.data(), 64); std::memcpy(&Ti[16 * j], jobs[j].T_init.data(), 64);
    int q = offs[j];
    for (int id : *jobs[j].idx) { pts[2 * q] = K[2 * id]; pts[2 * q + 1] = K[2 * id + 1]; dep[q] = D[id]; flo[2 * q] = F[2 * id]; flo[2 * q + 1] = F[2 * id + 1]; ++q; }
  }
  flow_out.assign(2 * (size_t)tot + 2, 0.0); inlier.assign((size_t)tot + 1, 0); stats.assign(8 * (size_t)np, 0.0);
  TK(vdo_pose_opt_flow2_batch(t->ctx, t->p.quirk, np, mode.data(), offs.data(), pts.data(), dep.data(), flo.data(), Kc.data(), Tl.data(), Ti.data(), To.data(),
                              flow_out.data(), inlier.data(), stats.data()));
  T_out.resize(np);
  for (int j = 0; j < np; ++j) std::memcpy(T_out[j].data(), &To[16 * j], 64);
  return VDO_OK;
}

int track_frame(vdo_tracker* t, FrameState& C, FrameState& L) {
  const vdo_tracker_params& p = t->p;
  const float K4[4] = {p.fx, p.fy, p.cx, p.cy};
  // ---------------- camera (Tracking.cc:672-711) ----------------
  const int Ns = (int)C.statKeys.size() / 2;
  t->temperalMatch.resize(Ns);
  for (int i = 0; i < Ns; ++i) t->temperalMatch[i] = i;
  {   // GetInitModelCam (:1614-1715)
    StageTimer stage_timer_4(&t->stage_ms[4]);
    std::vector<float> obj3(3 * (size_t)Ns + 3), img2(2 * (size_t)Ns + 2);
    for (int i = 0; i < Ns; ++i) {
      img2[2 * i] = C.statKeys[2 * i]; img2[2 * i + 1] = C.statKeys[2 * i + 1];
      unproject_world(L.statKeys[2 * i], L.statKeys[2 * i + 1], L.statDepth[i], p, L.Tcw, &obj3[3 * i]);
    }
    const M4 mm = t->has_velocity ? mul4(t->velocity, L.Tcw) : L.Tcw;
    const int offs[2] = {0, Ns}; const unsigned char has = 1;
    M4 T0; int nsub = 0; std::vector<int> sub(Ns + 1);
    TK(vdo_init_model_batch(t->ctx, 1, offs, obj3.data(), img2.data(), K4, 500, 0.4, 0.98, mm.data(), &has, T0.data(), &nsub, sub.data(), nullptr, nullptr, nullptr));
    t->temperalMatchSubset.assign(sub.begin(), sub.begin() + nsub);        // MatchId[i] == i
    C.Tcw = T0;
  }
  {   // PoseOptimizationFlow2Cam (src/Optimizer.cc:2333-2542)
    StageTimer stage_timer_5(&t->stage_ms[5]);
    std::vector<FlowJob> jobs{{0, &t->temperalMatchSubset, C.Tcw}};
    std::vector<M4> To; std::vector<double> fo, st; std::vector<unsigned char> inl; std::vector<int> offs;
    if ((int)t->temperalMatchSubset.size() >= 3) {
      TK(run_flow(t, L, false, jobs, To, fo, inl, offs, st));
      C.Tcw = To[0];
      for (size_t i = 0; i < t->temperalMatchSubset.size(); ++i) {
        const int id = t->temperalMatchSubset[i];
        if (inl[i]) {
          C.statKeys[2 * id] = (float)((double)L.statKeys[2 * id] + fo[2 * i]);
          C.statKeys[2 * id + 1] = (float)((double)L.statKeys[2 * id + 1] + fo[2 * i + 1]);
        } else t->temperalMatchSubset[i] = -1;
      }
    }
  }
  t->velocity = mul4(C.Tcw, inv4(L.Tcw)); t->has_velocity = true;           // :700-706
  // ---------------- objects (:735-1003) ----------------
  const int No = (int)C.objKeys.size() / 2;
  C.flow3d.assign(3 * (size_t)No, 0.f);
  StageTimer* st_obj = new StageTimer(&t->stage_ms[6]);
  struct Guard { StageTimer*& p; ~Guard() { delete p; p = nullptr; } } guard{st_obj};
  if (No > 0) {   // GetSceneFlowObj (:1278-1364)
    std::vector<float> up(No), vp(No), uc(No), vc(No); std::vector<unsigned char> valid(No);
    for (int i = 0; i < No; ++i) { up[i] = L.objKeys[2 * i]; vp[i] = L.objKeys[2 * i + 1]; uc[i] = C.objKeys[2 * i]; vc[i] = C.objKeys[2 * i + 1]; }
    TK(vdo_scene_flow(t->ctx, No, up.data(), vp.data(), L.objDepth.data(), L.Tcw.data(), uc.data(), vc.data(), C.objDepth.data(), C.Tcw.data(), K4,
                      L.semObjLabel.data(), C.semObjLabel.data(), C.flow3d.data(), nullptr, valid.data()));
    for (int i = 0; i < No; ++i) if (!valid[i]) C.objLabel[i] = -1;
  }
  // DynObjTracking (:1366-1612)
  std::vector<int> ob(257), oi(No + 1), ml(256), sp(256);
  int nobj = 0;
  {
    std::vector<float> kx(No + 1), ky(No + 1);
    for (int i = 0; i < No; ++i) { kx[i] = C.objKeys[2 * i]; ky[i] = C.objKeys[2 * i + 1]; }
    TK(vdo_dyn_obj_tracking(t->ctx, No, C.semObjLabel.data(), C.objLabel.data(), kx.data(), ky.data(), C.objDepth.data(), C.flow3d.data(), L.semObjLabel.data(),
                            (int)L.nSemPosition.size(), L.nSemPosition.data(), L.bObjStat.data(), L.nModLabel.data(), p.height, p.width, p.is_kitti ? 25 : 0,
                            p.is_kitti ? 50 : 0, p.sf_mg_thres, p.sf_ds_thres, p.th_depth_obj, t->f_id, &t->max_id, 256, &nobj, ob.data(), oi.data(), ml.data(),
                            sp.data()));
  }
  C.nModLabel.assign(ml.begin(), ml.begin() + nobj); C.nSemPosition.assign(sp.begin(), sp.begin() + nobj);
  C.bObjStat.assign(nobj, 1); C.vObjMod.assign(nobj, eye4()); C.vnObjID.assign(nobj, {}); C.vnObjInlierID.assign(nobj, {});
  C.vObjCentre3D.assign(3 * (size_t)nobj, 0.f);
  std::vector<std::vector<int>> objIdNew(nobj);
  for (int i = 0; i < nobj; ++i) objIdNew[i].assign(oi.begin() + ob[i], oi.begin() + ob[i + 1]);
  // per object: ground-truth presence gate (:767-810), initial model (:1717-1849), joint flow / motion LM (src/Optimizer.cc:2755-2972).
  // The objects are independent of each other (disjoint point sets), so the two device stages run as one batch each.
  std::vector<int> live;
  for (int i = 0; i < nobj; ++i) {
    const int sem = C.nSemPosition[i];
    const bool g1 = std::find(L.semPosiGt.begin(), L.semPosiGt.end(), sem) != L.semPosiGt.end();
    const bool g2 = std::find(C.semPosiGt.begin(), C.semPosiGt.end(), sem) != C.semPosiGt.end();
    if (!g1 || !g2) { C.bObjStat[i] = 0; C.vnObjInlierID[i] = objIdNew[i]; continue; }
    C.vnObjID[i] = objIdNew[i];
    live.push_back(i);
  }
  if (!live.empty()) {
    const int np = (int)live.size();
    std::vector<int> offs(np + 1, 0);
    for (int j = 0; j < np; ++j) offs[j + 1] = offs[j] + (int)objIdNew[live[j]].size();
    const int tot = offs[np];
    std::vector<float> obj3(3 * (size_t)tot + 3), img2(2 * (size_t)tot + 2), Tmm(16 * (size_t)np), Tin(16 * (size_t)np);
    std::vector<unsigned char> has(np, 0);
    std::vector<int> nsub(np), sub(tot + 1);
    for (int j = 0; j < np; ++j) {
      const int i = live[j]; int q = offs[j];
      float cs[3] = {0.f, 0.f, 0.f};
      for (int id : objIdNew[i]) {
        img2[2 * q] = C.objKeys[2 * id]; img2[2 * q + 1] = C.objKeys[2 * id + 1];
        unproject_world(L.objKeys[2 * id], L.objKeys[2 * id + 1], L.objDepth[id], p, L.Tcw, &obj3[3 * q]);
        for (int r = 0; r < 3; ++r) cs[r] = cs[r] + obj3[3 * q + r];                       // ObjCentre3D_pre + x3D_p, float
        ++q;
      }
      const float inv_n = (float)(1.0 / (double)objIdNew[i].size());                     // cv::Mat / size(): convertTo with alpha = 1/n, float
      for (int r = 0; r < 3; ++r) C.vObjCentre3D[3 * (size_t)i + r] = cs[r] * inv_n;
      int pre = -1;
      for (size_t k = 0; k < L.nModLabel.size(); ++k) if (L.nModLabel[k] == C.nModLabel[i]) { pre = (int)k; break; }
      if (pre != -1) { has[j] = 1; const M4 mm = mul4(C.Tcw, L.vObjMod[pre]); std::memcpy(&Tmm[16 * j], mm.data(), 64); }
    }
    TK(vdo_init_model_batch(t->ctx, np, offs.data(), obj3.data(), img2.data(), K4, 500, 0.4, 0.98, Tmm.data(), has.data(), Tin.data(), nsub.data(), sub.data(), nullptr,
                            nullptr, nullptr));
    std::vector<std::vector<int>> idIn(np);
    std::vector<FlowJob> jobs; std::vector<int> jobObj;
    for (int j = 0; j < np; ++j) {
      const int i = live[j];
      const std::vector<int>& ids = objIdNew[i];
      std::vector<char> kept(ids.size(), 0);
      idIn[j].resize(nsub[j]);
      for (int q = 0; q < nsub[j]; ++q) { const int loc = sub[offs[j] + q]; idIn[j][q] = ids[loc]; kept[loc] = 1; }
      for (size_t q = 0; q < ids.size(); ++q) if (!kept[q]) C.objLabel[ids[q]] = -1;       // :1841-1845
      if ((int)idIn[j].size() < 50) { C.bObjStat[i] = 0; C.vnObjInlierID[i] = idIn[j]; continue; }   // :885-897
      M4 Ti; std::memcpy(Ti.data(), &Tin[16 * j], 64);
      jobs.push_back({1, &idIn[j], Ti}); jobObj.push_back(i);
    }
    if (!jobs.empty()) {
      std::vector<M4> To; std::vector<double> fo, st; std::vector<unsigned char> inl; std::vector<int> fo_offs;
      TK(run_flow(t, L, true, jobs, To, fo, inl, fo_offs, st));
      const M4 Twc = inv4(C.Tcw);
      for (size_t j = 0; j < jobs.size(); ++j) {
        const int i = jobObj[j]; const std::vector<int>& ids = *jobs[j].idx;
        std::vector<int> inlierID;
        for (size_t q = 0; q < ids.size(); ++q) {
          const int id = ids[q]; const size_t g = (size_t)fo_offs[j] + q;
          if (inl[g]) {
            C.objKeys[2 * id] = (float)((double)L.objKeys[2 * id] + fo[2 * g]);
            C.objKeys[2 * id + 1] = (float)((double)L.objKeys[2 * id + 1] + fo[2 * g + 1]);
            inlierID.push_back(id);
          } else C.objLabel[id] = -1;
        }
        C.vObjMod[i] = mul4(Twc, To[j]);                                   // :907
        C.vnObjInlierID[i] = inlierID;
      }
    }
  }
  delete st_obj; st_obj = nullptr;
  // ---------------- RenewFrameInfo (:2660-2995) ----------------
  {
    StageTimer stage_timer_7(&t->stage_ms[7]);
    const M4 Twc = inv4(C.Tcw);
    std::vector<int> ib(nobj + 1, 0), ii;
    for (int i = 0; i < nobj; ++i) { ii.insert(ii.end(), C.vnObjInlierID[i].begin(), C.vnObjInlierID[i].end()); ib[i + 1] = (int)ii.size(); }
    const std::vector<float>& samp = p.use_sample_feature ? C.sampKeys : C.keys;     // mvKeysSample (:2716-2721)
    const int nTm = (int)t->temperalMatchSubset.size(), nSamp = (int)samp.size() / 2, nTmp = (int)t->tmpSemObjLabel.size();
    const int capS = nTm + nSamp + 8, capO = (int)ii.size() + (nobj + 1) * nTmp + 8;
    std::vector<float> sk(2 * (size_t)capS), sc(2 * (size_t)capS), sf(2 * (size_t)capS), sd(capS), s3(3 * (size_t)capS);
    std::vector<int> sid(capS);
    std::vector<float> okk(2 * (size_t)capO), od(capO), oc(2 * (size_t)capO), of(2 * (size_t)capO), o3(3 * (size_t)capO);
    std::vector<int> osem(capO), oid(capO), olab(capO);
    int ns = 0, no = 0;
    TK(vdo_renew_frame_info(C.img, nTm, t->temperalMatchSubset.data(), Ns, C.statKeys.data(), nSamp, samp.data(), p.max_track_bg, nobj, ib.data(), ii.data(),
                            C.bObjStat.data(), C.nSemPosition.data(), C.nModLabel.data(), No, C.objKeys.data(), C.objLabel.data(), nTmp, t->tmpObjKeys.data(),
                            t->tmpObjDepth.data(), t->tmpSemObjLabel.data(), t->tmpObjFlowNext.data(), t->tmpObjCorres.data(), p.max_track_obj, K4, Twc.data(), capS, &ns,
                            sk.data(), sc.data(), sf.data(), sid.data(), sd.data(), s3.data(), capO, &no, okk.data(), od.data(), oc.data(), of.data(), osem.data(),
                            oid.data(), olab.data(), o3.data()));
    C.statKeysTmp.assign(sk.begin(), sk.begin() + 2 * (size_t)ns); C.corres.assign(sc.begin(), sc.begin() + 2 * (size_t)ns);
    C.flowNext.assign(sf.begin(), sf.begin() + 2 * (size_t)ns); C.statDepthTmp.assign(sd.begin(), sd.begin() + ns);
    C.stat3DTmp.assign(s3.begin(), s3.begin() + 3 * (size_t)ns); C.staInlierID.assign(sid.begin(), sid.begin() + ns);
    C.objKeys.assign(okk.begin(), okk.begin() + 2 * (size_t)no); C.objDepth.assign(od.begin(), od.begin() + no);
    C.objCorres.assign(oc.begin(), oc.begin() + 2 * (size_t)no); C.objFlowNext.assign(of.begin(), of.begin() + 2 * (size_t)no);
    C.obj3D.assign(o3.begin(), o3.begin() + 3 * (size_t)no); C.semObjLabel.assign(osem.begin(), osem.begin() + no);
    C.dynInlierID.assign(oid.begin(), oid.begin() + no); C.objLabel.assign(olab.begin(), olab.begin() + no);
  }
  return VDO_OK;
}

void push_map(vdo_tracker* t, const FrameState& C, bool first) {          // Tracking.cc:1235-1246 (first frame), :1016-1070
  MapSlice& m = t->map;
  m.featSta.push_back(C.statKeysTmp); m.depSta.push_back(C.statDepthTmp); m.p3dSta.push_back(C.stat3DTmp);
  m.featDyn.push_back(C.objKeys); m.depDyn.push_back(C.objDepth); m.p3dDyn.push_back(C.obj3D);
  m.cameraPose.push_back(first ? eye4() : inv4(C.Tcw));
  m.cameraPose_RF.push_back(m.cameraPose.back());
  if (first) return;
  m.assoSta.push_back(C.staInlierID); m.assoDyn.push_back(C.dynInlierID); m.featLabel.push_back(C.objLabel);
  std::vector<M4> mot{inv4(t->velocity)}; std::vector<int> rl{0}, sl{0};
  std::vector<float> cen{0.f, 0.f, 0.f};
  for (size_t i = 0; i < C.vObjMod.size(); ++i) {
    if (!C.bObjStat[i]) continue;
    mot.push_back(C.vObjMod[i]); rl.push_back(C.nModLabel[i]); sl.push_back(C.nSemPosition[i]);
    for (int r = 0; r < 3; ++r) cen.push_back(C.vObjCentre3D[3 * i + r]);
  }
  m.rigidMotion.push_back(mot); m.rigidMotion_RF.push_back(mot); m.rmLabel.push_back(rl); m.smLabel.push_back(sl); m.rigidCentre.push_back(cen);
}

// depth / mask at the truncated pixel of propagated keys (src/Tracking.cc:262-312)
int lookup_points(vdo_tracker* t, FrameState& C, const std::vector<float>& keys, std::vector<float>& d, std::vector<int>& m) {
  const int n = (int)keys.size() / 2;
  d.resize(n + 1); m.resize(n + 1);
  if (n == 0) return VDO_OK;
  return vdo_frame_gather(C.img, n, keys.data(), d.data(), m.data());
}
}  // namespace

extern "C" void vdo_tracker_params_default(vdo_tracker_params* p) {       // example/kitti-0000-0013.yaml
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->width = 1242; p->height = 375; p->fx = 721.5377f; p->fy = 721.5377f; p->cx = 609.5593f; p->cy = 172.8540f; p->bf = 387.5744f; p->depth_factor = 256.f;
  p->th_depth_bg = 40.f; p->th_depth_obj = 25.f; p->max_track_bg = 1200; p->max_track_obj = 800; p->sf_mg_thres = 0.12f; p->sf_ds_thres = 0.3f;
  p->n_features = 2500; p->scale_factor = 1.2f; p->n_levels = 8; p->ini_th_fast = 20; p->min_th_fast = 7; p->is_kitti = 1; p->quirk = 1;
  p->window_size = 20; p->overlap_size = 4; p->local_batch = 1;
}

extern "C" int vdo_tracker_create(vdo_ctx* ctx, const vdo_tracker_params* params, vdo_tracker** out) {
  // width == height == 0: a MAP-ONLY handle (no frame buffers): frames are pushed with vdo_tracker_map_push and optimised with
  // vdo_tracker_batch_optimize -- the form Optimizer::FullBatchOptimization(Map*, K) / PartialBatchOptimization take their input in
  const bool map_only = params && params->width == 0 && params->height == 0;
  if (!ctx || !params || !out || (!map_only && (params->width < 64 || params->height < 64))) return VDO_ERR_ARG;
  vdo_tracker* t = new vdo_tracker;
  t->ctx = ctx; t->p = *params;
  for (int i = 0; i < 2 && !map_only; ++i)
    if (vdo_frame_create(ctx, params->width, params->height, &t->fr[i].img) != VDO_OK) { vdo_tracker_destroy(t); return VDO_ERR_CUDA; }
  *out = t;
  return VDO_OK;
}
// One frame of an externally built Map (include/Map.h:34-84; what Tracking::Track pushes per frame, src/Tracking.cc:1016-1105).  Frame 0
// carries no associations / motions (n_mot == 0).  Arrays: feat (x, y) pairs, p3d xyz triples, asso / label one int per feature,
// camera_pose16 = vmCameraPose[i] (Twc, row-major), rigid_motion16 = vmRigidMotion[i - 1] (n_mot matrices, entry 0 = camera), rm_label likewise.
extern "C" int vdo_tracker_map_push(vdo_tracker* t, int n_sta, const float* feat_sta, const float* dep_sta, const float* p3d_sta, const int* asso_sta, int n_dyn,
                                    const float* feat_dyn, const float* dep_dyn, const float* p3d_dyn, const int* asso_dyn, const int* feat_label,
                                    const float* camera_pose16, int n_mot, const float* rigid_motion16, const int* rm_label) {
  if (!t || n_sta < 0 || n_dyn < 0 || n_mot < 0 || !camera_pose16) return VDO_ERR_ARG;
  if ((n_sta && (!feat_sta || !dep_sta || !p3d_sta)) || (n_dyn && (!feat_dyn || !dep_dyn || !p3d_dyn)) || (n_mot && (!rigid_motion16 || !rm_label))) return VDO_ERR_ARG;
  MapSlice& m = t->map;
  const bool first = m.featSta.empty();
  if (first != (n_mot == 0)) { t->err = "vdo_tracker_map_push: frame 0 has no motions, every later frame has at least the camera motion"; return VDO_ERR_ARG; }
  if (!first && ((n_sta && !asso_sta) || (n_dyn && (!asso_dyn || !feat_label)))) return VDO_ERR_ARG;
  m.featSta.emplace_back(feat_sta, feat_sta + 2 * (size_t)n_sta); m.depSta.emplace_back(dep_sta, dep_sta + n_sta); m.p3dSta.emplace_back(p3d_sta, p3d_sta + 3 * (size_t)n_sta);
  m.featDyn.emplace_back(feat_dyn, feat_dyn + 2 * (size_t)n_dyn); m.depDyn.emplace_back(dep_dyn, dep_dyn + n_dyn); m.p3dDyn.emplace_back(p3d_dyn, p3d_dyn + 3 * (size_t)n_dyn);
  M4 P; std::memcpy(P.data(), camera_pose16, 64);
  m.cameraPose.push_back(P); m.cameraPose_RF.push_back(P);
  if (first) return VDO_OK;
  m.assoSta.emplace_back(asso_sta, asso_sta + n_sta); m.assoDyn.emplace_back(asso_dyn, asso_dyn + n_dyn); m.featLabel.emplace_back(feat_label, feat_label + n_dyn);
  std::vector<M4> mot(n_mot);
  for (int j = 0; j < n_mot; ++j) std::memcpy(mot[j].data(), rigid_motion16 + 16 * (size_t)j, 64);
  m.rigidMotion.push_back(mot); m.rigidMotion_RF.push_back(mot);
  m.rmLabel.emplace_back(rm_label, rm_label + n_mot); m.smLabel.emplace_back(rm_label, rm_label + n_mot);
  m.rigidCentre.emplace_back(3 * (size_t)n_mot, 0.f);
  return VDO_OK;
}
extern "C" void vdo_tracker_destroy(vdo_tracker* t) {
  if (!t) return;
  for (int i = 0; i < 2; ++i) if (t->fr[i].img) vdo_frame_destroy(t->fr[i].img);
  delete t;
}
extern "C" const char* vdo_tracker_last_error(const vdo_tracker* t) { return t ? t->err.c_str() : "null tracker"; }

// System::TrackRGBD / Tracking::GrabImageRGBD (include/System.h:49-51, src/Tracking.cc:164-648)
extern "C" int vdo_tracker_track(vdo_tracker* t, int width, int height, const unsigned char* gray, float* depth, const float* flow, int* mask, int n_gt,
                                 const int* gt_sem_ids, int writeback, float* Tcw_out) {
  if (!t || !gray || !depth || !flow || !mask || n_gt < 0) return VDO_ERR_ARG;
  const vdo_tracker_params& p = t->p;
  if (!t->fr[0].img) { t->err = "vdo_tracker_track on a map-only handle"; return VDO_ERR_STATE; }
  if (width != p.width || height != p.height) {
    t->err = "vdo_tracker_track: buffers are " + std::to_string(width) + "x" + std::to_string(height) + " but the tracker was created for " + std::to_string(p.width) + "x" +
             std::to_string(p.height);
    return VDO_ERR_ARG;
  }
  if (!t->first) t->cur = 1 - t->cur;
  FrameState& C = t->fr[t->cur]; FrameState& L = t->fr[1 - t->cur];
  vdo_frame* img = C.img;
  C.clear_dynamic(); C.img = img; C.Tcw = eye4();
  if (t->first) t->f_id = 0;
  t->sample_seed = 0;
  {
    StageTimer stage_timer_0(&t->stage_ms[0]);
    TK(vdo_frame_upload(C.img, gray, depth, flow, mask));
    const int dataset = p.dataset ? p.dataset : (p.is_kitti ? 2 : 1);
    TK(vdo_frame_depth_prep(C.img, dataset == 3 ? 0.f : p.bf, p.depth_factor, writeback ? depth : nullptr));      // :180-204, in place on the caller's Mat
  }
  if (!t->first) {                                                                            // UpdateMask (:2997-3110)
    const int n = (int)L.semObjLabel.size();
    std::vector<float> cx(n + 1), cy(n + 1);
    for (int i = 0; i < n; ++i) { cx[i] = L.objCorres[2 * i]; cy[i] = L.objCorres[2 * i + 1]; }
    int nw = 0;
    StageTimer stage_timer_1(&t->stage_ms[1]);
    TK(vdo_update_mask(C.img, L.img, n, L.semObjLabel.data(), cx.data(), cy.data(), nullptr, &nw, nullptr));
    if (writeback && nw > 0) TK(vdo_frame_read_mask(C.img, mask));        // the caller's buffer already holds the mask unless an object was warped into it
  }
  {
    StageTimer stage_timer_2(&t->stage_ms[2]);
    TK(build_frame(t, C));
  }
  if (!t->first) {                                                                            // :254-312
    StageTimer stage_timer_3(&t->stage_ms[3]);
    C.statKeys = L.corres;
    std::vector<int> mk;
    TK(lookup_points(t, C, C.statKeys, C.statDepth, mk));
    const int Ns = (int)C.statKeys.size() / 2;
    C.statDepth.resize(Ns);
    for (int i = 0; i < Ns; ++i) {
      const int u = (int)C.statKeys[2 * i], v = (int)C.statKeys[2 * i + 1];
      const bool in = u < p.width - 1 && u > 0 && v < p.height - 1 && v > 0;
      C.statDepth[i] = (in && C.statDepth[i] > 0) ? C.statDepth[i] : -1.f;
    }
    t->tmpObjKeys = C.objKeys; t->tmpObjDepth = C.objDepth; t->tmpSemObjLabel = C.semObjLabel; t->tmpObjFlowNext = C.objFlowNext; t->tmpObjCorres = C.objCorres;
    C.objKeys = L.objCorres;
    std::vector<float> od; std::vector<int> om;
    TK(lookup_points(t, C, C.objKeys, od, om));
    const int No = (int)C.objKeys.size() / 2;
    C.objDepth.assign(No, 0.1f); C.semObjLabel.assign(No, 0);
    for (int i = 0; i < No; ++i) {
      const int u = (int)C.objKeys[2 * i], v = (int)C.objKeys[2 * i + 1];
      if (u < p.width - 1 && u > 0 && v < p.height - 1 && v > 0 && od[i] < p.th_depth_obj && od[i] > 0) { C.objDepth[i] = od[i]; C.semObjLabel[i] = om[i]; }
    }
  }
  C.semPosiGt.assign(gt_sem_ids, gt_sem_ids + n_gt);
  C.objLabel.assign(C.objKeys.size() / 2, -2);                                                // :345
  if (t->first) {                                                                             // Initialization (:1215-1276)
    const int ns = (int)C.statKeysTmp.size() / 2, no = (int)C.objKeys.size() / 2;
    C.stat3DTmp.resize(3 * (size_t)ns); C.obj3D.resize(3 * (size_t)no);
    for (int i = 0; i < ns; ++i) get3d_camera(C.statKeysTmp[2 * i], C.statKeysTmp[2 * i + 1], C.statDepthTmp[i], p, &C.stat3DTmp[3 * i]);
    for (int i = 0; i < no; ++i) get3d_camera(C.objKeys[2 * i], C.objKeys[2 * i + 1], C.objDepth[i], p, &C.obj3D[3 * i]);
    C.Tcw = eye4();
    push_map(t, C, true);
    t->first = false;
  } else {
    TK(track_frame(t, C, L));
    push_map(t, C, false);
  }
  // mLastFrame = Frame(mCurrentFrame) with the "new added" overrides (:1006-1014): the next call reads this frame through L
  C.statKeys = C.statKeysTmp; C.statDepth = C.statDepthTmp;
  // windowed optimisation on the reference's schedule (src/Tracking.cc:1150-1160)
  if (p.local_batch && p.window_size > p.overlap_size && p.overlap_size >= 0 && (t->f_id - p.overlap_size + 1) % (p.window_size - p.overlap_size) == 0 &&
      t->f_id >= p.window_size - 1) {
    StageTimer stage_timer_ba(&t->stage_ms[8]);
    vdo_lm_stats st;
    TK(vdo_tracker_batch_optimize(t, 0, nullptr, &st, nullptr));
    t->local_ba_runs += 1; t->local_ba_iters += st.iterations;
  }
  t->f_id += 1; t->frames += 1;
  if (Tcw_out) std::memcpy(Tcw_out, C.Tcw.data(), 64);
  return VDO_OK;
}

// Named read-back of the state after the last vdo_tracker_track call (parity tests, host shim).  kind: 'f' float, 'i' int.
// Names: Tcw, mvKeys, mvStatKeys(Tmp), mvStatDepth(Tmp), mvCorres, mvFlowNext, mvStat3DPointTmp, nStaInlierID, mvObjKeys, mvObjDepth, mvObjCorres,
// mvObjFlowNext, mvObj3DPoint, vSemObjLabel, vObjLabel, nDynInlierID, vFlow_3d, nModLabel, nSemPosition, bObjStat, vObjMod, TemperalMatch_subset,
// max_id, f_id, mVelocity, sample_seed
extern "C" int vdo_tracker_get(const vdo_tracker* t, const char* name, void* out, int cap_elems, int* n_elems) {
  if (!t || !name || !n_elems) return VDO_ERR_ARG;
  const FrameState& C = t->fr[t->cur];
  const std::string s(name);
  auto put_f = [&](const float* p, size_t n) { *n_elems = (int)n; if (out && (int)n <= cap_elems && n) std::memcpy(out, p, n * 4); return (out && (int)n > cap_elems) ? VDO_ERR_ARG : VDO_OK; };
  auto put_i = [&](const int* p, size_t n) { *n_elems = (int)n; if (out && (int)n <= cap_elems && n) std::memcpy(out, p, n * 4); return (out && (int)n > cap_elems) ? VDO_ERR_ARG : VDO_OK; };
  if (s == "Tcw") return put_f(C.Tcw.data(), 16);
  if (s == "mVelocity") return put_f(t->velocity.data(), 16);
  if (s == "mvKeys") return put_f(C.keys.data(), C.keys.size());
  if (s == "mvStatKeys" || s == "mvStatKeysTmp") return put_f(C.statKeysTmp.data(), C.statKeysTmp.size());
  if (s == "mvStatDepth" || s == "mvStatDepthTmp") return put_f(C.statDepthTmp.data(), C.statDepthTmp.size());
  if (s == "mvCorres") return put_f(C.corres.data(), C.corres.size());
  if (s == "mvFlowNext") return put_f(C.flowNext.data(), C.flowNext.size());
  if (s == "mvStat3DPointTmp") return put_f(C.stat3DTmp.data(), C.stat3DTmp.size());
  if (s == "nStaInlierID") return put_i(C.staInlierID.data(), C.staInlierID.size());
  if (s == "mvObjKeys") return put_f(C.objKeys.data(), C.objKeys.size());
  if (s == "mvObjDepth") return put_f(C.objDepth.data(), C.objDepth.size());
  if (s == "mvObjCorres") return put_f(C.objCorres.data(), C.objCorres.size());
  if (s == "mvObjFlowNext") return put_f(C.objFlowNext.data(), C.objFlowNext.size());
  if (s == "mvObj3DPoint") return put_f(C.obj3D.data(), C.obj3D.size());
  if (s == "vSemObjLabel") return put_i(C.semObjLabel.data(), C.semObjLabel.size());
  if (s == "vObjLabel") return put_i(C.objLabel.data(), C.objLabel.size());
  if (s == "nDynInlierID") return put_i(C.dynInlierID.data(), C.dynInlierID.size());
  if (s == "vFlow_3d") return put_f(C.flow3d.data(), C.flow3d.size());
  if (s == "nModLabel") return put_i(C.nModLabel.data(), C.nModLabel.size());
  if (s == "nSemPosition") return put_i(C.nSemPosition.data(), C.nSemPosition.size());
  if (s == "TemperalMatch_subset") return put_i(t->temperalMatchSubset.data(), t->temperalMatchSubset.size());
  if (s == "bObjStat") { std::vector<int> v(C.bObjStat.begin(), C.bObjStat.end()); return put_i(v.data(), v.size()); }
  if (s == "vObjCentre3D") return put_f(C.vObjCentre3D.data(), C.vObjCentre3D.size());
  if (s == "vObjMod") { std::vector<float> v; for (auto& m : C.vObjMod) v.insert(v.end(), m.begin(), m.end()); return put_f(v.data(), v.size()); }
  if (s == "max_id") return put_i(&t->max_id, 1);
  if (s == "f_id") return put_i(&t->f_id, 1);
  if (s == "stage_ms") { float v[9]; for (int i = 0; i < 9; ++i) v[i] = (float)t->stage_ms[i]; return put_f(v, 9); }
  if (s == "local_ba") { const int v[2] = {t->local_ba_runs, t->local_ba_iters}; return put_i(v, 2); }
  if (s == "sample_seed") return put_i(reinterpret_cast<const int*>(&t->sample_seed), 1);
  return VDO_ERR_ARG;
}

// ------------------------------------------------------------------------------------------------ Map -> factor graph (SURVEY.md 8f N2)
// Graph construction of Optimizer::FullBatchOptimization (src/Optimizer.cc:1232-1767) and Optimizer::PartialBatchOptimization
// (:42-805) from the tracker's map, emitted as the arrays of the vdo_graph_* calls; refined camera poses, object motions and
// points are written back like :2094-2172 / :983-1050.  Where the reference would dereference a null vertex (a track whose
// previous position never received a vertex) the edge is skipped.
#include "ba_math.cuh"

namespace {
struct GraphArrays {
  std::vector<double> se3, pt, prior_Z, prior_w, se3e_Z, se3e_w, se3e_delta, obs_z, obs_w, obs_delta, ter_w, ter_delta;
  std::vector<int> prior_v, se3e_ij, obs_cp, ter_pph;
  std::vector<int> cam_vid;                       // per frame: se3 index of the camera vertex (-1 outside the window)
  std::vector<std::vector<int>> mot_vid;          // per frame pair: se3 index of each rigid-motion vertex (entry 0 unused)
  std::vector<std::vector<int>> makS, makD;       // per frame, per feature: point index (-1 = not in the graph)
  int max_iters = 300; double gain = 1e-4;
};
struct BatchConsts { float sigma2_cam, sigma2_3d_sta, sigma2_obj_smo, sigma2_obj, sigma2_3d_dyn; double prior_w; bool static_only; int max_iters; double gain; };
const BatchConsts kFull{0.001f, 80.f, 0.001f, 100.f, 80.f, 100000.0, false, 300, 1e-4};                 // src/Optimizer.cc:1330-1335
const BatchConsts kPartial{0.0001f, 16.f, 0.1f, 20.f, 16.f, 1.0 / 0.0000001, true, 100, 1e-3};          // :190-195, :230

// Converter::toSE3Quat (src/Converter.cc:25-35) + SE3Quat -> Isometry3d (se3quat.h): rotation re-normalised through the quaternion
void to_iso(const M4& T, double* out) {
  double R[9], q[4];
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) R[3 * i + j] = (double)T[4 * i + j];
  vdo::quat_from_rot(R, q);
  if (q[3] < 0) { q[0] = -q[0]; q[1] = -q[1]; q[2] = -q[2]; q[3] = -q[3]; }
  const double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int k = 0; k < 4; ++k) q[k] /= n;
  vdo::rot_from_quat(q, out);
  out[9] = (double)T[3]; out[10] = (double)T[7]; out[11] = (double)T[11];
}
// getEstimateData -> Quaterniond -> rotation matrix -> Converter::toCvSE3 (src/Optimizer.cc:2094-2110)
M4 from_iso(const double* T) {
  double q[4], R[9];
  vdo::quat_from_rot(T, q);
  const double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int k = 0; k < 4; ++k) q[k] /= n;
  vdo::rot_from_quat(q, R);
  M4 m = eye4();
  for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) m[4 * i + j] = (float)R[3 * i + j]; m[4 * i + 3] = (float)T[9 + i]; }
  return m;
}

int build_tracklets(const std::vector<std::vector<int>>& asso, const std::vector<std::vector<int>>* labels, std::vector<std::vector<std::pair<int, int>>>& tracks,
                    std::vector<int>& obj_id) {
  const int n_rows = (int)asso.size();
  std::vector<int> rb(n_rows + 1, 0), flat, lab;
  for (int i = 0; i < n_rows; ++i) {
    flat.insert(flat.end(), asso[i].begin(), asso[i].end());
    if (labels) lab.insert(lab.end(), (*labels)[i].begin(), (*labels)[i].end());
    rb[i + 1] = (int)flat.size();
  }
  int cnt = 0;
  for (int v : flat) cnt += v != -1;
  const int max_t = cnt + 1, max_e = 2 * cnt + 2;
  std::vector<int> tb(max_t + 1), tf(max_e), tk(max_e), oid(max_t);
  int nt = 0;
  const int rc = vdo_tracklets_build(n_rows, rb.data(), flat.data(), labels ? lab.data() : nullptr, max_t, max_e, &nt, tb.data(), tf.data(), tk.data(), oid.data());
  if (rc != VDO_OK) return rc;
  tracks.assign(nt, {});
  for (int t = 0; t < nt; ++t) for (int e = tb[t]; e < tb[t + 1]; ++e) tracks[t].push_back({tf[e], tk[e]});
  obj_id.assign(oid.begin(), oid.begin() + nt);
  return VDO_OK;
}

int build_graph(vdo_tracker* t, bool full, GraphArrays& G) {
  const MapSlice& m = t->map;
  const BatchConsts& c = full ? kFull : kPartial;
  const int N = (int)m.featSta.size(), window = t->p.window_size;
  if (N < 2 || (!full && (window < 2 || N < window))) return VDO_ERR_STATE;
  std::vector<std::vector<std::pair<int, int>>> staT, dynT; std::vector<int> objId, dummy;
  TK(build_tracklets(m.assoSta, nullptr, staT, dummy));
  TK(build_tracklets(m.assoDyn, &m.featLabel, dynT, objId));
  std::vector<std::vector<int>> labS(N), labD(N);
  G = GraphArrays();
  G.makS.resize(N); G.makD.resize(N); G.cam_vid.assign(N, -1); G.mot_vid.resize(N - 1);
  for (int i = 0; i < N; ++i) {
    labS[i].assign(m.featSta[i].size() / 2, -1); G.makS[i].assign(m.featSta[i].size() / 2, -1);
    labD[i].assign(m.featDyn[i].size() / 2, -1); G.makD[i].assign(m.featDyn[i].size() / 2, -1);
    if (i < N - 1) G.mot_vid[i].assign(m.rmLabel[i].size(), -1);
  }
  for (size_t k = 0; k < staT.size(); ++k) if (staT[k].size() >= 3) for (auto& pr : staT[k]) labS[pr.first][pr.second] = (int)k;
  for (size_t k = 0; k < dynT.size(); ++k) if (dynT[k].size() >= 3) for (auto& pr : dynT[k]) labD[pr.first][pr.second] = (int)k;
  G.max_iters = c.max_iters; G.gain = c.gain;
  const double huber = (double)0.0001f;
  const double ident[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
  auto n_se3 = [&]() { return (int)G.se3.size() / 12; };
  auto n_pt = [&]() { return (int)G.pt.size() / 3; };
  auto add_obs = [&](int cam, int p, const float* key, float dep, double w) {
    G.obs_cp.push_back(cam); G.obs_cp.push_back(p);
    float X[3]; get3d_camera(key[0], key[1], dep, t->p, X);
    for (int k = 0; k < 3; ++k) G.obs_z.push_back((double)X[k]);
    G.obs_w.push_back(w); G.obs_delta.push_back(huber);
  };
  auto add_pt = [&](const float* X) { for (int k = 0; k < 3; ++k) G.pt.push_back((double)X[k]); return n_pt() - 1; };
  auto find_pos = [](const std::vector<std::pair<int, int>>& tr, int f, int j) { for (size_t k = 0; k < tr.size(); ++k) if (tr[k].first == f && tr[k].second == j) return (int)k; return -1; };
  const int start = full ? 0 : N - window;
  int pre = -1;
  for (int i = start; i < N; ++i) {
    const int cur = n_se3();
    double iso[12]; to_iso(m.cameraPose[i], iso);
    G.se3.insert(G.se3.end(), iso, iso + 12); G.cam_vid[i] = cur;
    if (cur == 0 && (full || N == window)) { G.prior_v.push_back(cur); G.prior_Z.insert(G.prior_Z.end(), iso, iso + 12); G.prior_w.push_back(c.prior_w); }
    if (i != start) {
      double z[12]; to_iso(m.rigidMotion[i - 1][0], z);
      G.se3e_ij.push_back(pre); G.se3e_ij.push_back(cur); G.se3e_Z.insert(G.se3e_Z.end(), z, z + 12);
      G.se3e_w.push_back(1.0 / (double)c.sigma2_cam); G.se3e_delta.push_back(huber);
    }
    for (size_t j = 0; j < labS[i].size(); ++j) {                       // static points (:1402-1516 / :254-349)
      const int tid = labS[i][j];
      if (tid == -1) continue;
      const int pos = find_pos(staT[tid], i, (int)j);
      if (pos == -1) continue;
      const double w = 1.0 / (double)c.sigma2_3d_sta;
      int p;
      if (pos == 0) p = add_pt(&m.p3dSta[i][3 * j]);
      else { p = G.makS[staT[tid][pos - 1].first][staT[tid][pos - 1].second]; if (p == -1) continue; }
      add_obs(cur, p, &m.featSta[i][2 * j], m.depSta[i][j], w);
      G.makS[i][j] = p;
    }
    if (!c.static_only && i == 0) {                                    // :1521-1549
      for (size_t j = 0; j < labD[i].size(); ++j) {
        if (labD[i][j] == -1) continue;
        const int p = add_pt(&m.p3dDyn[i][3 * j]);
        add_obs(cur, p, &m.featDyn[i][2 * j], m.depDyn[i][j], 1.0 / (double)c.sigma2_3d_dyn);
        G.makD[i][j] = p;
      }
    } else if (!c.static_only) {                                       // :1551-1762
      std::vector<int> objUid;
      for (size_t j = 1; j < m.rigidMotion[i - 1].size(); ++j) {
        const int v = n_se3();
        G.se3.insert(G.se3.end(), ident, ident + 12);
        if (i > 2) {
          int trace = -1;
          for (size_t k = 0; k < m.rmLabel[i - 2].size(); ++k) if (m.rmLabel[i - 2][k] == m.rmLabel[i - 1][j]) { trace = (int)k; break; }
          if (trace != -1 && G.mot_vid[i - 2][trace] != -1) {
            G.se3e_ij.push_back(G.mot_vid[i - 2][trace]); G.se3e_ij.push_back(v); G.se3e_Z.insert(G.se3e_Z.end(), ident, ident + 12);
            G.se3e_w.push_back(1.0 / (double)c.sigma2_obj_smo); G.se3e_delta.push_back(huber);
          }
        }
        objUid.push_back(v); G.mot_vid[i - 1][j] = v;
      }
      for (size_t j = 0; j < labD[i].size(); ++j) {
        const int tid = labD[i][j];
        if (tid == -1) continue;
        const int pos = find_pos(dynT[tid], i, (int)j);
        if (pos == -1) continue;
        int objv = -1;
        for (size_t k = 1; k < m.rmLabel[i - 1].size(); ++k) if (m.rmLabel[i - 1][k] == objId[tid]) { objv = objUid[k - 1]; break; }
        if (objv == -1 && pos != 0) continue;
        const int p = add_pt(&m.p3dDyn[i][3 * j]);
        add_obs(cur, p, &m.featDyn[i][2 * j], m.depDyn[i][j], 1.0 / (double)c.sigma2_3d_dyn);
        if (pos != 0) {
          const int q = G.makD[dynT[tid][pos - 1].first][dynT[tid][pos - 1].second];
          if (q != -1) { G.ter_pph.push_back(q); G.ter_pph.push_back(p); G.ter_pph.push_back(objv); G.ter_w.push_back(1.0 / (double)c.sigma2_obj); G.ter_delta.push_back(huber); }
        }
        G.makD[i][j] = p;
      }
    }
    pre = cur;
  }
  return VDO_OK;
}
}  // namespace

// mode 0 = PartialBatchOptimization over the last window_size frames, 1 = FullBatchOptimization.  Builds the graph from the map,
// runs vdo_graph_optimize (opt may be NULL: the reference's iteration cap and gain threshold) and writes the refined camera poses,
// motions and points back into the map.  info (may be NULL): n_se3, n_pt, n_prior, n_se3_edges, n_obs, n_ternary.
extern "C" int vdo_tracker_batch_optimize(vdo_tracker* t, int mode, const vdo_lm_options* opt, vdo_lm_stats* stats, int* info) {
  if (!t || (mode != 0 && mode != 1)) return VDO_ERR_ARG;
  GraphArrays G;
  const bool prof = std::getenv("VDO_PROFILE") != nullptr;
  const auto tp0 = std::chrono::steady_clock::now();
  auto lap_ms = [&](const std::chrono::steady_clock::time_point& a) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count(); };
  TK(build_graph(t, mode == 1, G));
  const double ms_build = lap_ms(tp0);
  const int ns = (int)G.se3.size() / 12, np = (int)G.pt.size() / 3;
  if (info) { info[0] = ns; info[1] = np; info[2] = (int)G.prior_v.size(); info[3] = (int)G.se3e_w.size(); info[4] = (int)G.obs_w.size(); info[5] = (int)G.ter_w.size(); }
  vdo_graph* g = nullptr;
  TK(vdo_graph_create(t->ctx, &g));
  int rc = vdo_graph_set_vertices(g, ns, G.se3.data(), np, G.pt.data());
  if (rc == VDO_OK && !G.prior_v.empty()) rc = vdo_graph_add_edges_se3_prior(g, (int)G.prior_v.size(), G.prior_v.data(), G.prior_Z.data(), G.prior_w.data());
  if (rc == VDO_OK && !G.se3e_w.empty()) rc = vdo_graph_add_edges_se3(g, (int)G.se3e_w.size(), G.se3e_ij.data(), G.se3e_Z.data(), G.se3e_w.data(), G.se3e_delta.data());
  if (rc == VDO_OK && !G.obs_w.empty()) rc = vdo_graph_add_edges_se3_pointxyz(g, (int)G.obs_w.size(), G.obs_cp.data(), G.obs_z.data(), G.obs_w.data(), G.obs_delta.data());
  if (rc == VDO_OK && !G.ter_w.empty()) rc = vdo_graph_add_edges_landmark_motion(g, (int)G.ter_w.size(), G.ter_pph.data(), G.ter_w.data(), G.ter_delta.data());
  if (rc == VDO_OK) rc = vdo_graph_finalize(g);
  const double ms_ingest = lap_ms(tp0) - ms_build;
  vdo_lm_options o;
  if (opt) o = *opt; else { vdo_lm_options_default(&o); o.max_iterations = G.max_iters; o.gain_threshold = G.gain; }
  vdo_lm_stats st_local;
  if (rc == VDO_OK) rc = vdo_graph_optimize(g, &o, stats ? stats : &st_local, nullptr);
  const double ms_opt = lap_ms(tp0) - ms_build - ms_ingest;
  std::vector<double> se3(12 * (size_t)ns + 12), pt(3 * (size_t)np + 3);
  if (rc == VDO_OK) rc = vdo_graph_get_vertices(g, se3.data(), pt.data());
  vdo_graph_destroy(g);
  if (prof) std::fprintf(stderr, "[vdo_b200] batch_optimize mode %d: %d se3, %d points, %d obs | build %.2f ms | ingest %.2f | optimise %.2f (%d LM it) | read-back+free %.2f\n", mode, ns, np,
                         (int)G.obs_w.size(), ms_build, ms_ingest, ms_opt, (stats ? stats : &st_local)->iterations, lap_ms(tp0) - ms_build - ms_ingest - ms_opt);
  if (rc != VDO_OK) { t->err = std::string("batch optimisation failed: ") + vdo_last_error(t->ctx); return rc; }
  MapSlice& m = t->map;
  const int N = (int)m.featSta.size();
  // PartialBatchOptimization writes vmCameraPose / vmRigidMotion (src/Optimizer.cc:1058-1101); FullBatchOptimization writes
  // vmCameraPose_RF[i + 1] / vmRigidMotion_RF and leaves the initial estimates alone (:2094-2133); both update the points
  std::vector<M4>& camOut = mode == 1 ? m.cameraPose_RF : m.cameraPose;
  std::vector<std::vector<M4>>& motOut = mode == 1 ? m.rigidMotion_RF : m.rigidMotion;
  for (int i = 0; i < N; ++i) {
    if (G.cam_vid[i] != -1 && (mode == 0 || i > 0)) camOut[i] = from_iso(&se3[12 * (size_t)G.cam_vid[i]]);
    for (size_t j = 0; j < G.makS[i].size(); ++j) if (G.makS[i][j] != -1) for (int k = 0; k < 3; ++k) m.p3dSta[i][3 * j + k] = (float)pt[3 * (size_t)G.makS[i][j] + k];
    for (size_t j = 0; j < G.makD[i].size(); ++j) if (G.makD[i][j] != -1) for (int k = 0; k < 3; ++k) m.p3dDyn[i][3 * j + k] = (float)pt[3 * (size_t)G.makD[i][j] + k];
  }
  for (int i = 0; i + 1 < N; ++i) {
    if (mode == 0) { if (G.cam_vid[i] != -1 && G.cam_vid[i + 1] != -1) m.rigidMotion[i][0] = mul4(inv4(m.cameraPose[i]), m.cameraPose[i + 1]); }   // :1001
    for (size_t j = 1; j < G.mot_vid[i].size(); ++j) if (G.mot_vid[i][j] != -1) motOut[i][j] = from_iso(&se3[12 * (size_t)G.mot_vid[i][j]]);
  }
  return VDO_OK;
}

// graph arrays of the last build for a mode (parity tests): name in {se3, pt, prior_Z, prior_w, se3e_Z, se3e_w, se3e_delta, obs_z, obs_w, obs_delta, ter_w,
// ter_delta} (f64) or {prior_v, se3e_ij, obs_cp, ter_pph} (i32; out is then an int buffer)
extern "C" int vdo_tracker_graph_export(vdo_tracker* t, int mode, const char* name, void* out, int cap_elems, int* n_elems) {
  if (!t || !name || !n_elems) return VDO_ERR_ARG;
  GraphArrays G;
  TK(build_graph(t, mode == 1, G));
  const std::string s(name);
  const std::vector<double>* d = nullptr; const std::vector<int>* iv = nullptr;
  if (s == "se3") d = &G.se3; else if (s == "pt") d = &G.pt; else if (s == "prior_Z") d = &G.prior_Z; else if (s == "prior_w") d = &G.prior_w;
  else if (s == "se3e_Z") d = &G.se3e_Z; else if (s == "se3e_w") d = &G.se3e_w; else if (s == "se3e_delta") d = &G.se3e_delta; else if (s == "obs_z") d = &G.obs_z;
  else if (s == "obs_w") d = &G.obs_w; else if (s == "obs_delta") d = &G.obs_delta; else if (s == "ter_w") d = &G.ter_w; else if (s == "ter_delta") d = &G.ter_delta;
  else if (s == "prior_v") iv = &G.prior_v; else if (s == "se3e_ij") iv = &G.se3e_ij; else if (s == "obs_cp") iv = &G.obs_cp; else if (s == "ter_pph") iv = &G.ter_pph;
  else return VDO_ERR_ARG;
  const size_t n = d ? d->size() : iv->size();
  *n_elems = (int)n;
  if (!out) return VDO_OK;
  if ((int)n > cap_elems) return VDO_ERR_ARG;
  if (n) std::memcpy(out, d ? (const void*)d->data() : (const void*)iv->data(), n * (d ? 8 : 4));
  return VDO_OK;
}

// map read-back: "vmCameraPose" / "vmCameraPose_RF" (N x 16 f32), "vmRigidMotion" / "vmRigidMotion_RF" (all frames concatenated, 16 f32 each),
// "vmRigidCentre" (3 f32 each, same order), "vnRMLabel" (i32, same order), "n_per_frame" (entries per frame, i32), "n_frames"
extern "C" int vdo_tracker_map_get(const vdo_tracker* t, const char* name, void* out, int cap_elems, int* n_elems) {
  if (!t || !name || !n_elems) return VDO_ERR_ARG;
  const std::string s(name);
  std::vector<float> f; std::vector<int> iv; bool is_f = true;
  if (s == "vmCameraPose") for (auto& T : t->map.cameraPose) f.insert(f.end(), T.begin(), T.end());
  else if (s == "vmCameraPose_RF") for (auto& T : t->map.cameraPose_RF) f.insert(f.end(), T.begin(), T.end());
  else if (s == "vmRigidMotion") { for (auto& fr : t->map.rigidMotion) for (auto& T : fr) f.insert(f.end(), T.begin(), T.end()); }
  else if (s == "vmRigidMotion_RF") { for (auto& fr : t->map.rigidMotion_RF) for (auto& T : fr) f.insert(f.end(), T.begin(), T.end()); }
  else if (s == "vmRigidCentre") { for (auto& fr : t->map.rigidCentre) f.insert(f.end(), fr.begin(), fr.end()); }
  else if (s == "n_per_frame") { is_f = false; for (auto& fr : t->map.rmLabel) iv.push_back((int)fr.size()); }
  else if (s == "vp3DPointSta") { for (auto& fr : t->map.p3dSta) f.insert(f.end(), fr.begin(), fr.end()); }      // all frames concatenated, xyz per feature
  else if (s == "vp3DPointDyn") { for (auto& fr : t->map.p3dDyn) f.insert(f.end(), fr.begin(), fr.end()); }
  else if (s == "vnRMLabel") { is_f = false; for (auto& fr : t->map.rmLabel) iv.insert(iv.end(), fr.begin(), fr.end()); }
  else if (s == "n_frames") { is_f = false; iv.push_back((int)t->map.featSta.size()); }
  else return VDO_ERR_ARG;
  const size_t n = is_f ? f.size() : iv.size();
  *n_elems = (int)n;
  if (!out) return VDO_OK;
  if ((int)n > cap_elems) return VDO_ERR_ARG;
  if (n) std::memcpy(out, is_f ? (const void*)f.data() : (const void*)iv.data(), n * 4);
  return VDO_OK;
}
