"""oracle/sampled_features.py -- TEST INFRASTRUCTURE ONLY: CPU restatement of the sampled background features (UseSampleFeature: 1).

  cv::RNG                   OpenCV core (3.4 and 4.x): multiply-with-carry on a 64-bit state; pinned against cv2.randu in
                            tests/test_sampled_features.py
  Frame::SampleKeyPoints    src/Frame.cc:672-740
  Option II filter          src/Frame.cc:130-194
  RenewFrameInfo top-up     src/Tracking.cc:2716-2721 (mvKeysSample = mCurrentFrame.mvStatKeysTmp)

SampledOracleTracker extends the oracle pipeline of tracking_pipeline.py with the setting; with use_sample_feature=False it is that
pipeline unchanged.
"""
import numpy as np

from .tracking_pipeline import OracleTracker

f32 = np.float32


class CvRNG:
    """cv::RNG, exact integers."""
    A = 4164903690
    M = A * 2 ** 32 - 1                    # one step == multiplication by R = 2^-32 modulo M
    R = pow(2 ** 32, -1, M)

    def __init__(self, seed):
        self.state = seed if seed else 0xFFFFFFFF

    def next(self):
        self.state = (self.state & 0xFFFFFFFF) * self.A + (self.state >> 32)
        return self.state & 0xFFFFFFFF

    def uniform(self, a, b):
        """RNG::uniform(int a, int b): draws nothing when a == b."""
        return a if a == b else self.next() % (b - a) + a

    @classmethod
    def state_after(cls, seed, k):
        """State after k draws in closed form: seed * R^k mod M."""
        return (seed if seed else 0xFFFFFFFF) * pow(cls.R, k, cls.M) % cls.M


SAMPLE_N, SAMPLE_DIV = 3000, 20


def sample_keypoints(rows, cols, seed):
    """Frame::SampleKeyPoints with cv::RNG(seed): (3000, 2) float32 pixels, cell-major (KeyinGrid[i*20+j]), draw order within a cell."""
    rng = CvRNG(seed)
    N, n_div = SAMPLE_N, SAMPLE_DIV
    grid = [[] for _ in range(n_div * n_div)]
    x_step, y_step = cols // n_div, rows // n_div
    key_num = 0
    while key_num < N:
        for i in range(n_div):
            for j in range(n_div):
                x = float(rng.uniform(i * x_step, (i + 1) * x_step))
                y = float(rng.uniform(j * y_step, (j + 1) * y_step))
                if x >= cols or y >= rows or x <= 0 or y <= 0:
                    continue
                grid[i * n_div + j].append((x, y))
                key_num += 1
                if key_num >= N:
                    break
            if key_num >= N:
                break
    return np.asarray([k for cell in grid for k in cell], f32).reshape(-1, 2)


def filter_sampled(keys, mask, depth, flow, th_depth):
    """Option II of the Frame constructor: the samples with mask == 0, 0 < depth <= th, non-zero flow whose target is strictly inside the
    image.  Returns kept keys (n, 2), correspondences (n, 2), flows (n, 2), depths (-1 where not > 0)."""
    h, w = mask.shape
    kk, cc, ff, dd = [], [], [], []
    for kx, ky in np.asarray(keys, f32):
        x, y = int(kx), int(ky)
        if mask[y, x] != 0:
            continue
        d = depth[y, x]
        if d > f32(th_depth) or d <= 0:
            continue
        fx, fy = flow[y, x, 0], flow[y, x, 1]
        if fx != 0 and fy != 0:
            tx, ty = f32(kx + fx), f32(ky + fy)
            if tx < w and ty < h and tx > 0 and ty > 0:
                kk.append((kx, ky)); cc.append((tx, ty)); ff.append((fx, fy)); dd.append(d if d > 0 else f32(-1))
    f2 = lambda a: np.asarray(a, f32).reshape(-1, 2)
    return f2(kk), f2(cc), f2(ff), np.asarray(dd, f32)


class SampledOracleTracker(OracleTracker):
    """OracleTracker with UseSampleFeature.  sample_seed is the cv::RNG seed of the next frame; a test may set it per frame to replay a
    time-seeded run."""

    def __init__(self, *args, use_sample_feature=False, sample_seed=1, **kw):
        super().__init__(*args, **kw)
        self.use_sample_feature, self.sample_seed = use_sample_feature, sample_seed

    def _build_frame(self, gray, depth, flow, mask):
        F = super()._build_frame(gray, depth, flow, mask)
        if self.use_sample_feature:                           # Option II replaces the ORB-based static candidates; ORB still runs
            samp = sample_keypoints(self.h, self.w, self.sample_seed) if len(F.keys) else np.zeros((0, 2), f32)   # Frame.cc:97-98
            F.statKeysTmp, F.corres, F.flowNext, F.statDepthTmp = filter_sampled(samp, mask, depth, flow, self.th_bg)
            F.sampKeys = F.statKeysTmp.copy()
        return F

    def _track(self, C, L, depth, flow, mask):
        if not self.use_sample_feature:
            return super()._track(C, L, depth, flow, mask)
        # Inside _track, C.keys is read only as RenewFrameInfo's top-up source (mvKeysSample), which is the filtered sample list here
        orb_keys, C.keys = C.keys, C.sampKeys
        try:
            return super()._track(C, L, depth, flow, mask)
        finally:
            C.keys = orb_keys
