// orb_slam2_shim.hpp -- header-only C++17 mirror of the reference's classes on top of the C ABI (include/orbx.h).
//
// Same names, argument order and error behaviour as the reference, so that its call sites compile unchanged:
//   ORBExtractor(image, nFeatures, pyramidLevels, scaleFactor, bfTemFp, maxThreshold, minThreshold)
//       include/ORB_SLAM2/ORBExtractor.h:107     .extract(keyPoints, descriptors)            :110
//       .getPyramid() :113     ::getScaledFactors() :116     ::mnLevels / mnBorderSize / mfScaledFactor :158-160
//   Frame::createStereo(l, r, nFeatures, briefFp, maxThresh, minThresh, pVoc, nLevels, scale)   include/ORB_SLAM2/Frame.h:313
//   Frame::createRGBD(color, depth, nFeatures, briefFp, maxThresh, minThresh, pVoc, dScale, nLevels, scale)          :325
//   ORBMatcher::searchByStereo(FramePtr)                                                 include/ORB_SLAM2/ORBMatcher.h:39
//   Camera statics (include/ORB_SLAM2/Camera.h:23-32), exceptions (include/ORB_SLAM2/Error.h:13-98)
// It needs only the cv:: value types (cv::Mat, cv::KeyPoint): real OpenCV headers when available, otherwise any header
// providing them (this image has no C++ OpenCV; the tests compile against oracle/stub/opencv2/opencv.hpp).
// All compute happens in liborbx.so (CUDA); there is no CPU code path here.
#pragma once

#include <array>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#if __has_include(<opencv2/core.hpp>)
#include <opencv2/core.hpp>
#else
#include <opencv2/opencv.hpp>
#endif

#include "../orbx.h"

// OpenCV's type codes of 8-bit 3- and 4-channel images (CV_MAKETYPE(CV_8U, n)), for cv:: headers that leave them out
#ifndef CV_8UC3
#define CV_8UC3 16
#endif
#ifndef CV_8UC4
#define CV_8UC4 24
#endif

namespace ORB_SLAM2_ROS2_B200
{

// ---- include/ORB_SLAM2/Error.h ------------------------------------------------------------------------------------
class ORBSlam2Error : public std::runtime_error
{
public:
  explicit ORBSlam2Error(const std::string &what) : std::runtime_error(what) {}
};
class ImageSizeError : public ORBSlam2Error
{
  using ORBSlam2Error::ORBSlam2Error;
};
class FileNotOpenError : public ORBSlam2Error
{
  using ORBSlam2Error::ORBSlam2Error;
};
class DeviceError : public ORBSlam2Error
{
  using ORBSlam2Error::ORBSlam2Error;
};

namespace detail
{
inline void check(orbx_ctx *ctx, int rc, const char *what)
{
  if (rc == ORBX_OK) return;
  std::string msg = std::string(what) + ": " + orbx_status_string(rc);
  if (ctx && orbx_last_error(ctx)[0]) msg += std::string(" (") + orbx_last_error(ctx) + ")";
  if (rc == ORBX_ERR_IMAGE_SIZE) throw ImageSizeError(msg);
  if (rc == ORBX_ERR_FILE_NOT_OPEN) throw FileNotOpenError(msg);
  if (rc == ORBX_ERR_CUDA || rc == ORBX_ERR_NO_DEVICE) throw DeviceError(msg);
  throw ORBSlam2Error(msg);
}
} // namespace detail

// ---- include/ORB_SLAM2/Camera.h (set once, like System::setSetting does, src/System.cc:27-73) ---------------------
struct Camera
{
  static inline float mfBf = 0, mfBl = 0, mfFx = 0, mfFy = 0, mfCx = 0, mfCy = 0;
  static inline std::array<float, 5> mDistCoeff = {0, 0, 0, 0, 0}; // k1 k2 p1 p2 k3
  static void set(float fx, float fy, float cx, float cy, float bl, const std::array<float, 5> &dist = {0, 0, 0, 0, 0})
  {
    mfFx = fx;
    mfFy = fy;
    mfCx = cx;
    mfCy = cy;
    mfBl = bl;
    mfBf = mfFx * mfBl;
    mDistCoeff = dist;
  }
  // Camera.Color: colour frames (CV_8UC3 / CV_8UC4) arrive as RGB(A) when true, as BGR(A), OpenCV's order, when false.
  // Set next to set(); the shim converts them to gray on the device instead of Tracking::grabFrame's cvtColor
  // (src/Tracking.cc:55-68).
  static inline bool mbRGB = false;
};

// ---- one CUDA context per distinct configuration (the reference keeps these tables in process-wide statics) ----
namespace detail
{
// the ORBX_FORMAT_* of an image: CV_8UC1 gray, CV_8UC3 / CV_8UC4 colour in the order Camera::mbRGB names; other types throw
inline int input_format(const cv::Mat &img)
{
  if (img.type() == CV_8U) return ORBX_FORMAT_GRAY8;
  if (img.type() == CV_8UC3) return Camera::mbRGB ? ORBX_FORMAT_RGB8 : ORBX_FORMAT_BGR8;
  if (img.type() == CV_8UC4) return Camera::mbRGB ? ORBX_FORMAT_RGBA8 : ORBX_FORMAT_BGRA8;
  throw ORBSlam2Error("unsupported image type: expected CV_8UC1, CV_8UC3 or CV_8UC4");
}

struct CtxKey
{
  int w, h, nFeatures, nLevels, iniTh, minTh;
  float scale, fx, fy, cx, cy, bf, dScale;
  std::array<float, 5> dist;
  std::string tmpl;
  int format;
  auto tie() const { return std::tie(w, h, nFeatures, nLevels, iniTh, minTh, scale, fx, fy, cx, cy, bf, dScale, dist, tmpl, format); }
  bool operator<(const CtxKey &o) const { return tie() < o.tie(); }
};

// A context is not re-entrant (include/orbx.h): the cache hands every host thread its OWN context per configuration, so
// the reference's pattern of two extract() calls on two std::threads (src/Frame.cc:100-105) runs on two contexts, and
// every call into a context holds its mutex (a Frame may be queried from another thread than the one that made it).
struct Context
{
  orbx_ctx *raw = nullptr;
  std::mutex mu;
  explicit Context(orbx_ctx *c) : raw(c) {}
  Context(const Context &) = delete;
  Context &operator=(const Context &) = delete;
  ~Context() { orbx_destroy(raw); }
};
typedef std::shared_ptr<Context> ContextPtr;
typedef std::lock_guard<std::mutex> Lock;

inline ContextPtr context_for(int w, int h, int nFeatures, int nLevels, float scale, const std::string &tmpl, int iniTh, int minTh, float dScale,
                              int format = ORBX_FORMAT_GRAY8)
{
  static std::mutex mtx;
  static std::map<std::pair<CtxKey, std::thread::id>, ContextPtr> cache;
  CtxKey key{w, h, nFeatures, nLevels, iniTh, minTh, scale, Camera::mfFx, Camera::mfFy, Camera::mfCx, Camera::mfCy, Camera::mfBf, dScale, Camera::mDistCoeff, tmpl,
             format};
  const auto full = std::make_pair(key, std::this_thread::get_id());
  std::lock_guard<std::mutex> lock(mtx);
  auto it = cache.find(full);
  if (it != cache.end()) return it->second;
  std::vector<float> pattern(1024);
  check(nullptr, orbx_load_brief_template(tmpl.c_str(), pattern.data()), "BRIEF template"); // FileNotOpenError (:247-250)
  orbx_config cfg;
  orbx_default_config(&cfg);
  cfg.width = w;
  cfg.height = h;
  cfg.n_features = nFeatures;
  cfg.n_levels = nLevels;
  cfg.scale_factor = scale;
  cfg.ini_th_fast = iniTh;
  cfg.min_th_fast = minTh;
  cfg.fx = Camera::mfFx;
  cfg.fy = Camera::mfFy;
  cfg.cx = Camera::mfCx;
  cfg.cy = Camera::mfCy;
  cfg.bf = Camera::mfBf;
  for (int i = 0; i < 5; ++i) cfg.dist[i] = Camera::mDistCoeff[i];
  cfg.depth_scale = dScale;
  cfg.max_batch = 1;
  cfg.pattern = pattern.data();
  orbx_ctx *raw = nullptr;
  check(nullptr, orbx_create(&cfg, &raw), "orbx_create"); // ImageSizeError (:310-314)
  ContextPtr sp = std::make_shared<Context>(raw);
  check(raw, orbx_set_input_format(raw, format), "orbx_set_input_format");
  cache[full] = sp;
  return sp;
}

inline void to_cv(const std::vector<orbx_keypoint> &src, int n, std::vector<cv::KeyPoint> &dst)
{
  static_assert(sizeof(cv::KeyPoint) == sizeof(orbx_keypoint), "orbx_keypoint mirrors cv::KeyPoint");
  dst.resize((size_t)n);
  if (n) std::memcpy((void *)dst.data(), src.data(), (size_t)n * sizeof(orbx_keypoint));
}

// n rows of one contiguous N x 32 block, each a 1x32 CV_8U header sharing the block (vector<cv::Mat> for DBoW3)
inline void to_cv(const cv::Mat &block, int n, std::vector<cv::Mat> &dst)
{
  dst.clear();
  dst.reserve((size_t)n);
  for (int i = 0; i < n; ++i) dst.push_back(block.rowRange(i, i + 1));
}

inline std::vector<cv::Mat> fetch_pyramid(orbx_ctx *ctx, int side)
{
  std::vector<cv::Mat> pyr;
  const int nl = orbx_num_levels(ctx);
  for (int l = 0; l < nl; ++l)
  {
    int32_t w = 0, h = 0;
    check(ctx, orbx_level_info(ctx, l, &w, &h, nullptr, nullptr), "orbx_level_info");
    cv::Mat m(h, w, CV_8U);
    check(ctx, orbx_get_pyramid(ctx, side, l, 0, m.data, (size_t)m.step), "orbx_get_pyramid");
    pyr.push_back(m);
  }
  return pyr;
}
} // namespace detail

// ---- include/ORB_SLAM2/ORBExtractor.h:99-161 ------------------------------------------------------------------------
class ORBExtractor
{
public:
  typedef std::shared_ptr<ORBExtractor> SharedPtr;

  ORBExtractor(const cv::Mat &image, int nFeatures, int pyramidLevels, float scaleFactor, const std::string &bfTemFp, int maxThreshold, int minThreshold)
      : mImage(image), mnFeats(nFeatures), mnPyrLevels(pyramidLevels), mfScale(scaleFactor), mTmpl(bfTemFp), mIniTh(maxThreshold), mMinTh(minThreshold)
  {
    // FileNotOpenError / ImageSizeError surface here, as in the reference's constructor (src/ORBExtractor.cc:205-214)
    detail::ContextPtr ctx = context();
    // the reference keeps these as process-wide statics initialised by the first constructor (src/ORBExtractor.cc:283-302)
    mnLevels = pyramidLevels;
    mfScaledFactor = scaleFactor;
    std::vector<float> sf((size_t)pyramidLevels);
    for (int l = 0; l < pyramidLevels; ++l) detail::check(ctx->raw, orbx_level_info(ctx->raw, l, nullptr, nullptr, &sf[(size_t)l], nullptr), "orbx_level_info");
    static std::mutex sfm;
    detail::Lock lock(sfm);
    scaledFactors() = sf;
  }

  // Runs on the CALLING thread's context (two extractors of one configuration may extract concurrently on two threads).
  void extract(std::vector<cv::KeyPoint> &keyPoints, std::vector<cv::Mat> &descriptors)
  {
    detail::Lock self(mMu);
    run(&keyPoints, &descriptors);
    mvPyramids.clear(); // fetched on demand (getPyramid)
  }

  // The reference builds the pyramid in the constructor (src/ORBExtractor.cc:205-214), so it is valid from then on; here it is
  // produced by the same launches as the keypoints and copied back only when asked for.  If the context has moved on to
  // another image since extract() (or extract() was never called), the image is simply run again.
  const std::vector<cv::Mat> &getPyramid() const
  {
    detail::Lock self(mMu);
    if (!mvPyramids.empty()) return mvPyramids;
    bool fresh = false;
    if (mCtx)
    {
      detail::Lock lock(mCtx->mu);
      if (orbx_frame_epoch(mCtx->raw) == mEpoch)
      {
        mvPyramids = detail::fetch_pyramid(mCtx->raw, 0);
        fresh = true;
      }
    }
    if (!fresh)
    {
      const_cast<ORBExtractor *>(this)->run(nullptr, nullptr, true);
    }
    return mvPyramids;
  }
  static const std::vector<float> &getScaledFactors() { return scaledFactors(); }

  static inline int mnLevels = 0;
  static inline int mnBorderSize = 19;
  static inline float mfScaledFactor = 0.f;

private:
  static std::vector<float> &scaledFactors()
  {
    static std::vector<float> v;
    return v;
  }
  detail::ContextPtr context() const
  {
    return detail::context_for(mImage.cols, mImage.rows, mnFeats, mnPyrLevels, mfScale, mTmpl, mIniTh, mMinTh, 1.f, detail::input_format(mImage));
  }
  void run(std::vector<cv::KeyPoint> *keyPoints, std::vector<cv::Mat> *descriptors, bool want_pyramid = false)
  {
    mCtx = context();
    detail::Lock lock(mCtx->mu);
    std::vector<orbx_keypoint> k((size_t)mnFeats);
    mDescBlock = cv::Mat(mnFeats, 32, CV_8U);
    int32_t n = 0;
    detail::check(mCtx->raw, orbx_extract(mCtx->raw, mImage.data, (size_t)mImage.step, k.data(), mDescBlock.data, &n), "orbx_extract");
    mEpoch = orbx_frame_epoch(mCtx->raw);
    if (keyPoints) detail::to_cv(k, n, *keyPoints);
    if (descriptors) detail::to_cv(mDescBlock, n, *descriptors);
    if (want_pyramid) mvPyramids = detail::fetch_pyramid(mCtx->raw, 0);
  }
  cv::Mat mImage;
  int mnFeats, mnPyrLevels;
  float mfScale;
  std::string mTmpl;
  int mIniTh, mMinTh;
  mutable std::mutex mMu;
  mutable detail::ContextPtr mCtx; // the context the last extract() ran on
  mutable uint64_t mEpoch = 0;     // ... and its epoch right after it
  cv::Mat mDescBlock;
  mutable std::vector<cv::Mat> mvPyramids;
};

class ORBMatcher;

// ---- DBoW3::Vocabulary as the reference uses it (src/System.cc:93, include/ORB_SLAM2/Frame.h:224-231) ----------------
typedef std::map<unsigned, double> BowVector;                    // DBoW3::BowVector: WordId -> WordValue
typedef std::map<unsigned, std::vector<unsigned>> FeatureVector; // DBoW3::FeatureVector: NodeId -> feature indices
class Vocabulary
{
public:
  // text vocabulary (ORB-SLAM2's ORBvoc.txt layout); the tree lives on the device of the context for (width, height, ...)
  Vocabulary(const std::string &filename, detail::ContextPtr ctx) : mCtx(std::move(ctx))
  {
    detail::Lock lock(mCtx->mu);
    detail::check(mCtx->raw, orbx_vocab_load_text(mCtx->raw, filename.c_str(), &mVoc), "orbx_vocab_load_text");
  }
  ~Vocabulary() { orbx_vocab_destroy(mVoc); }
  Vocabulary(const Vocabulary &) = delete;
  Vocabulary &operator=(const Vocabulary &) = delete;
  unsigned size() const
  {
    int32_t words = 0;
    orbx_vocab_info(mVoc, nullptr, nullptr, nullptr, &words);
    return (unsigned)words;
  }
  const orbx_vocab *handle() const { return mVoc; }

private:
  detail::ContextPtr mCtx;
  orbx_vocab *mVoc = nullptr;
};

// ---- the hot-path part of include/ORB_SLAM2/Frame.h:303-371 --------------------------------------------------------
class Frame
{
  friend class ORBMatcher;

public:
  typedef std::shared_ptr<Frame> SharedPtr;

  static SharedPtr createStereo(cv::Mat leftImg, cv::Mat rightImg, int nFeatures, const std::string &briefFp, int maxThresh, int minThresh, void *pVoc,
                                int nLevels, float scale);
  static SharedPtr createRGBD(cv::Mat colorImg, cv::Mat depthImg, int nFeatures, const std::string &briefF, int maxThresh, int minThresh, void *pVoc,
                              float dScale, int nLevels, float scale)
  {
    (void)pVoc;
    SharedPtr f(new Frame());
    f->mCapacity = nFeatures;
    f->mLeftIm = colorImg;
    f->mCtx = detail::context_for(colorImg.cols, colorImg.rows, nFeatures, nLevels, scale, briefF, maxThresh, minThresh, dScale, detail::input_format(colorImg));
    if (depthImg.rows != colorImg.rows || depthImg.cols != colorImg.cols) throw ORBSlam2Error("createRGBD: depth image size differs from the colour image");
    if (depthImg.type() != CV_16U && depthImg.type() != CV_32F)
    { // any other depth type goes through the reference's own conversion (depthImg.convertTo(CV_32F), src/Frame.cc:130)
      cv::Mat asFloat;
      depthImg.convertTo(asFloat, CV_32F);
      depthImg = asFloat;
    }
    const int dtype = depthImg.type() == CV_32F ? ORBX_DEPTH_F32 : ORBX_DEPTH_U16;
    detail::Lock lock(f->mCtx->mu);
    std::vector<orbx_keypoint> kraw((size_t)nFeatures), kund((size_t)nFeatures);
    f->mDescLeft = cv::Mat(nFeatures, 32, CV_8U);
    std::vector<double> ur((size_t)nFeatures), dp((size_t)nFeatures);
    int32_t n = 0;
    detail::check(f->mCtx->raw,
                  orbx_rgbd_frame(f->mCtx->raw, colorImg.data, (size_t)colorImg.step, depthImg.data, (size_t)depthImg.step, dtype, kraw.data(), kund.data(),
                                  f->mDescLeft.data, &n, ur.data(), dp.data()),
                  "orbx_rgbd_frame");
    f->mEpoch = orbx_frame_epoch(f->mCtx->raw);
    detail::to_cv(kund, n, f->mvFeatsLeft);
    detail::to_cv(f->mDescLeft, n, f->mvLeftDescriptor);
    f->mvFeatsRightU.assign(ur.begin(), ur.begin() + n);
    f->mvDepths.assign(dp.begin(), dp.begin() + n);
    f->mnN = 0;
    for (double d : f->mvDepths) f->mnN += d > 0;
    return f;
  }

  const std::vector<cv::KeyPoint> &getLeftKeyPoints() const { return mvFeatsLeft; }
  const std::vector<cv::KeyPoint> &getRightKeyPoints() const { return mvFeatsRight; }
  const std::vector<cv::Mat> &getLeftDescriptor() const { return mvLeftDescriptor; }
  const std::vector<cv::Mat> &getRightDescriptor() const { return mRightDescriptor; }
  const std::vector<cv::Mat> &getDescriptor() const { return mvLeftDescriptor; }
  const std::vector<double> &getDepth() const { return mvDepths; }
  const std::vector<double> &getRightU() const { return mvFeatsRightU; }
  const cv::Mat &getLeftImage() const { return mLeftIm; }
  const cv::Mat &getRightImage() const { return mRightIm; }
  // VirtualFrame::mGrids (include/ORB_SLAM2/Frame.h:289, built by initGrid src/Frame.cc:53-69): [row][col] -> keypoint indices
  typedef std::vector<std::vector<std::vector<std::size_t>>> GridsType;
  GridsType getGrids() const
  {
    Resident here(*this, "getGrids");
    int32_t rows = 0, cols = 0;
    detail::check(mCtx->raw, orbx_grid_info(mCtx->raw, &rows, &cols, nullptr, nullptr, nullptr, nullptr), "orbx_grid_info");
    std::vector<int32_t> start((size_t)rows * cols + 1);
    std::vector<int32_t> all((size_t)orbx_capacity());
    detail::check(mCtx->raw, orbx_get_grid(mCtx->raw, 0, start.data(), all.data()), "orbx_get_grid");
    GridsType g((size_t)rows, std::vector<std::vector<std::size_t>>((size_t)cols));
    for (int r = 0; r < rows; ++r)
      for (int c = 0; c < cols; ++c)
        for (int i = start[(size_t)r * cols + c]; i < start[(size_t)r * cols + c + 1]; ++i) g[(size_t)r][(size_t)c].push_back((std::size_t)all[(size_t)i]);
    return g;
  }
  // orbslam2.KeyFrameData bytes for a keyframe made from this frame (KeyFrame::serializeToProtobuf, src/KeyFrame.cc:553-647;
  // proto/Keyframe.proto:45-64), assembled on the device.  The frame must be the context's most recent one.
  std::string serializeKeyFrameData(uint64_t id, const float *poseRt /* R row-major [9] + t [3], or nullptr */ = nullptr, bool withMapPoints = true) const
  {
    Resident here(*this, "serializeKeyFrameData");
    std::string out((size_t)orbx_serialized_capacity(mCtx->raw), '\0');
    int64_t n = 0;
    detail::check(mCtx->raw, orbx_serialize_keyframe(mCtx->raw, 0, id, poseRt, withMapPoints ? 1 : 0, (uint8_t *)&out[0], out.size(), &n),
                  "orbx_serialize_keyframe");
    out.resize((size_t)n);
    return out;
  }
  // VirtualFrame::computeBow (include/ORB_SLAM2/Frame.h:224-231): mpVoc->transform(mvLeftDescriptor, mBowVec, mFeatVec, 4)
  void computeBow(const Vocabulary &voc, BowVector &bowVec, FeatureVector &featVec, int levelsup = 4) const
  {
    Resident here(*this, "computeBow");
    const std::size_t N = (std::size_t)orbx_capacity();
    std::vector<int32_t> ids(N), nodes(N), start(N + 1), feats(N);
    std::vector<double> vals(N);
    int32_t nb = 0, nf = 0;
    detail::check(mCtx->raw,
                  orbx_bow_transform(mCtx->raw, voc.handle(), 0, levelsup, ids.data(), vals.data(), &nb, nodes.data(), start.data(), feats.data(), &nf),
                  "orbx_bow_transform");
    bowVec.clear();
    featVec.clear();
    for (int i = 0; i < nb; ++i) bowVec.emplace_hint(bowVec.end(), (unsigned)ids[(std::size_t)i], vals[(std::size_t)i]);
    for (int j = 0; j < nf; ++j)
      featVec.emplace_hint(featVec.end(), (unsigned)nodes[(std::size_t)j],
                           std::vector<unsigned>(feats.begin() + start[(std::size_t)j], feats.begin() + start[(std::size_t)j + 1]));
  }
  detail::ContextPtr context() const { return mCtx; }
  std::vector<cv::Mat> getLeftPyramid() const
  {
    Resident here(*this, "getLeftPyramid");
    return detail::fetch_pyramid(mCtx->raw, 0);
  }
  std::vector<cv::Mat> getRightPyramid() const
  {
    Resident here(*this, "getRightPyramid");
    return detail::fetch_pyramid(mCtx->raw, 1);
  }
  int getN() const { return mnN; }

private:
  Frame() = default;
  int orbx_capacity() const { return mCapacity; }
  int mCapacity = 0; // nFeatures of the context: size of the fixed-stride result arrays
  std::vector<cv::KeyPoint> mvFeatsLeft, mvFeatsRight;
  std::vector<cv::Mat> mvLeftDescriptor, mRightDescriptor;
  std::vector<double> mvDepths, mvFeatsRightU;
  std::vector<double> mStereoU, mStereoDepth; // computed with the frame, published by ORBMatcher::searchByStereo
  int mStereoMatches = 0;
  int mnN = 0;
  cv::Mat mLeftIm, mRightIm, mDescLeft, mDescRight;
  detail::ContextPtr mCtx;
  uint64_t mEpoch = 0; // the context's epoch right after this frame was made: device-side queries need it unchanged

  // Holds the frame's context for one query and checks that the frame is still the one resident on it: the context keeps the
  // device state (pyramids, grid, descriptors) of its MOST RECENT frame only, so a query on an older Frame must not silently
  // answer with the newer frame's data.
  struct Resident
  {
    detail::Lock lock;
    Resident(const Frame &f, const char *what) : lock(f.mCtx->mu)
    {
      if (orbx_frame_epoch(f.mCtx->raw) != f.mEpoch)
        throw ORBSlam2Error(std::string(what) + ": this Frame is no longer resident on its device context (a newer frame was created on the same thread and "
                                                "configuration); query a frame before creating the next one");
    }
  };
};

// ---- the stereo entry (include/ORB_SLAM2/ORBMatcher.h:39) and the projection matchers (:50-53) ---------------------------------------------------------
class ORBMatcher
{
public:
  typedef std::shared_ptr<ORBMatcher> SharedPtr;
  explicit ORBMatcher(float ratio = 0.6f, bool checkOri = true) : mfRatio(ratio), mbCheckOri(checkOri) {}
  // fills mvFeatsRightU / mvDepths (-1 = no match) and returns the match count, like src/ORBMatcher.cc:18-81.  The GPU
  // computed them together with the features (one launch sequence per frame); this call publishes them.
  int searchByStereo(Frame::SharedPtr pFrame)
  {
    pFrame->mvFeatsRightU = pFrame->mStereoU;
    pFrame->mvDepths = pFrame->mStereoDepth;
    return pFrame->mStereoMatches;
  }

  // ---- tracking-side matchers (include/ORB_SLAM2/ORBMatcher.h:50-53,105) -------------------------------------------
  // The reference walks MapPoint objects; here the caller passes what it derives from them as per-keypoint masks.  The
  // frame searched must be the one most recently created on its context (its keypoints, descriptors and grid are still
  // resident on the device).
  struct AreaMatch
  {
    int idx = -1;   // best candidate among the frame's left keypoints, -1 = no candidate
    int distance = 0;
    float ratio = 0.f;
    int nCandidates = 0;
  };

  // findFeaturesInArea + exclusion + getBestMatch for every query (src/Frame.cc:286-311, src/ORBMatcher.cc:322-331,967-990):
  // kps[i].pt / kps[i].octave, radius[i] (before the sf^2 scaling), candidate octaves in [minLevel[i], maxLevel[i]]
  static std::vector<AreaMatch> searchInArea(Frame::SharedPtr pFrame, const std::vector<cv::KeyPoint> &kps, const std::vector<float> &radius,
                                             const std::vector<int> &minLevel, const std::vector<int> &maxLevel, const std::vector<cv::Mat> &descs,
                                             const std::vector<bool> *exclude = nullptr)
  {
    const std::size_t n = kps.size();
    std::vector<orbx_area_query> q(n);
    std::vector<uint8_t> qd(n * 32), ex;
    for (std::size_t i = 0; i < n; ++i)
    {
      q[i] = orbx_area_query{kps[i].pt.x, kps[i].pt.y, radius[i], kps[i].octave, minLevel[i], maxLevel[i]};
      std::memcpy(&qd[32 * i], descs[i].data, 32);
    }
    if (exclude)
    {
      ex.assign((std::size_t)pFrame->orbx_capacity(), 0);
      for (std::size_t i = 0; i < exclude->size() && i < ex.size(); ++i) ex[i] = (*exclude)[i] ? 1 : 0;
    }
    std::vector<int32_t> idx(n), dist(n), nc(n);
    std::vector<float> ratio(n);
    Frame::Resident here(*pFrame, "searchInArea");
    detail::check(pFrame->mCtx->raw,
                  orbx_search_in_area(pFrame->mCtx->raw, 0, (int)n, q.data(), qd.data(), exclude ? ex.data() : nullptr, idx.data(), dist.data(), ratio.data(),
                                      nc.data()),
                  "orbx_search_in_area");
    std::vector<AreaMatch> out(n);
    for (std::size_t i = 0; i < n; ++i) out[i] = AreaMatch{idx[i], dist[i], ratio[i], nc[i]};
    return out;
  }

  // searchByProjection(pFrame1, pFrame2, matches, th, bFuse) (src/ORBMatcher.cc:265-347).  kps2 / desc2 = pFrame2's left
  // keypoints and descriptors; valid2[idx] = mps2[idx] is a good map point (and, for bFuse, in view of pFrame1);
  // hasMp1[i] = pFrame1's keypoint i already has a good map point; tlcZ = z of pFrame1's camera centre in pFrame2's
  // camera frame (:275-281, compared with Camera::mfBl).
  int searchByProjection(Frame::SharedPtr pFrame1, const std::vector<cv::KeyPoint> &kps2, const std::vector<cv::Mat> &desc2, const std::vector<bool> &valid2,
                         const std::vector<bool> &hasMp1, std::vector<cv::DMatch> &matches, float th, float tlcZ = 0.f, bool bFuse = false)
  {
    matches.clear();
    bool up = false, down = false;
    if (std::abs(tlcZ) > Camera::mfBl) tlcZ > 0 ? up = true : down = true;
    std::vector<cv::KeyPoint> q;
    std::vector<cv::Mat> qd;
    std::vector<float> radius;
    std::vector<int> lo, hi, src;
    for (std::size_t idx = 0; idx < kps2.size(); ++idx)
    {
      if (!valid2[idx]) continue;
      const int o = kps2[idx].octave;
      q.push_back(kps2[idx]);
      qd.push_back(desc2[idx]);
      radius.push_back(th);
      lo.push_back(up ? o : down ? 0 : std::max(0, o - 1));
      hi.push_back(up ? 7 : down ? o : std::min(o + 1, 7));
      src.push_back((int)idx);
    }
    std::vector<AreaMatch> r = searchInArea(pFrame1, q, radius, lo, hi, qd, bFuse ? nullptr : &hasMp1);
    for (std::size_t i = 0; i < r.size(); ++i)
      if (r[i].nCandidates > 0 && r[i].ratio < mfRatio && r[i].distance < mnMinThreshold) matches.emplace_back(r[i].idx, src[i], (float)r[i].distance);
    return (int)matches.size();
  }

  // searchByBow(pFrame, pKframe, matches, bAddMPs, bLoop) (src/ORBMatcher.cc:170-255).  The keyframe is given by its left
  // keypoints / descriptors and its FeatureVector (from Frame::computeBow when it was the current frame); kfGood[i] /
  // frameGood[i] = "the feature has a good map point" (for bAddMPs: "... that is in the map").  pFrame must be the
  // context's most recent frame; its BoW is computed here like pFrame->computeBow() (:172).
  int searchByBow(Frame::SharedPtr pFrame, const Vocabulary &voc, const std::vector<cv::KeyPoint> &kfKeyPoints, const std::vector<cv::Mat> &kfDescriptors,
                  const FeatureVector &kfFeatVec, const std::vector<bool> &kfGood, const std::vector<bool> &frameGood, std::vector<cv::DMatch> &matches,
                  bool bAddMPs = false, bool bLoop = false, int levelsup = 4)
  {
    matches.clear();
    BowVector bv;
    FeatureVector fv;
    pFrame->computeBow(voc, bv, fv, levelsup);
    std::vector<int32_t> nodes, start(1, 0), feats;
    for (auto &kv : kfFeatVec)
    {
      nodes.push_back((int32_t)kv.first);
      for (unsigned i : kv.second) feats.push_back((int32_t)i);
      start.push_back((int32_t)feats.size());
    }
    const std::size_t nk = kfDescriptors.size(), N = (std::size_t)pFrame->orbx_capacity(), nl = feats.size();
    std::vector<uint8_t> kd(nk * 32), qok(nk, 0), cok(N, 0);
    for (std::size_t i = 0; i < nk; ++i)
    {
      std::memcpy(&kd[32 * i], kfDescriptors[i].data, 32);
      const bool g = i < kfGood.size() && kfGood[i];
      qok[i] = bAddMPs ? !g : (bLoop ? 1 : g); // :195-212
    }
    for (std::size_t i = 0; i < N; ++i)
    {
      const bool g = i < frameGood.size() && frameGood[i];
      cok[i] = bLoop ? 1 : !g; // :216-233 (bAddMPs and the default mode both want frame features without a map point)
    }
    std::vector<int32_t> idx(nl), dist(nl), nc(nl);
    std::vector<float> ratio(nl);
    {
      Frame::Resident here(*pFrame, "searchByBow");
      detail::check(pFrame->mCtx->raw,
                  orbx_search_by_bow(pFrame->mCtx->raw, 0, (int)nodes.size(), nodes.data(), start.data(), feats.data(), kd.data(), (int)nk, qok.data(),
                                     cok.data(), idx.data(), dist.data(), ratio.data(), nc.data()),
                  "orbx_search_by_bow");
    }
    for (std::size_t e = 0; e < nl; ++e)
      if (nc[e] > 0 && !(dist[e] > mnMinThreshold || ratio[e] > mfRatio)) matches.emplace_back(idx[e], feats[e], (float)dist[e]); // :240-245
    if (mbCheckOri) verifyAngle(pFrame, matches, pFrame->getLeftKeyPoints(), kfKeyPoints);
    return (int)matches.size();
  }

  // ORBMatcher::verifyAngle (src/ORBMatcher.cc:1013-1051); `owner` provides the device context
  static void verifyAngle(Frame::SharedPtr owner, std::vector<cv::DMatch> &matches, const std::vector<cv::KeyPoint> &keyPoints1,
                          const std::vector<cv::KeyPoint> &keyPoints2)
  {
    const std::size_t n = matches.size();
    std::vector<int32_t> qi(n), ti(n);
    std::vector<float> di(n);
    for (std::size_t i = 0; i < n; ++i) qi[i] = matches[i].queryIdx, ti[i] = matches[i].trainIdx, di[i] = matches[i].distance;
    std::vector<orbx_keypoint> k1(keyPoints1.size()), k2(keyPoints2.size());
    if (!k1.empty()) std::memcpy(k1.data(), keyPoints1.data(), k1.size() * sizeof(orbx_keypoint));
    if (!k2.empty()) std::memcpy(k2.data(), keyPoints2.data(), k2.size() * sizeof(orbx_keypoint));
    int32_t m = 0;
    detail::Lock lock(owner->mCtx->mu);
    detail::check(owner->mCtx->raw,
                  orbx_verify_angle(owner->mCtx->raw, (int)n, qi.data(), ti.data(), di.data(), k1.data(), (int)k1.size(), k2.data(), (int)k2.size(), &m),
                  "orbx_verify_angle");
    matches.resize((std::size_t)m);
    for (int i = 0; i < m; ++i) matches[(std::size_t)i] = cv::DMatch(qi[(std::size_t)i], ti[(std::size_t)i], di[(std::size_t)i]);
  }

  static inline int mnMaxThreshold = 100, mnMinThreshold = 50, mnMeanThreshold = 75; // src/ORBMatcher.cc:1086-1088
  static inline int mnBinNum = 30, mnBinChoose = 3;                                  // :1091-1092

private:
  float mfRatio = 0.6f;
  bool mbCheckOri = true;
};

inline Frame::SharedPtr Frame::createStereo(cv::Mat leftImg, cv::Mat rightImg, int nFeatures, const std::string &briefFp, int maxThresh, int minThresh,
                                            void *pVoc, int nLevels, float scale)
{
  (void)pVoc;
  SharedPtr f(new Frame());
  f->mCapacity = nFeatures;
  f->mLeftIm = leftImg;
  f->mRightIm = rightImg;
  const int format = detail::input_format(leftImg);
  if (detail::input_format(rightImg) != format) throw ORBSlam2Error("createStereo: the right image's type differs from the left one's");
  f->mCtx = detail::context_for(leftImg.cols, leftImg.rows, nFeatures, nLevels, scale, briefFp, maxThresh, minThresh, 1.f, format);
  std::vector<orbx_keypoint> kl((size_t)nFeatures), kr((size_t)nFeatures);
  f->mDescLeft = cv::Mat(nFeatures, 32, CV_8U);
  f->mDescRight = cv::Mat(nFeatures, 32, CV_8U);
  f->mStereoU.resize((size_t)nFeatures);
  f->mStereoDepth.resize((size_t)nFeatures);
  int32_t nl = 0, nr = 0, nm = 0;
  {
    detail::Lock lock(f->mCtx->mu);
    detail::check(f->mCtx->raw,
                orbx_stereo_frame(f->mCtx->raw, leftImg.data, (size_t)leftImg.step, rightImg.data, (size_t)rightImg.step, kl.data(), f->mDescLeft.data, &nl,
                                  kr.data(), f->mDescRight.data, &nr, f->mStereoU.data(), f->mStereoDepth.data(), &nm),
                "orbx_stereo_frame");
    f->mEpoch = orbx_frame_epoch(f->mCtx->raw);
  }
  detail::to_cv(kl, nl, f->mvFeatsLeft);
  detail::to_cv(kr, nr, f->mvFeatsRight);
  detail::to_cv(f->mDescLeft, nl, f->mvLeftDescriptor);
  detail::to_cv(f->mDescRight, nr, f->mRightDescriptor);
  f->mStereoU.resize((size_t)nl);
  f->mStereoDepth.resize((size_t)nl);
  f->mStereoMatches = nm;
  ORBMatcher::SharedPtr mpMatcher = std::make_shared<ORBMatcher>(); // Frame.h:317-319
  f->mnN = mpMatcher->searchByStereo(f);
  return f;
}

} // namespace ORB_SLAM2_ROS2_B200
