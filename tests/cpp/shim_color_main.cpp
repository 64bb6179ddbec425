// Drives the C++ shim with colour frames (CV_8UC3 / CV_8UC4, order from Camera::mbRGB) the way Tracking::grabFrame hands
// them over once its cvtColor is gone, and dumps the results for comparison with gray calls on cv2.cvtColor's output.
//   shim_color_main types
//   shim_color_main stereo <w> <h> <nFeatures> <nLevels> <scale> <template> <left.raw> <right.raw> <out.bin> <channels> <rgb>
//   shim_color_main rgbd   <w> <h> <nFeatures> <nLevels> <scale> <template> <color.raw> <depth_u16.raw> <out.bin> <channels> <rgb> <dScale>
// Colour images are headers over the driver's own buffers with an explicit row step (w * channels bytes).
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <vector>

#include <orbx/orb_slam2_shim.hpp>

using namespace ORB_SLAM2_ROS2_B200;

static std::vector<uchar> read_bytes(const char *path, size_t n)
{
  std::vector<uchar> b(n);
  std::ifstream f(path, std::ios::binary);
  f.read((char *)b.data(), (std::streamsize)n);
  if (!f) throw std::runtime_error(std::string("cannot read ") + path);
  return b;
}

template <typename T> static void put(std::ofstream &o, const T &v) { o.write((const char *)&v, sizeof(T)); }

static void dump(std::ofstream &o, const std::vector<cv::KeyPoint> &k, const std::vector<cv::Mat> &d)
{
  put(o, (int32_t)k.size());
  for (auto &kp : k) o.write((const char *)&kp, sizeof(cv::KeyPoint));
  for (auto &m : d) o.write((const char *)m.data, 32);
}

int main(int argc, char **argv)
{
  try
  {
    std::string mode = argv[1];
    if (mode == "types")
    { // image types other than CV_8UC1 / 3 / 4 are refused before any device work
      int ok = 0;
      uchar buf[64 * 48 * 4] = {};
      for (int type : {CV_16U, CV_32F})
        try
        {
          ORBExtractor ex(cv::Mat(48, 64, type, buf, 64 * 4), 500, 4, 1.2f, "/nonexistent/brief_template.txt", 20, 7);
        }
        catch (const FileNotOpenError &)
        {
        }
        catch (const ORBSlam2Error &)
        {
          ++ok;
        }
      std::printf("types ok=%d\n", ok);
      return ok == 2 ? 0 : 1;
    }
    if (argc < 13) throw std::runtime_error("missing arguments");
    const int w = atoi(argv[2]), h = atoi(argv[3]), nf = atoi(argv[4]), nl = atoi(argv[5]);
    const float scale = (float)atof(argv[6]);
    const std::string tmpl = argv[7];
    std::ofstream out(argv[10], std::ios::binary);
    const int ch = atoi(argv[11]);
    const int type = ch == 4 ? CV_8UC4 : CV_8UC3;
    Camera::mbRGB = atoi(argv[12]) != 0;
    const size_t step = (size_t)w * ch;
    if (mode == "stereo")
    {
      Camera::set(718.856f, 718.856f, 607.1928f, 185.2157f, 0.537166f);
      std::vector<uchar> lb = read_bytes(argv[8], step * h), rb = read_bytes(argv[9], step * h);
      cv::Mat l(h, w, type, lb.data(), step), r(h, w, type, rb.data(), step);
      ORBExtractor ex(l, nf, nl, scale, tmpl, 20, 7);
      std::vector<cv::KeyPoint> k;
      std::vector<cv::Mat> d;
      ex.extract(k, d);
      dump(out, k, d);
      const cv::Mat &l0 = ex.getPyramid()[0]; // level 0 is the converted gray image
      for (int y = 0; y < l0.rows; ++y) out.write((const char *)l0.ptr<uchar>(y), l0.cols);
      Frame::SharedPtr f = Frame::createStereo(l, r, nf, tmpl, 20, 7, nullptr, nl, scale);
      dump(out, f->getLeftKeyPoints(), f->getLeftDescriptor());
      dump(out, f->getRightKeyPoints(), f->getRightDescriptor());
      put(out, (int32_t)f->getN());
      for (double v : f->getRightU()) put(out, v);
      for (double v : f->getDepth()) put(out, v);
    }
    else if (mode == "rgbd")
    {
      Camera::set(520.908620f, 521.007327f, 325.141442f, 249.701764f, 0.0767889f, {0.231222f, -0.784899f, -0.003257f, -0.000105f, 0.917205f});
      std::vector<uchar> cb = read_bytes(argv[8], step * h), db = read_bytes(argv[9], (size_t)w * h * 2);
      cv::Mat c(h, w, type, cb.data(), step), dep(h, w, CV_16U, db.data(), (size_t)w * 2);
      Frame::SharedPtr f = Frame::createRGBD(c, dep, nf, tmpl, 20, 7, nullptr, (float)atof(argv[13]), nl, scale);
      dump(out, f->getLeftKeyPoints(), f->getLeftDescriptor());
      put(out, (int32_t)f->getN());
      for (double v : f->getRightU()) put(out, v);
      for (double v : f->getDepth()) put(out, v);
    }
    return 0;
  }
  catch (const std::exception &e)
  {
    std::fprintf(stderr, "shim_color_main: %s\n", e.what());
    return 2;
  }
}
