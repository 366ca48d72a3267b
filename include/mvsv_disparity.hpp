// mvsv_disparity.hpp -- C++ host-side mirror of the reference's disparity interface on top of the C ABI (mvsv.h).
//
// Same names, argument meaning and error behaviour as reference inc/disparity.h:15-36 / src/disparity.cpp:6-22,60-108
// and struct Stereopair (inc/utility.h:31-41), so that a driver such as trgt/demo.cpp compiles against it after
// replacing  cv::Ptr<cv::StereoSGBM>  by  mvsv::Matcher  (see INTEGRATION.md).  Header-only; needs only libmvsv.so.
//
// With -DMVSV_WITH_OPENCV the image type is cv::Mat; without OpenCV (this build image has no OpenCV C++ headers) a
// minimal Mat with the same fields the path touches (rows, cols, step, data, type) is used.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

#include "mvsv.h"

#ifdef MVSV_WITH_OPENCV
#include <opencv2/core.hpp>
namespace mvsv { using Mat = cv::Mat; }
#else
namespace mvsv {
enum { MVSV_8UC1 = 0, MVSV_16SC1 = 3 };   // numerically equal to CV_8UC1 / CV_16SC1
// Minimal stand-in for cv::Mat: row-major, `step` bytes per row, optionally a view into someone else's memory
// (ROI views with step > cols are what Stereosystem::getRectifiedImagepair hands out, src/Stereosystem.cpp:255-256).
struct Mat {
    int rows = 0, cols = 0, mtype = MVSV_8UC1;
    size_t step = 0;
    unsigned char* data = nullptr;
    std::shared_ptr<std::vector<unsigned char>> owner;

    Mat() {}
    Mat(int r, int c, int t) { create(r, c, t); }
    Mat(int r, int c, int t, void* ext, size_t ext_step) : rows(r), cols(c), mtype(t), step(ext_step), data((unsigned char*)ext) {}
    int type() const { return mtype; }
    size_t elemSize() const { return mtype == MVSV_16SC1 ? 2 : 1; }
    bool empty() const { return data == nullptr || rows == 0 || cols == 0; }
    void create(int r, int c, int t)
    {
        if (r == rows && c == cols && t == mtype && data) return;
        rows = r; cols = c; mtype = t; step = (size_t)c * elemSize();
        owner = std::make_shared<std::vector<unsigned char>>((size_t)r * step);
        data = owner->data();
    }
    template <class T> T& at(int r, int c) { return *reinterpret_cast<T*>(data + (size_t)r * step + (size_t)c * sizeof(T)); }
    template <class T> const T& at(int r, int c) const { return *reinterpret_cast<const T*>(data + (size_t)r * step + (size_t)c * sizeof(T)); }
    // ROI view, like cv::Mat::operator()(cv::Rect)
    Mat roi(int x, int y, int w, int h) const
    {
        Mat m; m.rows = h; m.cols = w; m.mtype = mtype; m.step = step; m.owner = owner;
        m.data = data + (size_t)y * step + (size_t)x * elemSize();
        return m;
    }
};
}  // namespace mvsv
#endif

// reference inc/utility.h:31-41
struct Stereopair {
    Stereopair() {}
    Stereopair(mvsv::Mat& l, mvsv::Mat& r) : mLeft(l), mRight(r) {}
    mvsv::Mat mLeft, mRight;
};

namespace mvsv {

// Owns one mvsv_ctx.  Stands where the reference holds cv::Ptr<cv::StereoSGBM> / cv::Ptr<cv::StereoBM>
// (trgt/demo.cpp:37,190-194).  The ctx is (re)created lazily for the size of the first pair it sees.
class Matcher {
public:
    explicit Matcher(int device = 0) : device_(device) {}
    ~Matcher() { mvsv_destroy(ctx_); }
    Matcher(const Matcher&) = delete;
    Matcher& operator=(const Matcher&) = delete;

    void setSgbm(const mvsv_sgbm_params& p) { sg_ = p; have_sg_ = true; if (ctx_) applied_ = (mvsv_set_sgbm_params(ctx_, &sg_) == MVSV_OK); }
    void setBm(const mvsv_bm_params& p) { bm_ = p; have_bm_ = true; if (ctx_) applied_bm_ = applyBm() == MVSV_OK; }
    // cv::StereoBM::setDisp12MaxDiff / setSpeckleWindowSize / setSpeckleRange (mvsv_set_bm_filters); default -1 / 0 / 0
    void setBmFilters(int disp12MaxDiff, int speckleWindowSize, int speckleRange)
    {
        bmf_[0] = disp12MaxDiff; bmf_[1] = speckleWindowSize; bmf_[2] = speckleRange;
        if (ctx_ && have_bm_) applied_bm_ = applyBm() == MVSV_OK;
    }
    const char* lastError() const { return err_.empty() ? mvsv_last_error(ctx_) : err_.c_str(); }
    mvsv_ctx* ctx() { return ctx_; }

    // returns MVSV_OK or an error code; cv::StereoMatcher::compute would throw cv::Exception instead
    int compute(const Mat& left, const Mat& right, Mat& out, unsigned stage)
    {
        err_.clear();
        if (left.empty() || right.empty() || left.rows != right.rows || left.cols != right.cols ||
            left.elemSize() != 1 || right.elemSize() != 1) { err_ = "compute: need two equal-size CV_8UC1 images"; return MVSV_ERR_INVALID; }
        if (!ctx_ || w_ != left.cols || h_ != left.rows) {
            mvsv_destroy(ctx_); ctx_ = nullptr;
            int rc = mvsv_init(device_, left.cols, left.rows, 1, &ctx_);
            if (rc != MVSV_OK) { err_ = mvsv_last_error(nullptr); return rc; }
            w_ = left.cols; h_ = left.rows; applied_ = applied_bm_ = false;
        }
        int rc;
        if (stage == MVSV_STAGE_SGBM && !applied_) {
            if (!have_sg_) { mvsv_sgbm_params z; std::memset(&z, 0, sizeof z); sg_ = z; }   // StereoSGBM::create(0,0,0,...) as trgt/demo.cpp:190
            if ((rc = mvsv_set_sgbm_params(ctx_, &sg_)) != MVSV_OK) return rc;
            applied_ = true;
        }
        if (stage == MVSV_STAGE_BM && !applied_bm_) {
            if (!have_bm_) { err_ = "BM parameters not set"; return MVSV_ERR_STATE; }
            if ((rc = applyBm()) != MVSV_OK) return rc;
            applied_bm_ = true;
        }
        if ((rc = mvsv_compute(ctx_, left.data, left.step, right.data, right.step, 0, 1, stage)) != MVSV_OK) return rc;
#ifdef MVSV_WITH_OPENCV
        out.create(left.rows, left.cols, CV_16SC1);
#else
        out.create(left.rows, left.cols, MVSV_16SC1);
#endif
        return mvsv_download(ctx_, reinterpret_cast<int16_t*>(out.data), out.step, nullptr, nullptr, 0, nullptr, nullptr);
    }

    // Disparity::tm (reference src/disparity.cpp:25-58)
    int computeTm(const Mat& left, const Mat& right, Mat& out, unsigned kernelSize)
    {
        err_.clear();
        if (left.empty() || right.empty() || left.rows != right.rows || left.cols != right.cols ||
            left.elemSize() != 1 || right.elemSize() != 1) { err_ = "tm: need two equal-size CV_8UC1 images"; return MVSV_ERR_INVALID; }
        if (!ctx_ || w_ != left.cols || h_ != left.rows) {
            mvsv_destroy(ctx_); ctx_ = nullptr;
            int rc = mvsv_init(device_, left.cols, left.rows, 1, &ctx_);
            if (rc != MVSV_OK) { err_ = mvsv_last_error(nullptr); return rc; }
            w_ = left.cols; h_ = left.rows; applied_ = applied_bm_ = false;
        }
#ifdef MVSV_WITH_OPENCV
        out.create(left.rows, left.cols, CV_8UC1);
#else
        out.create(left.rows, left.cols, MVSV_8UC1);
#endif
        return mvsv_tm(ctx_, left.data, left.step, right.data, right.step, 0, 1, kernelSize, out.data, out.step);
    }

private:
    int applyBm()
    {
        const int rc = mvsv_set_bm_params(ctx_, &bm_);
        return rc != MVSV_OK ? rc : mvsv_set_bm_filters(ctx_, bmf_[0], bmf_[1], bmf_[2]);
    }

    int device_;
    mvsv_ctx* ctx_ = nullptr;
    int w_ = 0, h_ = 0;
    mvsv_sgbm_params sg_{};
    mvsv_bm_params bm_{};
    int bmf_[3] = {-1, 0, 0};
    bool have_sg_ = false, have_bm_ = false, applied_ = false, applied_bm_ = false;
    std::string err_;
};

// '%YAML:1.0' flat `key: number` reader standing in for cv::FileStorage on the reference's configs/*.yml
inline bool readFlatYaml(const std::string& filename, std::map<std::string, double>& kv)
{
    std::ifstream f(filename.c_str());
    if (!f.is_open()) return false;
    std::string line;
    while (std::getline(f, line)) {
        const size_t h = line.find('#');
        if (h != std::string::npos) line.erase(h);
        if (line.empty() || line[0] == '%' || line.compare(0, 3, "---") == 0) continue;
        const size_t c = line.find(':');
        if (c == std::string::npos) continue;
        std::string k = line.substr(0, c), v = line.substr(c + 1);
        auto trim = [](std::string& s) { const size_t a = s.find_first_not_of(" \t\r"); const size_t b = s.find_last_not_of(" \t\r"); s = a == std::string::npos ? "" : s.substr(a, b - a + 1); };
        trim(k); trim(v);
        char* end = nullptr;
        const double d = std::strtod(v.c_str(), &end);
        if (end != v.c_str()) kv[k] = d;
    }
    return true;
}

}  // namespace mvsv

namespace Disparity {

// reference inc/disparity.h:17-27
struct sgbmParameters {
    int minDisp, numDisp, blockSize, disp12MaxDiff, preFilterCap, uniquenessRatio, speckleWindowSize, speckleRange, disparityMode;
};

// reference src/disparity.cpp:6-10: dispCompute->compute(mLeft, mRight, output).  `void` like the reference; a
// failure (OpenCV would throw) leaves `output` untouched and is readable through Matcher::lastError().
inline void sgbm(Stereopair const& inputImages, mvsv::Mat& output, mvsv::Matcher& dispCompute)
{
    dispCompute.compute(inputImages.mLeft, inputImages.mRight, output, MVSV_STAGE_SGBM);
}

// reference src/disparity.cpp:18-22
inline void bm(Stereopair const& inputImages, mvsv::Mat& output, mvsv::Matcher& dispCompute)
{
    dispCompute.compute(inputImages.mLeft, inputImages.mRight, output, MVSV_STAGE_BM);
}

// reference src/disparity.cpp:25-58 (inc/disparity.h:33): the "self written template matching"; the reference has
// no matcher object here, the engine handle takes its place as the last argument
inline void tm(Stereopair const& inputImages, mvsv::Mat& output, unsigned int kernelSize, mvsv::Matcher& engine)
{
    engine.computeTm(inputImages.mLeft, inputImages.mRight, output, kernelSize);
}

// reference src/disparity.cpp:60-108: reads the nine keys, drives the eight setters + mode; never sets P1/P2.
inline bool loadSGBMParameters(std::string const filename, mvsv::Matcher& disparityObj, sgbmParameters& para)
{
    std::map<std::string, double> fs;
    if (!mvsv::readFlatYaml(filename, fs)) {
        std::fprintf(stderr, "Unable to open disparity parameters\n");
        return false;
    }
    if (!fs.count("numDisp") || !fs.count("blockSize") || !fs.count("speckleWindowSize") || !fs.count("speckleWindowRange")) {
        std::fprintf(stderr, "Node in %s is empty\n", filename.c_str());
        return false;
    }
    auto geti = [&](const char* k) { auto it = fs.find(k); return it == fs.end() ? 0 : (int)it->second; };   // missing FileNode >> int gives 0
    para.minDisp = geti("minDisp"); para.numDisp = geti("numDisp"); para.blockSize = geti("blockSize");
    para.disp12MaxDiff = geti("disp12MaxDiff"); para.preFilterCap = geti("preFilterCap");
    para.uniquenessRatio = geti("uniquenessRatio"); para.speckleWindowSize = geti("speckleWindowSize");
    para.speckleRange = geti("speckleWindowRange"); para.disparityMode = geti("mode");
    mvsv_sgbm_params p;
    std::memset(&p, 0, sizeof p);
    p.minDisp = para.minDisp; p.numDisp = para.numDisp; p.blockSize = para.blockSize; p.disp12MaxDiff = para.disp12MaxDiff;
    p.preFilterCap = para.preFilterCap; p.uniquenessRatio = para.uniquenessRatio; p.speckleWindowSize = para.speckleWindowSize;
    p.speckleRange = para.speckleRange; p.disparityMode = para.disparityMode == 1 ? 1 : 0;
    disparityObj.setSgbm(p);
    return true;
}

}  // namespace Disparity
